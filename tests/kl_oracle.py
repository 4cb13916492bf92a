"""CPU reference of the pathwise training objective (method 'kl' / 'kl_ito'): the training loops of
oracle/rollout_oracle.py with the SDE following the NON-detached control (generative_and_sde_ctrl, losses/oc.py:83-103,
i.e. ``lv=False``) run under autograd, loss = mean(rnd[mask]) (compute_loss, oc.py:105-131).

Per loss class (what the loss value carries):
  EM / EI / DDPM-like (RDS, PIS): simulate_em / simulate_ei, the Ito term included for every method;
  DDS: simulate_dds with compute_ito_int = method != 'kl' (oc.py:1399-1431);
  DIS (TimeReversalLoss): the training form - the log-weight starts at 0 (oc.py:1164-1165), no divergence integral
  (oc.py:1217), the Ito term only for 'kl_ito', ending with - target(x_K).

There is no reference checkout to produce golden files for this objective: this module is the pin, and
tests/test_kl_oracle.py checks it against central finite differences of the loss.
"""
from __future__ import annotations

import torch

from oracle import rollout_oracle as O


def simulate_dis_train(ts, x, noise, ctrl, sde, terminal_unnorm_log_prob, compute_ito_int):
    """TimeReversalLoss.simulate with train=True, change_sde_ctrl=False (oc.py:1133-1238): the loop of
    rollout_oracle.simulate_dis without the initial log-density and the divergence integral."""
    rnd = torch.zeros(x.shape[0], 1, dtype=x.dtype)
    for k, (s, t) in enumerate(zip(ts[:-1], ts[1:])):
        g = ctrl(s, x)
        sde_diff = sde.diff(s)
        dt = t - s
        rnd = rnd + 0.5 * (g ** 2).sum(dim=-1, keepdim=True) * dt
        db = noise[k] * dt.sqrt()
        x = x + (sde.drift_coeff(s) * x + sde_diff * g) * dt + sde_diff * db
        if compute_ito_int:
            rnd = rnd + (g * db).sum(dim=-1, keepdim=True)
    return x, rnd - terminal_unnorm_log_prob(x)


def kl_loss_and_grads(problem: dict, x0: torch.Tensor, noise: torch.Tensor, method: str = "kl",
                      max_rnd: float | None = 1e8, dtype=torch.float32):
    """(loss, dg [K, B, d] = d loss / d g_k, {state_dict key: d loss / d parameter}, rnd) of ``loss(ts, x, ...)`` with
    ``method`` 'kl' or 'kl_ito' for a linear-loss problem of tests/cases.py (em / ei / ddpm / dds / dis)."""
    problem = O._cast(problem, dtype)
    ctrl_desc = dict(problem["ctrl"])
    ctrl_desc["sd"] = {k: v.detach().to(dtype).clone().requires_grad_(True) for k, v in ctrl_desc["sd"].items()}
    x0, noise = x0.to(dtype), noise.to(dtype)
    ts = problem["ts"]
    target_logp, target_score = O.make_target(problem["target"])
    if problem.get("clip_target") is not None:  # TrainableDiff.clipped_target_unnorm_log_prob, solver/oc.py:80-87
        raw = target_logp
        target_logp = lambda x: O.clip(raw(x), problem["clip_target"])  # noqa: E731
    base = O.make_ctrl(ctrl_desc, target_score, dtype)
    gs = []

    def ctrl(t, x):  # the control of every step, kept for d loss / d g_k
        g = base(t, x)
        gs.append(g)
        return g

    kind = problem["method"]
    with torch.enable_grad():
        if kind in ("em", "ei", "ddpm"):
            sde = O.make_sde(problem["sde"], dtype)
            ref_ctrl, ref_logp = O.make_reference(problem["ref"], sde)
            if kind == "em":
                _, rnd, _ = O.simulate_em(ts, x0, noise, ctrl, sde, ref_ctrl, target_logp, ref_logp)
            else:
                _, rnd, _ = O.simulate_ei(ts, x0, noise, ctrl, sde, ref_ctrl, target_logp, ref_logp, ddpm=(kind == "ddpm"))
        elif kind == "dds":
            _, ref_logp = O.make_reference(problem["ref"], None)
            _, rnd, _ = O.simulate_dds(ts, x0, noise, ctrl, problem["alpha"], problem["sigma"], target_logp, ref_logp,
                                       compute_ito_int=(method != "kl"))
        elif kind == "dis":
            sde = O.make_sde(problem["sde"], dtype)
            _, rnd = simulate_dis_train(ts, x0, noise, ctrl, sde, target_logp, compute_ito_int=(method != "kl"))
        else:
            raise ValueError(f"no 'kl' training loop for method {kind!r}")
        mask = rnd.isfinite() if max_rnd is None else rnd < max_rnd
        loss = rnd[mask].mean()
        names = list(ctrl_desc["sd"])
        out = torch.autograd.grad(loss, [ctrl_desc["sd"][k] for k in names] + gs, allow_unused=True)
    grads = {k: (g if g is not None else torch.zeros_like(ctrl_desc["sd"][k])) for k, g in zip(names, out[:len(names)])}
    return loss.detach(), torch.stack(out[len(names):]).detach(), grads, rnd.detach()
