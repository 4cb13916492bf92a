"""CPU reference of the pathwise CMCD training objective (ControlledLangevinSDELoss with method 'kl' / 'kl_ito'): the
loop of oracle.rollout_oracle.simulate_cmcd with the SDE following the NON-detached control (``lv=False``) run under
autograd, in the training form - the log-weight starts at 0 (losses/oc.py:695-696), i.e. the rollout's log-weight minus
the prior log-density of x_0 - and loss = mean(rnd[mask]) (compute_loss, oc.py:105-131).  The Ito term is always part
of the CMCD log-weight, so 'kl' and 'kl_ito' are the same objective.

``kl_loss_and_grads`` also returns d loss / d u_j for the K + 1 trajectory points: the loop evaluates the control at
every interior point twice (as u_t of step j - 1 and u_s of step j), and the two derivatives are summed.
``adjoint_recursion`` is the reverse-time recursion of lrds_adjoint_cmcd (include/lrds_b200.h) in torch along the
oracle's own trajectory, with the Jacobians of the control and of the drift taken by autograd.

There is no reference checkout to produce golden files for this objective: this module is the pin, and
tests/test_cmcd_kl_oracle.py checks it against central finite differences of the loss.
"""
from __future__ import annotations

import torch

from oracle import rollout_oracle as O


def _parts(problem: dict, dtype):
    """(ts, target log-density, target score, prior log-density, prior score, drift(t, x), diff) of a CMCD problem of
    tests/cases.py, built like oracle.rollout_oracle.rollout."""
    p = O._cast({k: v for k, v in problem.items() if k != "ctrl"}, dtype)
    target_logp, target_score = O.make_target(p["target"])
    if p.get("clip_target") is not None:  # TrainableDiff.clipped_target_unnorm_log_prob, solver/oc.py:80-87
        raw = target_logp
        target_logp = lambda x: O.clip(raw(x), p["clip_target"])  # noqa: E731
    ploc, pscale = p["prior"]["loc"], p["prior"]["scale"]
    if p["prior"].get("isotropic", False):
        prior_logp = lambda x: O.isotropic_gauss_log_prob(x, float(ploc.flatten()[0]), float(pscale.flatten()[0]))  # noqa: E731
        prior_score = lambda x: (ploc.flatten()[0] - x) / pscale.flatten()[0] ** 2  # noqa: E731
    else:
        prior_logp = lambda x: O.gmm_log_prob(x, ploc.reshape(1, -1), pscale.reshape(1, -1), None)  # noqa: E731
        prior_score = lambda x: O.score_gauss(x, ploc.reshape(1, -1), torch.square(pscale.reshape(1, -1)))  # noqa: E731
    diff = torch.tensor(p["diff"], dtype=dtype)
    T = torch.tensor(p["T"], dtype=dtype)
    drift = lambda t, x: O.langevin_drift(t, x, target_score, prior_score, diff, T, p.get("clip_score"))  # noqa: E731
    return p["ts"], target_logp, prior_logp, drift, diff


def _ctrl_desc(problem: dict, dtype):
    c = dict(problem["ctrl"])
    c["sd"] = {k: v.detach().to(dtype).clone().requires_grad_(True) for k, v in c["sd"].items()}
    return c


def kl_loss_and_grads(problem: dict, x0: torch.Tensor, noise: torch.Tensor, method: str = "kl", dtype=torch.float32):
    """(loss, du [K + 1, B, d] = d loss / d u_j, {state_dict key: d loss / d parameter}, rnd) of the CMCD ``loss(ts, x,
    ...)`` with method 'kl' or 'kl_ito' (ClippedCtrl), in the training form."""
    if method not in ("kl", "kl_ito"):
        raise ValueError(method)
    x0, noise = x0.to(dtype), noise.to(dtype)
    ts, target_logp, prior_logp, drift, diff = _parts(problem, dtype)
    desc = _ctrl_desc(problem, dtype)
    base = O.make_ctrl(desc, None, dtype)
    calls = []

    def ctrl(t, x):  # every evaluation, for d loss / d u
        u = base(t, x)
        calls.append(u)
        return u

    with torch.enable_grad():
        _, rnd, _ = O.simulate_cmcd(ts, x0, noise, ctrl, drift, diff, target_logp, prior_logp, lv=False)
        rnd = rnd - prior_logp(x0)  # the training form starts at 0
        loss = rnd[rnd.isfinite()].mean()
        names = list(desc["sd"])
        out = torch.autograd.grad(loss, [desc["sd"][k] for k in names] + calls, allow_unused=True)
    K = len(ts) - 1
    g = out[len(names):]  # u_s of step 0, u_t of step 0, u_s of step 1, ...
    du = torch.zeros(K + 1, *x0.shape, dtype=dtype)
    for k in range(K):
        du[k] += g[2 * k]
        du[k + 1] += g[2 * k + 1]
    grads = {k: (v if v is not None else torch.zeros_like(desc["sd"][k])) for k, v in zip(names, out[:len(names)])}
    return loss.detach(), du, grads, rnd.detach()


def adjoint_recursion(problem: dict, x0: torch.Tensor, noise: torch.Tensor, w, dtype=torch.float64):
    """ubar [K + 1, B, d] of the recursion documented at lrds_adjoint_cmcd, along the oracle's trajectory from x0 with
    row weights ``w`` (a scalar or [B, 1]; d loss / d rnd_b)."""
    x0, noise = x0.to(dtype), noise.to(dtype)
    ts, target_logp, _, drift, sig = _parts(problem, dtype)
    desc = _ctrl_desc(problem, dtype)
    g = O.make_ctrl(desc, None, dtype)
    _, tscore = O.make_target(O._cast(problem["target"], dtype))
    K = len(ts) - 1

    def vjp(f, x, v):
        x = x.detach().requires_grad_(True)
        with torch.enable_grad():
            return torch.autograd.grad((f(x) * v).sum(), x)[0]

    with torch.no_grad():
        xs = [x0]
        for k in range(K):
            dt = ts[k + 1] - ts[k]
            xs.append(xs[k] + (drift(ts[k], xs[k]) + sig * g(ts[k], xs[k])) * dt + sig * dt.sqrt() * noise[k])
        u = [g(ts[j], xs[j]) for j in range(K + 1)]
        D = [drift(ts[j], xs[j]) for j in range(K + 1)]
        e = []
        for k in range(K):
            dt = ts[k + 1] - ts[k]
            e.append(w * (((D[k] + D[k + 1]) / sig + u[k] - u[k + 1]) * dt + dt.sqrt() * noise[k]))
        clip_t = problem.get("clip_target")
        lt = O.make_target(O._cast(problem["target"], dtype))[0](xs[K])
        wt = w * ((lt.abs() <= clip_t).to(dtype) if clip_t is not None else 1.0)
        ubar = torch.zeros(K + 1, *x0.shape, dtype=dtype)
        lam = -wt * tscore(xs[K])
        for j in range(K, -1, -1):
            ub = torch.zeros_like(x0)
            db = torch.zeros_like(x0)
            if j < K:
                dt = ts[j + 1] - ts[j]
                ub = ub + e[j] + sig * dt * lam
                db = db + e[j] / sig + dt * lam
            if j >= 1:
                ub = ub - e[j - 1]
                db = db + e[j - 1] / sig
            ubar[j] = ub
            if j == 0:
                break
            lam = lam + vjp(lambda x: g(ts[j], x), xs[j], ub) + vjp(lambda x: drift(ts[j], x), xs[j], db)
    return ubar
