"""CPU statement of the full-covariance Gaussian / mixture reference of RDS (eq/sdes.py:232-239 and
score_mog_full / log_prob_gaussian_full, distr/gauss.py:76-121) and the rollouts that use it.

A reference component N(mu_m, Sigma_m), Sigma_m = P_m diag(D_m) P_m^T, has the marginal at time t
    loc_m(t) = s(t) mu_m,   cov_m(t) = s(t)^2 (Sigma_m + sigma^2(t) I),
    prec_m(t) = P_m diag(1 / (D_m + sigma^2(t))) P_m^T / s(t)^2,
    log c_m(t) = log w_m - d/2 log 2 pi - 1/2 sum_i log(s(t)^2 (D_mi + sigma^2(t))),
and the score -sum_m r_m h_m with h_m = prec_m (x - loc_m), r = softmax_m(log c_m - (x - loc_m) . h_m / 2).

The reference kinds here extend ``oracle.rollout_oracle.make_reference`` (which stays the statement of the diagonal
kinds):
    {"kind": "gauss_full", "mean": [d], "cov": [d][d]}          or "evals" [d] / "evecs" [d][d] instead of "cov"
    {"kind": "gmm_full", "means": [M][d], "cov": [M][d][d], "weights": [M]}   or "evals" [M][d] / "evecs" [M][d][d]
``rollout`` / ``lv_loss_and_grads`` run the EM / EI / DDPM-like losses of the oracle with them."""
from __future__ import annotations

import math

import torch

from oracle import rollout_oracle as O


def eig(ref: dict, dtype):
    """(evals [M][d], evecs [M][d][d]) of a full reference dict, in ``dtype``; a matrix is decomposed in float64."""
    if "cov" in ref:
        c = ref["cov"].to(torch.float64)
        c = c.reshape(-1, c.shape[-1], c.shape[-1])
        D, P = torch.linalg.eigh(0.5 * (c + c.transpose(-1, -2)))
    else:
        d = ref["evecs"].shape[-1]
        D, P = ref["evals"].reshape(-1, d), ref["evecs"].reshape(-1, d, d)
    return D.to(dtype), P.to(dtype)


def marginal_full(sde, t, means, D, P):
    """(loc [M][d], prec [M][d][d], logdet term [M]) of the marginal at t, in the operation order of the module doc."""
    s, sig2 = sde.s(t), sde.sigma_sq(t)
    Ds = D + sig2
    prec = torch.matmul(P * (1.0 / Ds).unsqueeze(-2), P.transpose(-1, -2)) / s ** 2
    logc = -0.5 * means.shape[-1] * math.log(2.0 * math.pi) - 0.5 * torch.log(s ** 2 * Ds).sum(dim=-1)
    return s * means, prec, logc


def mixture_full(x, logw, loc, prec, logc):
    """(log-density (B, 1), score (B, d)) of the mixture with per-mode precision matrices."""
    y = x.unsqueeze(1) - loc.unsqueeze(0)                        # [B][M][d]
    h = torch.einsum("mij,bmj->bmi", prec, y)
    logits = logc.unsqueeze(0) + logw.unsqueeze(0) - 0.5 * (y * h).sum(dim=-1)
    r = torch.softmax(logits, dim=-1)
    return torch.logsumexp(logits, dim=-1, keepdim=True), -(r.unsqueeze(-1) * h).sum(dim=1)


def _parts(ref: dict, dtype):
    if ref["kind"] == "gauss_full":
        means = ref["mean"].reshape(1, -1).to(dtype)
        logw = torch.zeros(1, dtype=dtype)
    else:
        means = ref["means"].to(dtype)
        w = ref["weights"].to(dtype)
        logw = torch.log(w / w.sum())
    D, P = eig(ref, dtype)
    return means, logw, D, P


def make_reference(ref: dict | None, sde):
    """(reference_ctrl(t, x), reference_log_prob(x) -> (B, 1)) as oracle.rollout_oracle.make_reference, plus the full
    kinds."""
    if ref is None or ref["kind"] not in ("gauss_full", "gmm_full"):
        return O.make_reference(ref, sde)
    dtype = ref["means" if "means" in ref else "mean"].dtype
    means, logw, D, P = _parts(ref, dtype)

    def ctrl(t, x):
        return mixture_full(x, logw, *marginal_full(sde, t, means, D, P))[1]
    loc0, prec0, logc0 = marginal_full(sde, torch.zeros((), dtype=dtype), means, D, P)
    return ctrl, (lambda x: mixture_full(x, logw, loc0, prec0, logc0)[0])


def distr_full(ref: dict, x: torch.Tensor):
    """(log-density, score) of the full distribution itself (s = 1, sigma^2 = 0) at x."""
    means, logw, D, P = _parts(ref, x.dtype)
    prec = torch.matmul(P * (1.0 / D).unsqueeze(-2), P.transpose(-1, -2))
    logc = -0.5 * means.shape[-1] * math.log(2.0 * math.pi) - 0.5 * torch.log(D).sum(dim=-1)
    return mixture_full(x, logw, means, prec, logc)


def as_full(ref: dict, form: str = "cov") -> dict:
    """The diagonal reference ``ref`` ("gauss" / "gmm") restated with full matrices diag(v) ("cov") or as (v, I) ("eig")."""
    if ref["kind"] == "gauss":
        v = ref["var"].reshape(1, -1)
        out = {"kind": "gauss_full", "mean": ref["mean"].clone()}
    elif ref["kind"] == "gmm":
        v = ref["variances"]
        out = {"kind": "gmm_full", "means": ref["means"].clone(), "weights": ref["weights"].clone()}
    else:
        raise ValueError(ref["kind"])
    d = v.shape[-1]
    if form == "cov":
        out["cov"] = torch.diag_embed(v)
    else:
        out["evals"], out["evecs"] = v.clone(), torch.eye(d, dtype=v.dtype).expand(v.shape[0], d, d).clone()
    if ref["kind"] == "gauss":
        out = {k: (t[0] if k in ("cov", "evals", "evecs") else t) for k, t in out.items()}
    return out


def rollout(problem: dict, x0: torch.Tensor, noise: torch.Tensor, *, eubo: bool = False, return_traj: bool = False,
            dtype=torch.float32, lv: bool = False):
    """oracle.rollout_oracle.rollout for the EM / EI / DDPM-like losses with any reference kind of ``make_reference``."""
    problem = O._cast(problem, dtype)
    x0, noise = x0.to(dtype), noise.to(dtype)
    ts = problem["ts"]
    target_logp, target_score = O.make_target(problem["target"])
    ctrl = O.make_ctrl(problem["ctrl"], target_score, dtype)
    method = problem["method"]
    if method not in ("em", "ei", "ddpm"):
        raise ValueError(method)
    with (torch.enable_grad() if lv else torch.no_grad()):
        sde = O.make_sde(problem["sde"], dtype)
        ref_ctrl, ref_logp = make_reference(problem["ref"], sde)
        if eubo:
            if method == "ei":
                return O.eubo_ei(ts, x0, noise, ctrl, sde, ref_ctrl, target_logp, ref_logp)
            return O.eubo_em(ts, x0, noise, ctrl, sde, ref_ctrl, target_logp, ref_logp, use_rescaling=(method == "em"))
        if method == "em":
            return O.simulate_em(ts, x0, noise, ctrl, sde, ref_ctrl, target_logp, ref_logp, return_traj, lv=lv)
        return O.simulate_ei(ts, x0, noise, ctrl, sde, ref_ctrl, target_logp, ref_logp, return_traj,
                             ddpm=(method == "ddpm"), lv=lv)


def lv_loss_and_grads(problem: dict, x0: torch.Tensor, noise: torch.Tensor, max_rnd: float | None = 1e8,
                      dtype=torch.float32):
    """oracle.rollout_oracle.lv_loss_and_grads (method 'lv') for the reference kinds of ``make_reference``."""
    problem = dict(problem)
    ctrl = dict(problem["ctrl"])
    ctrl["sd"] = {k: v.detach().to(dtype).clone().requires_grad_(True) for k, v in ctrl["sd"].items()}
    cast = O._cast({k: v for k, v in problem.items() if k != "ctrl"}, dtype)
    cast["ctrl"] = ctrl
    _, rnd, _ = rollout(cast, x0, noise, dtype=dtype, lv=True)
    mask = rnd.isfinite() if max_rnd is None else rnd < max_rnd
    loss = rnd[mask].var()
    names = list(ctrl["sd"])
    grads = torch.autograd.grad(loss, [ctrl["sd"][k] for k in names], allow_unused=True)
    return loss.detach(), {k: (g if g is not None else torch.zeros_like(ctrl["sd"][k])) for k, g in zip(names, grads)}, rnd.detach()


def random_full_ref(M: int, d: int, seed: int, decades: float = 2.0, mean_scale: float = 1.0, var_scale: float = 1.0):
    """A gmm_full reference with random orthogonal P_m and eigenvalues spread over ``decades`` (condition number
    10^decades), float32 eigen form and the float64 covariance it stands for."""
    g = torch.Generator().manual_seed(seed)
    q, _ = torch.linalg.qr(torch.randn(M, d, d, generator=g, dtype=torch.float64))
    D = var_scale * torch.logspace(-decades / 2, decades / 2, d, dtype=torch.float64)
    D = D[torch.stack([torch.randperm(d, generator=g) for _ in range(M)])]
    means = mean_scale * torch.randn(M, d, generator=g, dtype=torch.float64)
    w = torch.rand(M, generator=g, dtype=torch.float64) + 0.5
    cov = (q * D.unsqueeze(-2)) @ q.transpose(-1, -2)
    return {"kind": "gmm_full", "means": means.float(), "cov": cov.float(), "weights": w.float()}, cov
