"""MCMC sampling of a target with the reference's Metropolis-adjusted Langevin algorithm
(sde_sampler/additions/mcmc.py: mala_step 75-134, heuristics_step_size 54-72) - the sampler whose output the GMM
reference of RDS is fitted to (experiments/benchmark_utils.py: mcmc_sample 268-333).  The reference runs the chain loop
in Python, ~25 eager ops and one autograd call per step on a handful of chains; here the whole loop (proposal, target
log-density and score, accept / reject, per-chain step-size heuristic) is ONE kernel launch (lrds_mala, one thread per
chain).  No CPU fallback."""
from __future__ import annotations

import ctypes as C

import torch

from .. import _native as N
from ..distr.base import Distribution


def mala_chains(target: Distribution, y_init: torch.Tensor, step_size, n_warmup_steps: int, n_mcmc_steps: int,
                adapt_step_size: bool = True, noise: torch.Tensor | None = None, unif: torch.Tensor | None = None,
                seed: int | None = None, return_log_acc: bool = False, mcmc_type: str = "mala"):
    """Runs ``n_warmup_steps + n_mcmc_steps`` MALA steps of ``y_init.shape[0]`` chains (``mcmc_type='rwmh'``: random-walk
    Metropolis-Hastings steps, rwmh_step of sde_sampler/additions/mcmc.py:258-290 - the other sampler of mcmc_sample).

    Returns (ys [n_mcmc_steps, C, d], step_size [C, 1]) and, with ``return_log_acc``, the log acceptance ratios
    [n_warmup_steps + n_mcmc_steps, C].  ``noise`` [S, C, d] / ``unif`` [S, C] replay recorded draws (validation mode);
    otherwise the kernel draws them with its counter-based generator keyed by ``seed``."""
    if not isinstance(target, Distribution):
        raise NotImplementedError("mala_chains needs a kernel-backed Distribution as target")
    if mcmc_type not in ("mala", "rwmh"):
        raise NotImplementedError(f"mcmc_type {mcmc_type!r}: the kernel runs 'mala' and 'rwmh' (the two samplers of mcmc_sample)")
    if not y_init.is_cuda:
        raise N.LrdsError("MALA runs on CUDA tensors only (no CPU fallback)")
    dev = y_init.device
    y0 = y_init.detach().to(torch.float32).contiguous()
    Cn, d = y0.shape
    if d != target.dim:
        raise ValueError("y_init and the target have different dimensions")
    S = int(n_warmup_steps) + int(n_mcmc_steps)
    h = torch.as_tensor(step_size, dtype=torch.float32, device=dev).reshape(-1)
    h = (h.expand(Cn) if h.numel() == 1 else h).contiguous().clone()
    if h.numel() != Cn:
        raise ValueError("step_size must be a scalar or hold one value per chain")
    for name, t, shape in (("noise", noise, (S, Cn, d)), ("unif", unif, (S, Cn))):
        if t is not None and tuple(t.shape) != shape:
            raise ValueError(f"{name} must have shape {shape}, got {tuple(t.shape)}")
    noise = None if noise is None else noise.detach().to(dev, torch.float32).contiguous()
    unif = None if unif is None else unif.detach().to(dev, torch.float32).contiguous()
    if seed is None:
        seed = int(torch.initial_seed()) ^ 0x5DEECE66D
    distr, keep = target.lrds_distr(dev)
    ys = torch.empty(int(n_mcmc_steps), Cn, d, device=dev, dtype=torch.float32)
    log_acc = torch.empty(S, Cn, device=dev, dtype=torch.float32) if return_log_acc else None
    with torch.cuda.device(dev):
        N.check(N.lib().lrds_mala(C.byref(distr), d, Cn, int(n_warmup_steps), int(n_mcmc_steps), int(bool(adapt_step_size)),
                                  N.MCMC_RWMH if mcmc_type == "rwmh" else N.MCMC_MALA, N.ptr(y0), N.ptr(h), N.ptr(noise), N.ptr(unif), N.seed_arg(seed),
                                  N.ptr(ys), N.ptr(log_acc), N.stream_ptr(dev)))
    del keep
    out = (ys, h.unsqueeze(-1))
    return (*out, log_acc) if return_log_acc else out
