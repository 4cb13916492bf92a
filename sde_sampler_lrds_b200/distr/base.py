"""Distribution base class: the reference's interface (sde_sampler/distr/base.py:24-157) evaluated by the
CUDA library.  ``unnorm_log_prob`` / ``score`` run lrds_distr_eval on CUDA tensors; there is no CPU path."""
from __future__ import annotations

import ctypes as C
import math
from pathlib import Path

import torch

from .. import _native as N

EXPECTATION_FNS = {
    "square": lambda x: (x ** 2).sum(dim=-1, keepdims=True),
    "abs": lambda x: x.abs().sum(dim=-1, keepdims=True),
    "sum": lambda x: x.sum(dim=-1, keepdims=True),
    "square_minus_sum": lambda x: (x ** 2 - x).sum(dim=-1, keepdims=True),
}
DATA_DIR = Path(__file__).parents[2] / "data"


def gmm_block(loc: torch.Tensor, var: torch.Tensor, weights: torch.Tensor | None, device):
    """Packs a diagonal mixture into the (logc, mu, ivar, sn) block of lrds_gmm (include/lrds_b200.h).

    loc/var may carry a leading step axis ([S][M][d]) for the time-marginal reference.  logc follows
    log_prob_gaussian (distr/gauss.py:67-73) + log of the normalised weights (gauss.py:100-104).  Rows are padded
    to d_pad = 8 ceil(d/8) floats and logc to a multiple of 4 entries (-inf), so that the kernels read everything
    as aligned 16-byte vectors; ``sn`` interleaves 1/sigma and -mu/sigma per (mode block, dim group, mode)."""
    loc = loc.detach().to("cpu", torch.float32)
    var = var.detach().to("cpu", torch.float32).expand_as(loc)
    d, M = loc.shape[-1], loc.shape[-2]
    logc = -0.5 * d * math.log(2.0 * math.pi) - 0.5 * torch.log(var).sum(dim=-1)
    if weights is not None:
        w = weights.detach().to("cpu", torch.float32)
        logc = logc + torch.log(w / w.sum())
    ivar = (1.0 / var.double()).float()
    siv64 = 1.0 / var.double().sqrt()
    siv, nmsiv = siv64.float(), (-(loc.double() * siv64)).float()
    pad, mpad = (-d) % 8, (-M) % 4
    F = torch.nn.functional
    loc, ivar = F.pad(loc, (0, pad)), F.pad(ivar, (0, pad))
    logc = F.pad(logc, (0, mpad), value=float("-inf"))
    lead = loc.shape[:-2]
    m4, nq = (M + mpad) // 4, (d + pad) // 4
    sn = torch.stack([F.pad(t, (0, pad, 0, mpad)).reshape(*lead, m4, 4, nq, 4).transpose(-3, -2) for t in (siv, nmsiv)],
                     dim=-2)  # [.., m4, nq, 4 modes, 2, 4 dims]
    out = [logc, loc, ivar, sn.reshape(*lead, m4 * nq * 32)]
    if M > 1:
        out.append(gmm_mix_tc_image(loc[..., :d], var, d + pad, logc[..., :M], ivar[..., :d]))
    return tuple(t.contiguous().to(device) for t in out)


def _pow2_scale(amax: torch.Tensor) -> torch.Tensor:
    """The power of two that puts ``amax`` into [2^14, 2^15) (1 for amax = 0), float64."""
    k = torch.where(amax > 0, 14 - torch.floor(torch.log2(amax.clamp(min=1e-300))), torch.zeros_like(amax))
    return torch.pow(torch.tensor(2.0, dtype=torch.float64), k.clamp(-100, 100))


def gmm_logit_tc_image(loc: torch.Tensor, logc: torch.Tensor, ivar: torch.Tensor, d_pad: int) -> torch.Tensor:
    """The logit part of a lrds_gmm.mix_tc block (include/lrds_b200.h): wc = mu / var - mean over the modes as a
    power-of-two scaled fp16 hi | lo matrix [j/8][m][j%8] (modes padded to a multiple of 16, dims to a multiple of 16),
    then c_m = logc_m - sum_j mu^2 / var / 2 minus its maximum over the modes (fp32, -inf for the padded modes), then four floats
    {un-scale, max_m |wc_m|_2, max_m |c_m|, variances shared ? 1 : 0}.  ``ivar`` = the fp32 1/var the kernels see."""
    lead = loc.shape[:-2]
    M, d = loc.shape[-2:]
    Mp, Kin = (M + 15) // 16 * 16, (d_pad + 15) // 16 * 16
    iv = ivar.double()
    w = loc.double() * iv
    wc = (w - w.mean(dim=-2, keepdim=True).float().double()).float()   # the mean is held in fp32, as the device packer does
    c = logc.double() - 0.5 * (loc.double() ** 2 * iv).sum(dim=-1)
    c = (c - c.max(dim=-1, keepdim=True).values).float()  # softmax-invariant shift: the error bound scales with max |c_m|
    F = torch.nn.functional
    V = F.pad(wc, (0, Kin - d, 0, Mp - M))                             # [.., m, j]
    scale = _pow2_scale(V.abs().flatten(-2).max(dim=-1).values.double())
    Vs = (V.double() * scale[..., None, None]).float()
    hi = Vs.half()
    lo = (Vs - hi.float()).half()
    parts = [t.reshape(*lead, Mp, Kin // 8, 8).transpose(-3, -2).contiguous().reshape(*lead, -1).view(torch.uint8)
             for t in (hi, lo)]
    cpad = F.pad(c, (0, Mp - M), value=float("-inf"))
    tail = torch.zeros(*lead, 4, dtype=torch.float32)
    tail[..., 0] = (1.0 / scale).float()
    tail[..., 1] = wc.double().pow(2).sum(dim=-1).sqrt().max(dim=-1).values.float()
    tail[..., 2] = c.abs().max(dim=-1).values
    dev = ((ivar[..., 1:, :] - ivar[..., :1, :]).abs() / ivar[..., :1, :].abs()).flatten(-2).max(dim=-1).values \
        if M > 1 else torch.zeros(lead)
    tail[..., 3] = (dev <= 1e-6).float()
    return torch.cat(parts + [cpad.contiguous().view(torch.uint8), tail.view(torch.uint8)], dim=-1).contiguous()


def gmm_mix_tc_image(loc: torch.Tensor, var: torch.Tensor, d_pad: int, logc: torch.Tensor | None = None,
                     ivar: torch.Tensor | None = None) -> torch.Tensor:
    """Tensor-core operand of the mixture-score contraction (lrds_gmm.mix_tc, include/lrds_b200.h): per block the
    matrix B[n][m] with rows n = 16 c + i over 8-dim chunks c (i < 8: -1/var_{m, 8c+i}; i >= 8: mu/var_{m, 8c+i-8}),
    scaled by the power of two that puts its largest entry into [2^14, 2^15) and split into fp16 (hi, lo), each part
    in the K-major no-swizzle tcgen05 layout [m/8][n][m%8], followed by 16 bytes holding the float un-scale; then the
    logit image (gmm_logit_tc_image) when ``logc`` is given."""
    lead = loc.shape[:-2]
    M, d = loc.shape[-2:]
    Mp = (M + 15) // 16 * 16
    iv = 1.0 / var.double()
    a, b = (-iv).float(), (loc.double() * iv).float()
    F = torch.nn.functional
    T = torch.stack([F.pad(t, (0, d_pad - d, 0, Mp - M)).reshape(*lead, Mp, d_pad // 8, 8) for t in (a, b)], dim=-2)
    V = T.reshape(*lead, Mp, 2 * d_pad)                       # [.., m, n]
    amax = V.abs().flatten(-2).max(dim=-1).values.double().clamp(min=1e-30)
    k = 14 - torch.floor(torch.log2(amax))
    scale = torch.pow(torch.tensor(2.0, dtype=torch.float64), k)
    Vs = (V.double() * scale[..., None, None]).float()        # exact: power-of-two scaling
    hi = Vs.half()
    lo = (Vs - hi.float()).half()
    parts = [t.reshape(*lead, Mp // 8, 8, 2 * d_pad).transpose(-1, -2).contiguous().reshape(*lead, -1).view(torch.uint8)
             for t in (hi, lo)]
    tail = torch.zeros(*lead, 4, dtype=torch.float32)
    tail[..., 0] = (1.0 / scale).float()
    blocks = parts + [tail.view(torch.uint8)]
    if logc is not None:
        blocks.append(gmm_logit_tc_image(loc, logc, ivar if ivar is not None else (1.0 / var.double()).float(), d_pad))
    return torch.cat(blocks, dim=-1).contiguous()


class FullBlock(tuple):
    """(logc, mu, prec) of a full-covariance block (lrds_gmm.layout = LRDS_GMM_FULL, include/lrds_b200.h)."""


def full_eig(cov: torch.Tensor):
    """(eigenvalues [..][d], eigenvectors [..][d][d]) of symmetric positive-definite covariances, decomposed once in
    float64 and returned as float32 (the per-step blocks are formed from them in float32)."""
    c = cov.detach().to("cpu", torch.float64)
    evals, evecs = torch.linalg.eigh(0.5 * (c + c.transpose(-1, -2)))
    if not bool((evals > 0).all()):
        raise ValueError("covariance matrices must be positive definite")
    return evals.float(), evecs.float()


def gmm_full_block(means: torch.Tensor, evals: torch.Tensor, evecs: torch.Tensor, weights: torch.Tensor | None, device,
                   s: torch.Tensor | None = None, sigma_sq: torch.Tensor | None = None):
    """Packs the full-covariance mixture N(s mu_m, s^2 (Sigma_m + sigma_sq I)), Sigma_m = P_m diag(D_m) P_m^T, into a
    FullBlock.  ``s`` / ``sigma_sq`` carry a leading step axis ([S][1][1]) for the time-marginal reference (then every
    array gets one block per step) and default to 1 / 0 (the distribution itself).  Float32, in the order
        loc = s mu,  prec = P diag(1 / (D + sigma_sq)) P^T / s^2,
        logc = log w - d/2 log(2 pi) - 1/2 sum_i log(s^2 (D_i + sigma_sq)),
    rows padded to d_pad = 8 ceil(d / 8) with zeros (prec in its padded rows and columns too), logc to a multiple of
    4 entries with -inf."""
    means = means.detach().to("cpu", torch.float32)
    D, P = evals.to("cpu", torch.float32), evecs.to("cpu", torch.float32)
    M, d = means.shape
    s = torch.ones((1, 1)) if s is None else s.to("cpu", torch.float32)
    sigma_sq = torch.zeros((1, 1)) if sigma_sq is None else sigma_sq.to("cpu", torch.float32)
    Ds = D + sigma_sq                                                     # [(S)][M][d]
    loc = s * means
    prec = torch.matmul(P * (1.0 / Ds).unsqueeze(-2), P.transpose(-1, -2)) / s.unsqueeze(-1) ** 2
    logc = -0.5 * d * math.log(2.0 * math.pi) - 0.5 * torch.log(s ** 2 * Ds).sum(dim=-1)
    if weights is not None:
        w = weights.detach().to("cpu", torch.float32)
        logc = logc + torch.log(w / w.sum())
    pad, mpad = (-d) % 8, (-M) % 4
    F = torch.nn.functional
    loc = F.pad(loc, (0, pad))
    prec = F.pad(prec, (0, pad, 0, pad))
    logc = F.pad(logc, (0, mpad), value=float("-inf"))
    return FullBlock(t.contiguous().to(device) for t in (logc, loc, prec))


def fill_gmm(g: N.Gmm, block, stepped: bool = False):
    if isinstance(block, FullBlock):
        logc, mu, prec = block
        g.layout = N.GMM_FULL
        g.M = mu.shape[-2]
        g.logc, g.mu, g.ivar, g.sn = logc.data_ptr(), mu.data_ptr(), None, prec.data_ptr()
        g.step_stride_logc = logc.shape[-1] if stepped else 0
        g.step_stride_param = g.M * mu.shape[-1] if stepped else 0
        g.step_stride_sn = g.M * mu.shape[-1] ** 2 if stepped else 0
        g.mix_tc, g.step_stride_mix_tc = None, 0
        return g
    g.layout = N.GMM_DIAG
    logc, mu, ivar, sn = block[:4]
    g.M = mu.shape[-2]
    g.logc, g.mu, g.ivar, g.sn = logc.data_ptr(), mu.data_ptr(), ivar.data_ptr(), sn.data_ptr()
    g.step_stride_logc = logc.shape[-1] if stepped else 0
    g.step_stride_param = g.M * mu.shape[-1] if stepped else 0
    g.step_stride_sn = sn.shape[-1] if stepped else 0
    if len(block) > 4:
        g.mix_tc = block[4].data_ptr()
        g.step_stride_mix_tc = block[4].shape[-1] if stepped else 0
    else:
        g.mix_tc, g.step_stride_mix_tc = None, 0
    return g


class Distribution(torch.nn.Module):
    """Base class for probability distributions (same constructor and public methods as the reference)."""

    def __init__(self, dim: int, log_norm_const: float = None, domain=None, n_reference_samples=None,
                 grid_points=None):
        super().__init__()
        self.dim = dim
        self.n_reference_samples = n_reference_samples
        self.grid_points = grid_points
        self.set_domain(domain)
        self.log_norm_const = log_norm_const
        self.register_buffer("stddevs", None, persistent=False)
        self.expectations = {}
        self._lrds_cache = {}

    def __getstate__(self):
        # copy.deepcopy / pickling: the packed blocks hold ctypes structs with device pointers; a copy re-packs
        state = self.__dict__.copy()
        state["_lrds_cache"] = {}
        return state

    # ---- packing hook: subclasses return (N.Distr, keepalive) for a device ------------------------------
    def _lrds_pack(self, device):
        raise NotImplementedError(f"{type(self).__name__} has no B200 kernel (no fallback is provided).")

    def lrds_distr(self, device):
        key = str(device)
        if key not in self._lrds_cache:
            self._lrds_cache[key] = self._lrds_pack(torch.device(device))
        return self._lrds_cache[key]

    def _apply(self, fn):
        out = super()._apply(fn)
        self._lrds_cache = {}
        self._initialize_distr()
        return out

    def _initialize_distr(self):
        pass

    def _eval(self, x: torch.Tensor, want_logp: bool, want_score: bool):
        if not x.is_cuda:
            raise N.LrdsError(f"{type(self).__name__}: CUDA tensor required (no CPU fallback); got device {x.device}")
        lead = x.shape[:-1]
        xf = x.detach().reshape(-1, self.dim).to(torch.float32).contiguous()
        B = xf.shape[0]
        logp = torch.empty(B, device=x.device, dtype=torch.float32) if want_logp else None
        score = torch.empty_like(xf) if want_score else None
        distr, _keep = self.lrds_distr(x.device)
        with torch.cuda.device(x.device):
            N.check(N.lib().lrds_distr_eval(C.byref(distr), self.dim, N.ptr(xf), B, N.ptr(logp), N.ptr(score),
                                            N.stream_ptr(x.device)))
        if logp is not None:
            logp = logp.reshape(*lead, 1)
        if score is not None:
            score = score.reshape(*lead, self.dim)
        return logp, score

    # ---- reference interface ------------------------------------------------------------------------------
    def has_entropy(self):
        return False

    def set_domain(self, d=None):
        if d is not None:
            if not isinstance(d, torch.Tensor):
                d = torch.tensor(d, dtype=torch.float)
            if d.ndim == 0:
                d = torch.stack([-d, d], dim=-1)
            if d.ndim == 1:
                d = d.unsqueeze(0)
            if d.shape == (1, 2):
                d = d.repeat(self.dim, 1)
            assert d.shape == (self.dim, 2)
        self.register_buffer("domain", d, persistent=False)

    def unnorm_log_prob(self, x: torch.Tensor, *args, **kwargs) -> torch.Tensor:
        return self._eval(x, True, False)[0]

    def log_prob(self, x: torch.Tensor) -> torch.Tensor:
        if self.log_norm_const is None:
            raise NotImplementedError
        return self.unnorm_log_prob(x) - self.log_norm_const

    def pdf(self, x):
        return self.log_prob(x).exp()

    def unnorm_pdf(self, x):
        return self.unnorm_log_prob(x).exp()

    def score(self, x: torch.Tensor, *args, **kwargs) -> torch.Tensor:
        return self._eval(x, False, True)[1]

    def forward(self, x):
        return self.unnorm_log_prob(x)

    @torch.no_grad()
    def compute_stats(self):
        """Monte-Carlo reference expectations from true samples (reference: base.py:61-70, 96-118)."""
        if hasattr(self, "sample") and self.n_reference_samples is not None:
            samples = self.sample((self.n_reference_samples,))
            for name, fn in EXPECTATION_FNS.items():
                if name not in self.expectations:
                    self.expectations[name] = fn(samples).mean().item()
            if self.stddevs is None:
                self.stddevs = samples.std(dim=0)


def sample_uniform(domain: torch.Tensor, batchsize: int = 1) -> torch.Tensor:
    diam = domain[:, 1] - domain[:, 0]
    return domain[:, 0] + torch.rand(batchsize, domain.shape[0], device=domain.device) * diam
