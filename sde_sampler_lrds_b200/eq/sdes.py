"""SDE coefficient algebra and transition kernels with the reference's class and method names
(sde_sampler/eq/sdes.py: TorchSDE 14-43, ControlledLangevinSDE 78-114, OU 117-351, ConstOU 354-403,
ScaledBM 406-424, VP 427-555, CosineVP 558-594, PinnedBM 597-678).

Time-only quantities (schedules, per-step coefficients, marginal parameters) are 0-dim / 1-D float32 torch
scalars evaluated with the same operation order as the reference, because they fill the per-step table the
rollout kernel consumes (include/lrds_b200.h, LRDS_STEP_*).  Per-particle work (integration steps, marginal
scores) is done by the CUDA library.
"""
from __future__ import annotations

import copy
import ctypes as C
import itertools

import torch
from torch.nn import Module

from .. import _native as N
from ..distr.base import Distribution, fill_gmm, full_eig, gmm_block, gmm_full_block
from ..distr.gauss import GMM, Gauss, GaussFull, GMMFull

_noise_calls = itertools.count()


def _axpy_step(x, s, z, a, b, c):
    """(a x + b s) + c z on the device; z drawn by the library's Philox generator when None."""
    if not x.is_cuda:
        raise N.LrdsError("integration steps run on CUDA tensors only (no CPU fallback)")
    xf = x.detach().to(torch.float32).contiguous()
    sf = s.detach().to(torch.float32).expand_as(xf).contiguous()
    if z is None:
        z = torch.empty_like(xf)
        seed = (int(torch.initial_seed()) & 0xFFFFFFFF) | (next(_noise_calls) << 32)
        flat = xf.reshape(-1, xf.shape[-1])
        # every rank of a torch.distributed job draws its own increments: the rank offsets the particle index
        rank = torch.distributed.get_rank() if torch.distributed.is_available() and torch.distributed.is_initialized() else 0
        with torch.cuda.device(x.device):
            N.check(N.lib().lrds_normals(seed, (rank & 0xFF) << 24, 0, 1, flat.shape[0], flat.shape[1], N.ptr(z), N.stream_ptr(x.device)))
    zf = z.detach().to(torch.float32).contiguous()
    out = torch.empty_like(xf)
    with torch.cuda.device(x.device):
        N.check(N.lib().lrds_axpy_step(N.ptr(xf), N.ptr(sf), N.ptr(zf), float(a), float(b), float(c), N.ptr(out),
                                       xf.numel(), N.stream_ptr(x.device)))
    return out, z


class TorchSDE(Module):
    """Generic SDE with a float32 ``terminal_t`` buffer."""

    noise_type: str = "diagonal"
    sde_type: str = "ito"

    def __init__(self, terminal_t: float = 1.0):
        super().__init__()
        self.register_buffer("terminal_t", torch.tensor(terminal_t, dtype=torch.float), persistent=False)
        object.__setattr__(self, "_host", None)  # plain attribute: the CPU copy must not become a child module

    def host(self):
        """CPU copy of the scalar algebra (used to fill per-step tables without device round trips)."""
        if self.terminal_t.device.type == "cpu":
            return self
        if self._host is None:
            object.__setattr__(self, "_host", copy.deepcopy(self).to("cpu"))
        return self._host

    def __getstate__(self):
        state = self.__dict__.copy()
        state["_host"] = None
        return state

    def _apply(self, fn):
        object.__setattr__(self, "_host", None)
        return super()._apply(fn)

    @property
    def device(self):
        return self.terminal_t.device

    def drift(self, t, x):
        raise NotImplementedError

    def diff(self, t, x):
        raise NotImplementedError

    def f(self, t, x):
        return self.drift(t, x).expand_as(x)

    def g(self, t, x):
        return self.diff(t, x).expand_as(x)


class ControlledLangevinSDE(TorchSDE):
    """Langevin SDE along the tempering path target^(t/T) prior^(1-t/T) (CMCD), eq/sdes.py:78-114."""

    def __init__(self, target_score, prior_score, diff_coeff: float = 1.0, terminal_t: float = 1.0,
                 clip_score: float | None = None, **kwargs):
        super().__init__(terminal_t=terminal_t, **kwargs)
        self.target_score = target_score
        self.prior_score = prior_score
        self.register_buffer("diff_coeff", torch.tensor(diff_coeff, dtype=torch.float), persistent=False)
        self.clip_score = clip_score

    def host(self):
        return self

    def drift(self, t, x):
        frac = t / self.terminal_t
        out = self.target_score(x) * frac + self.prior_score(x) * (1.0 - frac)
        out = out * (0.5 * self.diff_coeff ** 2)
        return out if self.clip_score is None else out.clip(-self.clip_score, self.clip_score)

    def diff(self, t, x):
        return self.diff_coeff


class OU(TorchSDE):
    """Linear SDE dX = drift_coeff_t(t) X dt + diff_coeff_t(t) dW with closed-form marginals."""

    def drift_coeff_t(self, t):
        raise NotImplementedError

    def diff_coeff_t(self, t):
        raise NotImplementedError

    def s(self, t):
        raise NotImplementedError

    def sigma_sq(self, t):
        raise NotImplementedError

    def drift(self, t, x):
        return self.drift_coeff_t(t) * x

    def diff(self, t, x=None):
        return self.diff_coeff_t(t)

    def drift_div(self, t, x):
        return self.drift_coeff_t(t) * x.shape[-1]

    def int_drift_coeff_t(self, s, t):
        raise NotImplementedError

    def drift_div_int(self, s, t, x):
        """Integral from s to t of the divergence of the drift (eq/sdes.py:137-141)."""
        return self.int_drift_coeff_t(s, t) * x.shape[-1]

    def transition_params(self, s, t):
        """X_t = mean X_s + sqrt(var) Z for s < t (generic form, eq/sdes.py:167-178)."""
        mean = torch.exp(torch.log(self.s(t)) - torch.log(self.s(s)))
        var = self.s(t) ** 2 * (self.sigma_sq(t) - self.sigma_sq(s))
        return mean, var

    def log_snr(self, t):
        a = self.s(t)
        return torch.log(torch.square(a) / (torch.square(a) * self.sigma_sq(t)))

    # ---- reference marginals p_t^ref ---------------------------------------------------------------------
    def marginal_params(self, t, x_init, var_init=None, is_mixture: bool = False):
        """(loc, var) of the marginal at t.  Full covariances (a matrix per component, or its eigen form (D, P)) come back
        in eigen form: (loc, (s^2 (D + sigma_sq), P)) (eq/sdes.py:232-239)."""
        if isinstance(var_init, tuple) or (var_init is not None and var_init.dim() > x_init.dim()):
            evals, evecs = var_init if isinstance(var_init, tuple) else full_eig(var_init)
            return self.s(t) * x_init, (self.s(t) ** 2 * (evals + self.sigma_sq(t)), evecs)
        loc = self.s(t) * x_init
        var = self.s(t) ** 2 * self.sigma_sq(t)
        if var_init is not None:
            var = var + self.s(t) ** 2 * var_init
        return loc, var

    def marginal_distr(self, t, x_init, var_init=None):
        loc, var = self.marginal_params(t, x_init, var_init=var_init)
        var = var * torch.ones_like(x_init)
        return Gauss(dim=x_init.shape[-1], loc=loc, scale=var.sqrt(), domain_tol=None)

    def marginal_score(self, t, x, x_init, var_init=None):
        return MarginalReference(self, "gaussian", x_init=x_init, var_init=var_init)(t, x)

    def marginal_gmm_params(self, t, means_init, variances_init, weights_init=None):
        means, variances = self.marginal_params(t, means_init, variances_init, is_mixture=True)
        if weights_init is None:
            weights_init = torch.ones((means.shape[0],), device=means.device) / means.shape[0]
        return weights_init, means, variances

    def marginal_gmm_distr(self, t, means_init, variances_init, weights_init=None):
        w, means, variances = self.marginal_gmm_params(t, means_init, variances_init, weights_init)
        return GMM(dim=means_init.shape[-1], loc=means, scale=torch.sqrt(variances), mixture_weights=w,
                   domain_tol=None)

    def marginal_gmm_score(self, t, x, means_init, variances_init, weights_init=None):
        return MarginalReference(self, "gmm", means_init=means_init, variances_init=variances_init,
                                 weights_init=weights_init)(t, x)

    # ---- denoising transition kernels -----------------------------------------------------------------------
    def ei_coeffs(self, t_k, t_k_p_1):
        """(a, b, c) of x' = a x + b s + c z for the exponential-integrator kernel."""
        raise NotImplementedError

    def ddpm_coeffs(self, t_k, t_k_p_1):
        raise NotImplementedError

    def ei_integration_step(self, x, t_k, t_k_p_1, s, z=None):
        a, b, c = self.ei_coeffs(t_k, t_k_p_1)
        return _axpy_step(x, s, z, a, b, c)

    def ddpm_integration_step(self, x, t_k, t_k_p_1, s, z=None):
        a, b, c = self.ddpm_coeffs(t_k, t_k_p_1)
        return _axpy_step(x, s, z, a, b, c)


class ConstOU(OU):
    """dX = -drift_coeff X dt + diff_coeff dW (eq/sdes.py:354-403)."""

    def __init__(self, drift_coeff: float = 2.0, diff_coeff: float = 2.0, **kwargs):
        if drift_coeff < 0 or diff_coeff <= 0:
            raise ValueError("Choose non-negative drift_coeff and positive diff_coeff.")
        super().__init__(**kwargs)
        self.register_buffer("drift_coeff", torch.tensor(drift_coeff, dtype=torch.float), persistent=False)
        self.register_buffer("diff_coeff", torch.tensor(diff_coeff, dtype=torch.float), persistent=False)

    def drift_coeff_t(self, t):
        return -self.drift_coeff

    def diff_coeff_t(self, t):
        return self.diff_coeff

    def int_drift_coeff_t(self, s, t):  # eq/sdes.py:385-389
        return -self.drift_coeff * (t - s)

    def s(self, t):
        return torch.exp(-self.drift_coeff * t)

    def sigma_sq(self, t):
        return -0.5 * self.diff_coeff ** 2 * (1.0 - torch.exp(2.0 * self.drift_coeff * t))


class ScaledBM(ConstOU):
    """dX = sigma dW (PIS), eq/sdes.py:406-424."""

    def __init__(self, *args, **kwargs):
        super().__init__(*args, drift_coeff=0.0, **kwargs)

    def s(self, t):
        return torch.ones_like(t)

    def sigma_sq(self, t):
        return self.diff_coeff ** 2 * t


class VP(OU):
    """Variance-preserving SDE, beta(t) linear in t (eq/sdes.py:427-555)."""

    def __init__(self, diff_coeff_sq_min: float = 0.1, diff_coeff_sq_max: float = 20.0,
                 scale_diff_coeff: float = 1.0, **kwargs):
        super().__init__(**kwargs)
        for name, val in (("scale_diff_coeff", scale_diff_coeff), ("diff_coeff_sq_min", diff_coeff_sq_min),
                          ("diff_coeff_sq_max", diff_coeff_sq_max)):
            self.register_buffer(name, torch.tensor(val, dtype=torch.float), persistent=False)

    def _diff_coeff_sq_t(self, t):
        return torch.lerp(self.diff_coeff_sq_min, self.diff_coeff_sq_max, t / self.terminal_t)

    def drift_coeff_t(self, t):
        return -0.5 * self._diff_coeff_sq_t(t)

    def diff_coeff_t(self, t):
        return self.scale_diff_coeff * torch.sqrt(self._diff_coeff_sq_t(t))

    def int_drift_coeff_t(self, s, t):  # eq/sdes.py:469-477
        return -0.25 * (self._diff_coeff_sq_t(t) + self._diff_coeff_sq_t(s)) * (t - s)

    def alpha_(self, t):
        return self.diff_coeff_sq_min * t + (0.5 * t ** 2 / self.terminal_t) * (
            self.diff_coeff_sq_max - self.diff_coeff_sq_min)

    def transition_params(self, s, t):
        lam = 1.0 - torch.exp(self.alpha_(s) - self.alpha_(t))
        return torch.sqrt(1.0 - lam), self.scale_diff_coeff ** 2 * lam

    def s(self, t):
        return torch.exp(-0.5 * self.alpha_(t))

    def sigma_sq(self, t):
        return -self.scale_diff_coeff ** 2 * (1.0 - (1.0 / self.s(t) ** 2))

    def _dalpha(self, t_k, t_k_p_1):
        return self.alpha_(self.terminal_t - t_k) - self.alpha_(self.terminal_t - t_k_p_1)

    def omega(self, t_k, t_k_p_1):
        return 4.0 * self.scale_diff_coeff ** 2 * torch.tanh(self._dalpha(t_k, t_k_p_1) / 4.0)

    def lambda_(self, t_k, t_k_p_1):
        return torch.exp(self._dalpha(t_k, t_k_p_1)) - 1.0

    def omega_ddpm(self, t_k, t_k_p_1):
        lk = 1.0 - torch.exp(-self.alpha_(self.terminal_t - t_k))
        lk1 = 1.0 - torch.exp(-self.alpha_(self.terminal_t - t_k_p_1))
        return self.scale_diff_coeff ** 2 * (lk / lk1) * self.lambda_(t_k, t_k_p_1)

    def ei_coeffs(self, t_k, t_k_p_1):
        lam = self.lambda_(t_k, t_k_p_1)
        root = torch.sqrt(1.0 + lam)
        return root, 2.0 * self.scale_diff_coeff ** 2 * (root - 1.0), self.scale_diff_coeff * torch.sqrt(lam)

    def ddpm_coeffs(self, t_k, t_k_p_1):
        T = self.terminal_t
        lam = self.lambda_(t_k, t_k_p_1)
        lam_rev = 1.0 - torch.exp(self.alpha_(T - t_k_p_1) - self.alpha_(T - t_k))
        lk = 1.0 - torch.exp(-self.alpha_(T - t_k))
        lk1 = 1.0 - torch.exp(-self.alpha_(T - t_k_p_1))
        half = self._dalpha(t_k, t_k_p_1) / 2.0
        var = self.scale_diff_coeff ** 2 * lam_rev * (lk1 / lk)
        return torch.sqrt(1.0 + lam), 2.0 * self.scale_diff_coeff ** 2 * torch.sinh(half), torch.sqrt(var)


class CosineVP(VP):
    """Variance-preserving SDE with the cosine schedule (eq/sdes.py:558-594; conf/sde/vp_cos.yaml).  Only the two scalar
    functions below differ from VP: everything per particle sees the schedule through the per-step table."""

    def __init__(self, c: float = 0.008, scale_diff_coeff: float = 1.0, **kwargs):
        super().__init__(scale_diff_coeff=scale_diff_coeff, **kwargs)
        self.register_buffer("c", torch.tensor(c, dtype=torch.float), persistent=False)

    def _diff_coeff_sq_t(self, t):
        return torch.pi * torch.tan(0.5 * torch.pi * ((t / self.terminal_t) + self.c) / (1.0 + self.c)) \
            / (self.terminal_t * (1.0 + self.c))

    def int_drift_coeff_t(self, s, t):
        raise NotImplementedError("int_drift_coeff_t is not yet implemented")  # as in the reference (eq/sdes.py:582-584)

    def alpha_(self, t):
        return -2.0 * torch.log(torch.cos(0.5 * torch.pi * ((t / self.terminal_t) + self.c) / (1.0 + self.c)))


class PinnedBM(OU):
    """Brownian motion pinned at terminal_t (eq/sdes.py:597-678)."""

    def __init__(self, diff_coeff: float = 2.0, **kwargs):
        if diff_coeff <= 0:
            raise ValueError("Choose positive diff_coeff.")
        super().__init__(**kwargs)
        self.register_buffer("diff_coeff", torch.tensor(diff_coeff, dtype=torch.float), persistent=False)

    def drift_coeff_t(self, t):
        return -1.0 / (self.terminal_t - t)

    def diff_coeff_t(self, t):
        return self.diff_coeff

    def transition_params(self, s, t):
        mean = (self.terminal_t - t) / (self.terminal_t - s)
        return mean, mean * (t - s) * self.diff_coeff ** 2

    def s(self, t):
        return (self.terminal_t - t) / self.terminal_t

    def sigma_sq(self, t):
        return self.diff_coeff ** 2 * self.terminal_t * t / (self.terminal_t - t)

    def omega(self, t_k, t_k_p_1):
        return self.diff_coeff ** 2 * (t_k / t_k_p_1) * (t_k_p_1 - t_k)

    def omega_ddpm(self, t_k, t_k_p_1):
        T = self.terminal_t
        return self.diff_coeff ** 2 * ((T - t_k) / (T - t_k_p_1)) * (t_k_p_1 - t_k)

    def ei_coeffs(self, t_k, t_k_p_1):
        ratio = t_k_p_1 / t_k
        dt = t_k_p_1 - t_k
        return ratio, self.diff_coeff ** 2 * dt, torch.sqrt(self.diff_coeff ** 2 * ratio * dt)

    def ddpm_coeffs(self, t_k, t_k_p_1):
        T = self.terminal_t
        dt = t_k_p_1 - t_k
        var = self.diff_coeff ** 2 * ((T - t_k_p_1) / (T - t_k)) * dt
        return t_k_p_1 / t_k, self.diff_coeff ** 2 * dt, torch.sqrt(var)


class MarginalReference:
    """The time-marginal reference score nabla log p_t^ref(x) of RDS (solver/oc.py:513-592) as an object the
    rollout can introspect: a Gaussian (``gaussian``/``default``) or mixture (``gmm``) pushed through the OU marginals
    (eq/sdes.py:208-248, 265-279, 329-345).  Covariances are diagonal ([d] / [M][d]) or full: a matrix ([d][d] /
    [M][d][d]) or the eigen form (eigenvalues [(M)][d], eigenvectors [(M)][d][d]); a matrix is decomposed once (fp64).
    The full kind packs LRDS_GMM_FULL blocks: per step the precision matrices P diag(1 / (D + sigma_sq)) P^T / s^2."""

    def __init__(self, sde: OU, kind: str, x_init=None, var_init=None, means_init=None, variances_init=None,
                 weights_init=None):
        self.sde, self.kind = sde, kind
        full_g = False
        if kind == "gaussian":
            self.means = x_init.reshape(1, -1)
            full_g = isinstance(var_init, tuple) or (var_init is not None and var_init.dim() == 2 and
                                                        var_init.shape[0] == var_init.shape[1] == self.means.shape[-1] > 1)
            self.variances = var_init if full_g or var_init is None else var_init.reshape(1, -1)
            self.weights = None
        elif kind == "gmm":
            self.means, self.variances, self.weights = means_init, variances_init, weights_init
            if self.weights is None:
                self.weights = torch.ones(means_init.shape[0]) / means_init.shape[0]
        else:
            raise NotImplementedError(f"reference type {kind!r} has no B200 kernel")
        M, d = self.means.shape
        self.full = isinstance(self.variances, tuple) or (self.variances is not None and self.variances.dim() == 3) or \
            (kind == "gaussian" and full_g)
        if self.full:
            if isinstance(self.variances, tuple):
                evals, evecs = self.variances
            else:
                evals, evecs = full_eig(self.variances.reshape(M, d, d))
            # tensors of the object key the cached rollout plans (losses/oc.py, _state)
            self.eigenvalues = evals.detach().to("cpu", torch.float32).reshape(M, d)
            self.eigenvectors = evecs.detach().to("cpu", torch.float32).reshape(M, d, d)
            if not bool((self.eigenvalues > 0).all()):
                raise ValueError("reference covariances must be positive definite")
        elif self.variances is not None and self.variances.dim() != 2:
            raise NotImplementedError("diagonal reference variances must be [M][d]")

    @property
    def dim(self):
        return self.means.shape[-1]

    def _s_sigma_sq(self, taus):
        h = self.sde.host()
        taus = taus.detach().to("cpu", torch.float32).reshape(-1, 1, 1)
        return h.s(taus), h.sigma_sq(taus)

    def params_at(self, taus: torch.Tensor):
        """(loc[S][M][d], var[S][M][d]) on the host for a 1-D tensor of times (diagonal kinds)."""
        if self.full:
            raise ValueError("params_at is the diagonal form; a full-covariance reference packs with block_at")
        h = self.sde.host()
        taus = taus.detach().to("cpu", torch.float32).reshape(-1, 1, 1)
        means = self.means.detach().to("cpu", torch.float32).unsqueeze(0)
        s = h.s(taus)
        loc = s * means
        var = s ** 2 * h.sigma_sq(taus)
        if self.variances is not None:
            var = var + s ** 2 * self.variances.detach().to("cpu", torch.float32).unsqueeze(0)
        return loc, var.expand_as(loc)

    def block_at(self, taus, device):
        if self.full:
            s, sig2 = self._s_sigma_sq(taus)
            return gmm_full_block(self.means, self.eigenvalues, self.eigenvectors, self.weights, device, s=s, sigma_sq=sig2)
        loc, var = self.params_at(taus)
        return gmm_block(loc, var, self.weights, device)

    def distr_at(self, t, device) -> Distribution:
        if self.full:
            s, sig2 = self._s_sigma_sq(torch.as_tensor(t).reshape(1))
            cls = GaussFull if self.kind == "gaussian" else GMMFull
            return cls.marginal(self.means.detach().cpu().float(), self.eigenvalues, self.eigenvectors,
                                None if self.weights is None else self.weights.detach().cpu().float(), s, sig2, device)
        loc, var = self.params_at(torch.as_tensor(t).reshape(1))
        if self.kind == "gaussian":
            return Gauss(dim=self.dim, loc=loc[0].to(device), scale=var[0].sqrt().to(device), domain_tol=None)
        return GMM(dim=self.dim, loc=loc[0].to(device), scale=var[0].sqrt().to(device),
                   mixture_weights=self.weights.to(device), domain_tol=None)

    def __call__(self, t, x):
        return self.distr_at(t, x.device).score(x)
