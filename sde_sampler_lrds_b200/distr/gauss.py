"""Diagonal Gaussian / Gaussian-mixture family with the reference's class names and constructors
(sde_sampler/distr/gauss.py: GMM 138-307, TwoModes 422-453, ManyModes 569-594, Gauss 597-629,
IsotropicGauss 720-787) and its functional helpers (log_prob_gaussian 67-73, score_mog 97-107,
score_gauss 124-126), plus the full-covariance Gaussian / mixture of the learned RDS references (GaussFull, GMMFull;
score_mog_full / log_prob_gaussian_full, distr/gauss.py:76-121).  Densities and scores are evaluated by the CUDA
library."""
from __future__ import annotations

import ctypes as C

import torch

from .. import _native as N
from .base import Distribution, fill_gmm, full_eig, gmm_block, gmm_full_block


class _AdHocMixture(Distribution):
    def __init__(self, loc, var, weights):
        super().__init__(dim=loc.shape[-1], log_norm_const=0.0)
        self._p = (loc, var, weights)

    def _lrds_pack(self, device):
        d = N.Distr()
        d.kind = N.DISTR_GMM
        block = gmm_block(*self._p, device)
        fill_gmm(d.gmm, block)
        return d, block


def score_mog(x, weights, means, variances):
    """Score of a diagonal mixture at x (reference: distr/gauss.py:97-107; the caller's weights are
    normalised in place there, here they are left untouched)."""
    return _AdHocMixture(means, variances, weights).score(x)


def score_gauss(x, means, variances):
    """Score of a diagonal Gaussian at x (reference: distr/gauss.py:124-126)."""
    means = means.reshape(1, -1)
    return _AdHocMixture(means, variances.reshape(1, -1).expand_as(means), None).score(x)


def log_prob_gaussian(x, mean, variance):
    """Per-component log-densities (B, M) of diagonal Gaussians (reference: distr/gauss.py:67-73)."""
    cols = [_AdHocMixture(mean[m:m + 1], variance[m:m + 1], None).unnorm_log_prob(x) for m in range(mean.shape[0])]
    return torch.cat(cols, dim=-1)


class GMM(Distribution):
    """Mixture of Gaussians with diagonal covariances."""

    def __init__(self, dim: int = 2, loc=None, scale=None, mixture_weights=None, n_reference_samples: int = int(1e7),
                 name=None, domain_scale: float = 5, domain_tol=1e-5, **kwargs):
        super().__init__(dim=dim, log_norm_const=0.0, n_reference_samples=n_reference_samples, **kwargs)
        if name is not None:
            raise NotImplementedError("named 2-D mixtures (gmm_params) are outside the rollout scope")
        self.n_mixtures = loc.shape[0]
        if not (loc.shape == scale.shape == (self.n_mixtures, self.dim)):
            raise ValueError("Shape missmatch between loc and scale.")
        if mixture_weights is None and self.n_mixtures > 1:
            raise ValueError("Require mixture weights.")
        if not (mixture_weights is None or mixture_weights.shape == (self.n_mixtures,)):
            raise ValueError("Shape missmatch for the mixture weights.")
        self.register_buffer("loc", loc, persistent=False)
        self.register_buffer("scale", scale, persistent=False)
        self.register_buffer("mixture_weights", mixture_weights, persistent=False)
        if self.domain is None:
            mean, std = self._moments()
            self.set_domain(torch.stack([mean - domain_scale * std, mean + domain_scale * std], dim=1))

    def _moments(self):
        if self.mixture_weights is None:
            return self.loc[0], self.scale[0]
        w = (self.mixture_weights / self.mixture_weights.sum()).unsqueeze(-1)
        mean = (w * self.loc).sum(0)
        var = (w * (self.scale ** 2 + self.loc ** 2)).sum(0) - mean ** 2
        return mean, var.sqrt()

    def _lrds_pack(self, device):
        d = N.Distr()
        d.kind = N.DISTR_GMM
        block = gmm_block(self.loc, torch.square(self.scale), self.mixture_weights, device)
        fill_gmm(d.gmm, block)
        return d, block

    def sample(self, shape=None) -> torch.Tensor:
        shape = tuple(shape or ())
        if self.mixture_weights is None:
            return self.loc[0] + self.scale[0] * torch.randn(*shape, self.dim, device=self.loc.device)
        n = int(torch.tensor(shape).prod()) if shape else 1
        comp = torch.multinomial(self.mixture_weights / self.mixture_weights.sum(), n, replacement=True)
        x = self.loc[comp] + self.scale[comp] * torch.randn(n, self.dim, device=self.loc.device)
        return x.reshape(*shape, self.dim)

    def has_entropy(self):
        return self.n_mixtures > 1


class TwoModes(GMM):
    """p = 2/3 N(-a 1, C) + 1/3 N(+a 1, C) (reference: distr/gauss.py:422-453)."""

    def __init__(self, dim=2, a=1.0, centered=False, ill_conditioned="not", **kwargs):
        assert ill_conditioned in ["not", "medium", "hard"]
        weights = torch.FloatTensor([2.0, 1.0])
        ones = torch.ones((dim,))
        loc = torch.stack([-a * ones, a * ones])
        if centered:
            loc = loc + (a / 3.0) * ones
        if ill_conditioned == "not":
            scale = torch.sqrt(0.05 * torch.ones_like(loc))
        else:
            lo = -1.0 if ill_conditioned == "medium" else -2.0
            scale = torch.sqrt(0.05 * torch.logspace(lo, 0.0, dim)).unsqueeze(0).expand(2, -1)
        super().__init__(dim=dim, loc=loc, scale=scale, mixture_weights=weights, **kwargs)


class BracketTwoModes(GMM):
    """p = 2/3 N(-a 1, C_1) + 1/3 N(+a 1, C_2), (C_1)_i = (C_2)_(dim-i) = linspace(var_min, var_max) (gauss.py:522-553)."""

    def __init__(self, dim=2, a=0.75, equilibrated=False, var_min=0.01, var_max=0.2, **kwargs):
        loc = torch.stack([-a * torch.ones((dim,)), a * torch.ones((dim,))], dim=0)
        variance_diag = torch.linspace(var_min, var_max, dim)
        scale = torch.sqrt(torch.stack([variance_diag, torch.flip(variance_diag, dims=(0,))], dim=0))
        weights = torch.ones((2,)) / 2.0 if equilibrated else torch.FloatTensor([2, 1]) / 2.0
        super().__init__(dim=dim, loc=loc, scale=scale, mixture_weights=weights, **kwargs)


class ManyModes(GMM):
    """n_modes isotropic components at seeded uniform locations, geometric weights (gauss.py:569-594)."""

    def __init__(self, n_modes=3, dim=2, seed_loc=42, mixture_weight_factor=3.0, var=0.1, **kwargs):
        gen = torch.Generator()
        gen.manual_seed(seed_loc)
        weights = torch.logspace(0.0, 1.0, n_modes, base=mixture_weight_factor)
        loc = 2 * n_modes * torch.rand((n_modes, dim), generator=gen) - n_modes
        scale = torch.sqrt(var * torch.ones_like(loc))
        super().__init__(dim=dim, loc=loc, scale=scale, mixture_weights=weights, **kwargs)


class Gauss(GMM):
    """Diagonal-covariance Gaussian (reference: distr/gauss.py:597-629)."""

    def __init__(self, dim: int = 1, loc=0.0, scale=1.0, **kwargs):
        loc, scale = Gauss._prepare_input(loc, dim), Gauss._prepare_input(scale, dim)
        super().__init__(dim=dim, loc=loc, scale=scale, **kwargs)
        self.stddevs = self.scale.squeeze(0)

    @staticmethod
    def _prepare_input(param, dim: int = 1):
        if not isinstance(param, torch.Tensor):
            param = torch.tensor(param, dtype=torch.float)
        param = torch.atleast_2d(param)
        if param.numel() == 1:
            param = param.repeat(1, dim)
        return param


class IsotropicGauss(Gauss):
    """Isotropic Gaussian, the usual prior (reference: distr/gauss.py:720-787)."""

    def __init__(self, dim: int = 1, loc: float = 0.0, scale: float = 1.0, truncate_quartile=None, **kwargs):
        super().__init__(dim=dim, loc=loc, scale=scale, **kwargs)
        assert torch.allclose(self.loc, self.loc[0, 0])
        assert torch.allclose(self.scale, self.scale[0, 0])
        if truncate_quartile is not None:
            raise NotImplementedError("truncated priors are not used by the rollout solvers")
        self.truncate_quartile = None

    def sample(self, shape=None) -> torch.Tensor:
        shape = tuple(shape or ())
        return self.loc[0, 0] + self.scale[0, 0] * torch.randn(*shape, self.dim, device=self.domain.device)


class GMMFull(Distribution):
    """Mixture of Gaussians with full covariance matrices: the learned RDS reference fitted with
    ``fit_gmm(em_type="full")`` and its time marginals (``MarginalReference.distr_at``).

    The reference names this class but its constructor could not be checked here; the signature below is this
    project's own.  ``covariance_matrix`` is [M][d][d] (symmetric positive definite), or ``eig`` = (eigenvalues [M][d],
    eigenvectors [M][d][d]) with Sigma_m = P_m diag(D_m) P_m^T, the form ``OU.marginal_params`` takes.  A matrix is
    decomposed once in float64.  ``log_prob`` / ``score`` run through lrds_distr_eval (full layout)."""

    def __init__(self, dim: int = 2, loc=None, covariance_matrix=None, mixture_weights=None, eig=None, **kwargs):
        super().__init__(dim=dim, log_norm_const=0.0, **kwargs)
        if (covariance_matrix is None) == (eig is None):
            raise ValueError("give exactly one of covariance_matrix and eig")
        self.n_mixtures = loc.shape[0]
        if loc.shape != (self.n_mixtures, dim):
            raise ValueError("loc must be [M][dim]")
        evals, evecs = full_eig(covariance_matrix) if eig is None else (eig[0].float(), eig[1].float())
        evals, evecs = evals.reshape(self.n_mixtures, dim), evecs.reshape(self.n_mixtures, dim, dim)
        if not bool((evals > 0).all()):
            raise ValueError("covariance matrices must be positive definite")
        if mixture_weights is None and self.n_mixtures > 1:
            raise ValueError("Require mixture weights.")
        self.register_buffer("loc", loc, persistent=False)
        self.register_buffer("eigenvalues", evals.to(loc.device), persistent=False)
        self.register_buffer("eigenvectors", evecs.to(loc.device), persistent=False)
        self.register_buffer("mixture_weights", mixture_weights, persistent=False)
        self._marginal = None  # (means_init, s, sigma_sq): packed in the time-marginal operation order

    @classmethod
    def marginal(cls, means, evals, evecs, weights, s, sigma_sq, device):
        """N(s mu_m, s^2 (Sigma_m + sigma_sq I)), packed with the arithmetic of the reference blocks (gmm_full_block)."""
        means, s, sigma_sq = means.float(), torch.as_tensor(s).float().reshape(1, 1), torch.as_tensor(sigma_sq).float().reshape(1, 1)
        out = cls.__new__(cls)
        GMMFull.__init__(out, dim=means.shape[-1], loc=(s * means).to(device), eig=(s ** 2 * (evals + sigma_sq), evecs),
                         mixture_weights=None if weights is None else weights.to(device))
        out._marginal = (means, evals, evecs, s, sigma_sq)
        return out

    @property
    def covariance_matrix(self):
        return (self.eigenvectors * self.eigenvalues.unsqueeze(-2)) @ self.eigenvectors.transpose(-1, -2)

    def block(self, device):
        if self._marginal is not None:
            means, evals, evecs, s, sigma_sq = self._marginal
            return gmm_full_block(means, evals, evecs, self.mixture_weights, device, s=s, sigma_sq=sigma_sq)
        return gmm_full_block(self.loc, self.eigenvalues, self.eigenvectors, self.mixture_weights, device)

    def _lrds_pack(self, device):
        d = N.Distr()
        d.kind = N.DISTR_GMM
        block = self.block(device)
        fill_gmm(d.gmm, block)
        return d, block

    def sample(self, shape=None) -> torch.Tensor:
        shape = tuple(shape or ())
        n = int(torch.tensor(shape).prod()) if shape else 1
        if self.mixture_weights is None:
            comp = torch.zeros(n, dtype=torch.long, device=self.loc.device)
        else:
            comp = torch.multinomial(self.mixture_weights / self.mixture_weights.sum(), n, replacement=True)
        z = torch.randn(n, self.dim, device=self.loc.device) * self.eigenvalues[comp].sqrt()
        x = self.loc[comp] + (self.eigenvectors[comp] @ z.unsqueeze(-1)).squeeze(-1)
        return x.reshape(*shape, self.dim)

    def has_entropy(self):
        return self.n_mixtures > 1


class GaussFull(GMMFull):
    """Gaussian with a full covariance matrix ``covariance_matrix`` [d][d] (or ``eig`` = (eigenvalues [d], eigenvectors
    [d][d])).  Constructor signature: this project's own, as for GMMFull."""

    def __init__(self, dim: int = 1, loc=0.0, covariance_matrix=None, eig=None, **kwargs):
        loc = Gauss._prepare_input(loc, dim)
        if covariance_matrix is not None:
            covariance_matrix = torch.as_tensor(covariance_matrix).reshape(1, dim, dim)
        super().__init__(dim=dim, loc=loc, covariance_matrix=covariance_matrix, eig=eig, **kwargs)
