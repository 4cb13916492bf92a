"""CPU: the full-covariance reference (tests/full_cov_oracle.py, GaussFull / GMMFull and the host packer of the
LRDS_GMM_FULL blocks) - the full kinds given diagonal matrices equal the oracle's diagonal kinds, the score is the
gradient of the log-density, the log-density is a torch.distributions mixture, the packed per-step blocks invert the
marginal covariances, and fit_gmm(em_type='full') returns SPD matrices."""
import math

import pytest
import torch

from oracle import rollout_oracle as O
from sde_sampler_lrds_b200 import _native as N
from sde_sampler_lrds_b200.distr.base import FullBlock, fill_gmm
from tests import full_cov_oracle as F

SDES = [{"kind": "vp", "beta_min": 0.1, "beta_max": 20.0, "scale": 1.0, "T": 1.0},
        {"kind": "vpcos", "c": 0.008, "scale": 1.0, "T": 1.0},
        {"kind": "pbm", "diff": 0.4472135954999579, "T": 5.0}]


def _diag_ref(M, d, seed, dtype=torch.float64):
    g = torch.Generator().manual_seed(seed)
    if M == 0:
        return {"kind": "gauss", "mean": torch.randn(d, generator=g, dtype=dtype),
                "var": 0.2 + torch.rand(d, generator=g, dtype=dtype)}
    return {"kind": "gmm", "means": torch.randn(M, d, generator=g, dtype=dtype),
            "variances": 0.2 + torch.rand(M, d, generator=g, dtype=dtype), "weights": torch.rand(M, generator=g, dtype=dtype) + 0.5}


@pytest.mark.parametrize("form", ["cov", "eig"])
@pytest.mark.parametrize("M", [0, 1, 4])
@pytest.mark.parametrize("sde", SDES, ids=["vp", "vpcos", "pbm"])
def test_full_kind_of_a_diagonal_reference_equals_the_diagonal_kind(sde, M, form):
    ref = _diag_ref(M, 7, seed=M + 3)
    full = F.as_full(ref, form)
    s = O.make_sde(sde, torch.float64)
    ctrl_d, logp_d = O.make_reference(ref, s)
    ctrl_f, logp_f = F.make_reference(full, s)
    x = 1.5 * torch.randn(64, 7, generator=torch.Generator().manual_seed(9), dtype=torch.float64)
    for t in (0.0, 0.13, 0.5, 0.97 * float(sde["T"])):
        t = torch.tensor(t, dtype=torch.float64)
        a, b = ctrl_d(t, x), ctrl_f(t, x)
        assert torch.allclose(a, b, rtol=1e-12, atol=1e-12), (a - b).abs().max()
    assert torch.allclose(logp_d(x), logp_f(x), rtol=1e-12, atol=1e-12)


def _random_spd(M, d, cond, seed):
    g = torch.Generator().manual_seed(seed)
    q, _ = torch.linalg.qr(torch.randn(M, d, d, generator=g, dtype=torch.float64))
    D = torch.logspace(0.0, math.log10(cond), d, dtype=torch.float64).expand(M, d) * 0.3
    return (q * D.unsqueeze(-2)) @ q.transpose(-1, -2)


@pytest.mark.parametrize("M,d,cond", [(1, 2, 10.0), (3, 5, 100.0), (5, 11, 100.0)])
@pytest.mark.parametrize("sde", SDES, ids=["vp", "vpcos", "pbm"])
def test_score_is_the_gradient_and_log_density_a_multivariate_normal_mixture(sde, M, d, cond):
    g = torch.Generator().manual_seed(M * 100 + d)
    cov = _random_spd(M, d, cond, seed=d)
    ref = {"kind": "gmm_full", "means": torch.randn(M, d, generator=g, dtype=torch.float64), "cov": cov,
           "weights": torch.rand(M, generator=g, dtype=torch.float64) + 0.2}
    s = O.make_sde(sde, torch.float64)
    means, logw, D, P = F._parts(ref, torch.float64)
    x = torch.randn(32, d, generator=g, dtype=torch.float64)
    for t in (0.0, 0.3, 0.8 * float(sde["T"])):
        t = torch.tensor(t, dtype=torch.float64)
        loc, prec, logc = F.marginal_full(s, t, means, D, P)
        xr = x.clone().requires_grad_(True)
        lp, score = F.mixture_full(xr, logw, loc, prec, logc)
        (grad,) = torch.autograd.grad(lp.sum(), xr)
        assert torch.allclose(score, grad, rtol=1e-10, atol=1e-10)
        covt = s.s(t) ** 2 * (cov + s.sigma_sq(t) * torch.eye(d, dtype=torch.float64))
        mvn = torch.distributions.MultivariateNormal(loc, covariance_matrix=covt)
        want = torch.logsumexp(mvn.log_prob(x.unsqueeze(1)) + logw, dim=-1, keepdim=True)
        assert torch.allclose(lp.detach(), want, rtol=1e-10, atol=1e-9)


@pytest.mark.parametrize("kind", ["gaussian", "gmm"])
@pytest.mark.parametrize("d", [3, 8, 13])
def test_packed_reference_blocks(kind, d):
    from sde_sampler_lrds_b200.eq.sdes import VP, MarginalReference
    M = 1 if kind == "gaussian" else 5
    cov = _random_spd(M, d, 50.0, seed=d + M).float()
    g = torch.Generator().manual_seed(4)
    means = torch.randn(M, d, generator=g)
    w = torch.rand(M, generator=g) + 0.5
    sde = VP(diff_coeff_sq_max=20.0)
    if kind == "gaussian":
        ref = MarginalReference(sde, "gaussian", x_init=means[0], var_init=cov[0])
    else:
        ref = MarginalReference(sde, "gmm", means_init=means, variances_init=cov, weights_init=w)
    assert ref.full
    taus = torch.tensor([0.0, 0.25, 0.6, 0.99])
    blk = ref.block_at(taus, "cpu")
    assert isinstance(blk, FullBlock)
    logc, mu, prec = blk
    dp = 8 * math.ceil(d / 8)
    assert prec.shape == (4, M, dp, dp) and mu.shape == (4, M, dp) and logc.shape == (4, 4 * math.ceil(M / 4))
    s, sig2 = sde.s(taus), sde.sigma_sq(taus)
    logw = torch.log(w / w.sum()).double() if kind == "gmm" else torch.zeros(1, dtype=torch.float64)
    for k in range(4):
        covt = s[k].double() ** 2 * (cov.double() + sig2[k].double() * torch.eye(d, dtype=torch.float64))
        eye = prec[k, :, :d, :d].double() @ covt
        assert torch.allclose(eye, torch.eye(d, dtype=torch.float64).expand_as(eye), atol=2e-4)
        assert torch.allclose(mu[k, :, :d], s[k] * means)
        want = torch.distributions.MultivariateNormal(torch.zeros(M, d, dtype=torch.float64), covt).log_prob(
            torch.zeros(1, M, d, dtype=torch.float64))[0] + logw
        assert torch.allclose(logc[k, :M].double(), want, rtol=1e-5, atol=1e-4)
        # padding: zero rows / columns / dims, -inf modes
        assert (prec[k, :, d:, :] == 0).all() and (prec[k, :, :, d:] == 0).all() and (mu[k, :, d:] == 0).all()
        assert torch.isneginf(logc[k, M:]).all()
    gm = N.Gmm()
    fill_gmm(gm, blk, stepped=True)
    assert gm.layout == N.GMM_FULL and gm.M == M and not gm.ivar and not gm.mix_tc
    assert gm.step_stride_sn == M * dp * dp and gm.step_stride_param == M * dp and gm.step_stride_logc == logc.shape[-1]
    # the distribution at t = 0 (the terminal term ref_0) packs the t = 0 block
    b0 = ref.distr_at(torch.tensor(0.0), "cpu").block("cpu")
    for a, b in zip(b0, blk):
        assert torch.equal(a, b[0])


def test_full_kind_is_detected_for_matrices_and_eigen_form():
    from sde_sampler_lrds_b200.eq.sdes import VP, MarginalReference
    sde = VP()
    d = 4
    cov = _random_spd(3, d, 10.0, seed=1).float()
    D, P = torch.linalg.eigh(cov.double())
    a = MarginalReference(sde, "gmm", means_init=torch.zeros(3, d), variances_init=cov, weights_init=torch.ones(3))
    b = MarginalReference(sde, "gmm", means_init=torch.zeros(3, d), variances_init=(D.float(), P.float()),
                          weights_init=torch.ones(3))
    for x, y in zip(a.block_at(torch.tensor([0.3]), "cpu"), b.block_at(torch.tensor([0.3]), "cpu")):
        assert torch.equal(x, y)
    diag = MarginalReference(sde, "gmm", means_init=torch.zeros(3, d), variances_init=torch.ones(3, d), weights_init=torch.ones(3))
    assert not diag.full and not isinstance(diag.block_at(torch.tensor([0.3]), "cpu"), FullBlock)
    with pytest.raises(ValueError):
        MarginalReference(sde, "gaussian", x_init=torch.zeros(d), var_init=-torch.eye(d))


def test_fit_gmm_full_returns_spd_covariances():
    pytest.importorskip("sklearn")
    from sde_sampler_lrds_b200.benchmark_utils import fit_gmm
    g = torch.Generator().manual_seed(0)
    d, n = 4, 3000
    A = torch.randn(d, d, generator=g)
    x = torch.cat([torch.randn(n, d, generator=g) @ A.T + 4.0, torch.randn(n, d, generator=g) @ A.T * 0.5 - 4.0])
    w, m, v = fit_gmm(2, x, em_type="full")
    assert w.shape == (2,) and m.shape == (2, d) and v.shape == (2, d, d)
    assert torch.allclose(v, v.transpose(-1, -2), atol=1e-6)
    assert (torch.linalg.eigvalsh(v.double()) > 0).all()
    wd, md, vd = fit_gmm(2, x, em_type="diag")
    assert vd.shape == (2, d)
