"""GPU: RDS with a full-covariance Gaussian / mixture reference (lrds_gmm.layout = LRDS_GMM_FULL) through the product's
loss objects -> C ABI -> the run-time-switched rollout kernels (tcgen05 network and fp32 SIMT), against the CPU oracle of
tests/full_cov_oracle.py on identical Brownian increments, and - for the golden cases, whose diagonal references are
restated as full matrices diag(v) - against the reference-generated fixtures.

Bars as tests/test_rollout_parity_gpu.py: x_T and log-weights within 1e-4 relative (denominator max(|ref|, 1)), log Z
within 1e-3 absolute - for every particle of the golden cases.  The random rotated references (condition number 100)
are held to the bar of tests/test_edge_cases_gpu.py instead: every particle within 1e-2 and >= 97 % within 1e-4
(>= 90 % at M = 16, d = 50).  Measured on a B200: at M = 16, d = 50 between 92 % and 98 % of the particles meet 1e-4,
the worst at 1.5e-3, and the fp32 SIMT anchor misses exactly like the tensor-core kernel.  The cause is fp32 rounding,
not the kernel: far from the reference modes the quadratic forms (x - mu) . prec (x - mu) reach ~1e3, so their fp32
rounding (~1e-4 absolute, summation order differs from the oracle's) moves the responsibilities of particles near a
tie between two modes by that much, and 200 such steps compound it."""
import math
import os

import pytest
import torch

from oracle import rollout_oracle as O
from tests import cases as T
from tests import full_cov_oracle as F
from tests.cases import CASES, initial_state, noise_for

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")
REF_CASES = [n for n, mk in CASES.items() if mk()["problem"]["method"] in ("em", "ei", "ddpm")
             and mk()["problem"]["ref"]["kind"] in ("gauss", "gmm")]


def err_rel(a, b):
    e = (a - b).abs() / b.abs().clamp(min=1.0)
    return e.max(dim=1).values if e.dim() == 2 and e.shape[1] > 1 else e.reshape(-1)


def built_full(case, device, precision):
    """tests.product_builders.Built with the case's full reference ("gauss_full" / "gmm_full") in place of the diagonal
    one: MarginalReference of the full kind, its t = 0 distribution (GaussFull / GMMFull) as reference_log_prob."""
    from sde_sampler_lrds_b200.eq.sdes import MarginalReference
    from sde_sampler_lrds_b200.losses import oc
    from tests.product_builders import Built
    p = case["problem"]
    ref = p["ref"]
    d = ref["mean" if ref["kind"] == "gauss_full" else "means"].shape[-1]
    if ref["kind"] == "gauss_full":
        stub = {"kind": "gauss", "mean": ref["mean"], "var": torch.ones(d)}
    else:
        stub = {"kind": "gmm", "means": ref["means"], "variances": torch.ones_like(ref["means"]), "weights": ref["weights"]}
    b = Built(dict(case, problem=dict(p, ref=stub)), device, precision)
    var = ref["cov"].clone() if "cov" in ref else (ref["evals"].clone(), ref["evecs"].clone())
    if ref["kind"] == "gauss_full":
        b.ref = MarginalReference(b.sde, "gaussian", x_init=ref["mean"].clone(), var_init=var)
    else:
        b.ref = MarginalReference(b.sde, "gmm", means_init=ref["means"].clone(), variances_init=var,
                                  weights_init=ref["weights"].clone())
    assert b.ref.full
    b.ref_distr = b.ref.distr_at(torch.tensor(0.0), device)
    cls = {"em": oc.EMReferenceSDELoss, "ei": oc.EIReferenceSDELoss, "ddpm": oc.DDPMLikeReferenceSDELoss}[p["method"]]
    b.loss = cls(sde=b.sde, reference_ctrl=b.ref, generative_ctrl=b.ctrl, generative_ctrl_ema=b.ctrl, method="lv",
                 max_rnd=1e8, precision=precision)
    b.args = (b.target.unnorm_log_prob, b.ref_distr.log_prob)
    return b


def run_and_check(case, device, precision, gold=None, need=1.0):
    """>= ``need`` of the particles within 1e-4 of the oracle (and of the fixtures); with need < 1, every particle
    within 1e-2."""
    x0, noise = initial_state(case), noise_for(case)
    b = built_full(case, device, precision)
    if case.get("eubo"):
        rnd = b.compute_eubo(x0, noise).cpu()
        ref = F.rollout(case["problem"], x0, noise, eubo=True)
        pairs = [(rnd, ref, "rnd vs oracle")]
        m = O.eubo_results(rnd)
    else:
        x, rnd, _ = b.simulate(x0, noise)
        x, rnd = x.cpu(), rnd.cpu()
        xo, ro, _ = F.rollout(case["problem"], x0, noise)
        pairs = [(x, xo, "x_T vs oracle"), (rnd, ro, "rnd vs oracle")]
        if gold is not None:
            pairs.append((x, gold["x_T"], "x_T vs golden"))
        m = O.compute_results(rnd)
    if gold is not None:
        pairs.append((rnd, gold["rnd"], "rnd vs golden"))
    for got, want, what in pairs:
        assert got.shape == want.shape and torch.isfinite(got).all(), what
        e = err_rel(got, want)
        assert (e <= 1e-4).float().mean().item() >= need, f"{what}: worst {e.max().item():.2e}"
        assert need == 1.0 or e.max().item() <= 1e-2, f"{what}: worst {e.max().item():.2e}"
    if gold is not None and need == 1.0:
        for k, v in gold["metrics"].items():
            tol = 1e-3 if "log_norm_const" in k else 1e-3 * max(1.0, abs(v))
            assert abs(m[k] - v) <= tol, (k, m[k], v)
    return b


# ---- 1. tied to the reference's own outputs: the golden cases with their references restated as diag(v) ---------
@pytest.mark.parametrize("precision", ["f16x3", "tf32x3", "fp32"])
@pytest.mark.parametrize("name", REF_CASES)
def test_diagonal_golden_cases_as_full_matrices(name, precision, device):
    case = CASES[name]()
    # the matrix form for the f16x3 / fp32 kernels, the eigen form (v, I) for tf32x3
    case["problem"]["ref"] = F.as_full(case["problem"]["ref"], "eig" if precision == "tf32x3" else "cov")
    gold = torch.load(os.path.join(GOLDEN, name + ".pt"))
    run_and_check(case, device, precision, gold)


# ---- 2. rotated covariances ---------------------------------------------------------------------------------------
# grids that stay off the ends where the DDPM-like coefficients divide by zero (as the snr grids of make_model do)
GRIDS = {"vp": (T.VP20, lambda K: T.uniform_ts(1.0 - 1e-4, K, start=1e-4), ("iso", 0.0, 1.0)),
         "vpcos": (T.VPCOS, lambda K: T.uniform_ts(1.0, K, start=1e-3), ("iso", 0.0, 1.0)),
         "pbm": (T.PBM, lambda K: T.uniform_ts(5.0 - 1e-4, K, start=1e-4), ("delta", 0.0))}


def rotated_case(M, d, method, sde, K=40, B=64, seed=0):
    s, grid, prior = GRIDS[sde]
    tgt = T.many_modes(4, d, var=0.5)
    ref, _ = F.random_full_ref(M, d, seed=1000 * M + d, decades=2.0, mean_scale=1.0)
    return {"problem": {"method": method, "sde": s, "ts": grid(K), "target": tgt,
                        "ctrl": T.ctrl(d, "score", seed=21 + d, out_gain=0.5, gamma=0.05), "ref": ref},
            "B": B, "seed": 300 + seed + M + d, "prior": prior}


@pytest.mark.parametrize("sde", ["vp", "vpcos", "pbm"])
@pytest.mark.parametrize("method", ["em", "ei", "ddpm"])
@pytest.mark.parametrize("M,d", [(1, 2), (2, 6), (5, 11), (16, 50)])
def test_rotated_covariances(M, d, method, sde, device):
    case = rotated_case(M, d, method, sde)
    need = 0.9 if d == 50 else 0.97
    run_and_check(case, device, "f16x3", need=need)
    run_and_check(dict(case, eubo=True, seed=case["seed"] + 7), device, "f16x3", need=need)


@pytest.mark.parametrize("method", ["em", "ei"])
def test_rotated_covariances_fp32_anchor(method, device):
    case = rotated_case(16, 50, method, "vp")
    run_and_check(case, device, "fp32", need=0.9)
    run_and_check(dict(case, eubo=True, seed=case["seed"] + 7), device, "fp32", need=0.9)


# ---- 3. edge shapes, both batch regimes, shard and mode independence -----------------------------------------------
@pytest.mark.parametrize("B", [1, 37, 129])
@pytest.mark.parametrize("d", [8, 9, 16, 17])
@pytest.mark.parametrize("M", [1, 3])
def test_edge_shapes(M, d, B, device):
    case = rotated_case(M, d, "ei", "vp", K=1, B=B)
    case["problem"]["ts"] = T.uniform_ts(1.0, 100)[:2].clone()
    run_and_check(case, device, "f16x3", need=0.97)
    run_and_check(dict(case, eubo=True, seed=case["seed"] + 7), device, "f16x3", need=0.97)


def test_batches_on_both_sides_of_the_small_batch_threshold(device):
    """A full reference never takes the specialised mixture kernels: a batch the small-batch dispatcher would take and
    one beyond 128 particles per SM both run the generic kernel and meet the oracle."""
    sms = torch.cuda.get_device_properties(device).multi_processor_count
    for B in (96, 128 * sms + 37):
        case = rotated_case(2, 6, "ei", "vp", K=4, B=B)
        case["problem"]["ts"] = T.uniform_ts(1.0, 100)[:5].clone()
        run_and_check(case, device, "f16x3", need=0.97)


@pytest.mark.parametrize("precision", ["f16x3", "fp32"])
def test_shards_and_production_mode(precision, device):
    """Production mode (in-kernel Philox) is bit-for-bit independent of how the particles are split into shards, and
    equals validation mode on the increments lrds_normals dumps."""
    from sde_sampler_lrds_b200 import _native as N
    case = rotated_case(5, 11, "ei", "vp", K=20, B=300)
    x0 = initial_state(case).to(device)
    b = built_full(case, device, precision)
    full = b.simulate(x0, None, seed=1234)
    halves = [b.simulate(x0[:130], None, seed=1234, particle_offset=0), b.simulate(x0[130:], None, seed=1234, particle_offset=130)]
    for i in (0, 1):
        assert torch.equal(full[i], torch.cat([h[i] for h in halves]))
    K, B, d = 20, 300, 11
    z = torch.empty(K, B, d, device=device)
    N.check(N.lib().lrds_normals(1234, 0, 0, K, B, d, N.ptr(z), N.stream_ptr(device)))
    val = b.simulate(x0, z)
    for i in (0, 1):
        assert torch.equal(full[i], val[i])


# ---- 4. the distributions ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("M,d", [(1, 3), (1, 17), (4, 9), (16, 50)])
def test_gauss_full_and_gmm_full_distributions(M, d, device):
    from sde_sampler_lrds_b200.distr.gauss import GaussFull, GMMFull
    ref, cov = F.random_full_ref(M, d, seed=M + d)
    if M == 1:
        ref = {"kind": "gauss_full", "mean": ref["means"][0], "cov": ref["cov"][0]}
        dist = GaussFull(dim=d, loc=ref["mean"], covariance_matrix=ref["cov"]).to(device)
    else:
        dist = GMMFull(dim=d, loc=ref["means"], covariance_matrix=ref["cov"], mixture_weights=ref["weights"]).to(device)
    x = 2.0 * torch.randn(500, d, generator=torch.Generator().manual_seed(d))
    lp, sc = dist.log_prob(x.to(device)).cpu(), dist.score(x.to(device)).cpu()
    lpo, sco = F.distr_full({k: (v.double() if torch.is_tensor(v) else v) for k, v in ref.items()}, x.double())
    assert lp.shape == (500, 1) and sc.shape == (500, d)
    assert (err_rel(lp.double(), lpo) <= 1e-4).all(), err_rel(lp.double(), lpo).max()
    scale = sco.abs().max(dim=1, keepdim=True).values.clamp(min=1.0)
    assert ((sc.double() - sco).abs() / scale).max() <= 1e-4
    # the sampler of the class draws from the same distribution: mean and covariance of a large draw
    if M == 1:
        s = dist.sample((200000,)).double().cpu()
        assert torch.allclose(s.mean(0), ref["mean"].double(), atol=0.05 * cov.diagonal(dim1=-2, dim2=-1).max().sqrt().item())


# ---- 5. the lv training objective ------------------------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "f16x3"])
@pytest.mark.parametrize("which", ["em_two_modes", "ei_many_modes"])
def test_lv_loss_and_gradient(which, precision, device):
    if which == "em_two_modes":
        case = T.case_em_two_modes("score")
        case["problem"]["ref"] = {"kind": "gauss_full", "mean": torch.zeros(2), "cov": torch.tensor([[1.5, 0.6], [0.6, 0.9]])}
    else:
        case = T.case_ei_many_modes(K=50, B=100, d=20, M=5)
        case["problem"]["ref"], _ = F.random_full_ref(5, 20, seed=7, decades=1.0, mean_scale=3.0)
    x0, noise = initial_state(case), noise_for(case)
    b = built_full(case, device, precision)
    loss, _ = b.train_loss(x0, noise)
    loss.backward()
    got = {n: p.grad.detach().cpu() for n, p in b.ctrl.named_parameters() if p.grad is not None}
    lo, go, _ = F.lv_loss_and_grads(case["problem"], x0, noise)
    assert abs(loss.item() - lo.item()) <= 1e-4 * max(1.0, abs(lo.item()))
    assert set(got) == set(go)
    for k in go:
        assert (got[k] - go[k]).abs().max() <= 1e-3 * go[k].abs().max().clamp(min=1e-12), k


# ---- 6. the solver API ---------------------------------------------------------------------------------------------
def test_make_model_with_a_full_mixture_reference(device):
    from sde_sampler_lrds_b200 import benchmark_utils as BU
    from sde_sampler_lrds_b200.additions.hacking import TrainableWrapper
    from sde_sampler_lrds_b200.distr.gauss import GMMFull
    d, M = 6, 5
    ref, _ = F.random_full_ref(M, d, seed=3, decades=1.0, mean_scale=2.0)
    details = {"sigma": 1.0, "weights_ref": ref["weights"], "means_ref": ref["means"], "variances_ref": ref["cov"]}
    model = BU.make_model(solver_type="vp-ref", ref_type="gmm", loss_type="lv", integrator_type="ei",
                          model_type="target_informed_zero_init", time_type="uniform", solver_details=details,
                          target_details=BU.make_target_details("many_modes", dim=d, n_modes=M),
                          training_details={"train_steps": 4, "train_batch_size": 64, "eval_batch_size": 1000},
                          n_steps=24, device=str(device))
    assert model.reference_score_t.full and isinstance(model.reference_distr, GMMFull)
    res = TrainableWrapper(model, verbose=False).evaluate()
    for k in ("eval/elbo", "eval/lv_loss", "eval/eubo"):
        assert math.isfinite(res.metrics[k]), k
    B = 1000
    x, rnd, _ = model.loss.simulate(model.eval_ts, model.prior.sample((B,)), model.clipped_target_unnorm_log_prob,
                                    model.reference_distr.log_prob, seed=5)
    got = type(model.loss).compute_results(rnd, compute_weights=True)
    want = O.compute_results(rnd.cpu())
    assert abs(got.metrics["eval/elbo"] - want["eval/elbo"]) < 1e-4 * max(1, abs(want["eval/elbo"]))
    assert abs(got.log_norm_const_preds["log_norm_const_is"] - want["log_norm_const_is"]) < 1e-3
    xt = model.target.sample((B,))
    rf = model.loss.compute_eubo(model.eval_ts, xt, model.clipped_target_unnorm_log_prob, model.reference_distr.log_prob, seed=6)
    eo = O.eubo_results(rf.cpu())
    assert abs(eo["eval/eubo"] + rf.double().mean().item()) < 1e-4 * max(1.0, abs(eo["eval/eubo"]))
    assert math.isfinite(eo["eval/log_norm_const_is_f"])


def test_mcmc_fit_full_gmm_rds_workflow(device):
    """MCMC data -> fit_gmm(em_type='full') -> RDS with that full-covariance reference (tests/test_mcmc.py's target)."""
    from sde_sampler_lrds_b200 import benchmark_utils as BU
    from tests.cases import MALA_CASES
    from tests.product_builders import build_target
    case = MALA_CASES["mala_many_modes"]()
    target = build_target(case["target"], device)
    data = BU.mcmc_sample(device, target, case["x_init"], step_size=0.05, n_chains_per_mode=4, dataset_length=2800,
                          n_warmup_steps=64, seed=5)
    weights, means, covs = BU.fit_gmm(7, data, means_init=case["x_init"], em_type="full")
    assert covs.shape == (7, 10, 10) and (torch.linalg.eigvalsh(covs.double()) > 0).all()
    details = {"sigma": 1.0, "weights_ref": weights, "means_ref": means, "variances_ref": covs}
    model = BU.make_model(solver_type="vp-ref", ref_type="gmm", loss_type="lv", integrator_type="ei",
                          model_type="target_informed_zero_init", time_type="snr", solver_details=details,
                          target_details=BU.make_target_details("many_modes", dim=10, n_modes=7),
                          training_details={"train_steps": 2, "train_batch_size": 64, "eval_batch_size": 512},
                          n_steps=32, device=str(device))
    assert model.reference_score_t.full
    res = model.compute_results()
    assert res.metrics["eval/elbo"] > -5.0 and abs(res.log_norm_const_preds["log_norm_const_is"]) < 1.0


def test_full_blocks_are_refused_where_no_kernel_reads_them(device):
    import ctypes
    from sde_sampler_lrds_b200 import _native as N
    from sde_sampler_lrds_b200.distr.gauss import GMMFull
    ref, _ = F.random_full_ref(3, 5, seed=1)
    dist = GMMFull(dim=5, loc=ref["means"], covariance_matrix=ref["cov"], mixture_weights=ref["weights"]).to(device)
    distr, _keep = dist.lrds_distr(device)
    y0 = torch.zeros(4, 5, device=device)
    h = torch.full((4,), 0.1, device=device)
    ys = torch.empty(1, 4, 5, device=device)
    code = N.lib().lrds_mala(ctypes.byref(distr), 5, 4, 0, 1, 0, 0, N.ptr(y0), N.ptr(h), None, None, 1,
                             N.ptr(ys), None, N.stream_ptr(device))
    assert code == -2  # LRDS_ERR_UNSUPPORTED
