"""GPU: the pathwise CMCD training objective (method 'kl' / 'kl_ito', ClippedCtrl) - fused rollout, reverse-time adjoint
kernel (lrds_adjoint_cmcd), parameter pass over the K + 1 trajectory points - against the CPU reference
tests/cmcd_kl_oracle.py on identical increments; then training steps through make_model.

Tolerances as for the linear 'kl' objective (test_kl_train_gpu.py): loss within 1e-4 relative; every cotangent point and
every parameter-gradient tensor within 1e-3 of its largest entry - here against the reference evaluated in fp64."""
import math

import pytest
import torch

from tests import cmcd_kl_oracle as CKO
from tests.cases import case_cmcd_gmm, case_cmcd_many_modes, ctrl, initial_state, many_modes, noise_for, phi4, uniform_ts

pytestmark = pytest.mark.gpu


def _cmcd(target, d, K, B, seed, prior_scale=2.0, clip_score=1e5, out_gain=0.5):
    return {"problem": {"method": "cmcd", "sde": None, "diff": 1.0, "T": 1.0, "clip_score": clip_score,
                        "ts": uniform_ts(1.0, K), "target": target, "ctrl": ctrl(d, "clipped", seed=seed, out_gain=out_gain),
                        "prior": {"loc": torch.zeros(d), "scale": prior_scale * torch.ones(d), "isotropic": True}},
            "B": B, "seed": seed + 100, "prior": ("iso", 0.0, prior_scale)}


def _both_masks():
    """case_cmcd_gmm with a drift clip and a control clip small enough that both fire for part of the coordinates."""
    case = case_cmcd_gmm()
    p = dict(case["problem"], clip_score=3.0)
    p["ctrl"] = dict(p["ctrl"], clip_model=0.1)
    return dict(case, problem=p)


def _k1():
    case = case_cmcd_gmm()
    return dict(case, problem=dict(case["problem"], ts=uniform_ts(1.0, 1)))


CASES = {
    "gmm": case_cmcd_gmm,                                               # fitted diagonal prior, d = 8
    "many_modes": lambda: case_cmcd_many_modes("clipped"),               # the CMCD mixture kernel, ragged B = 170
    "phi4": lambda: _cmcd(phi4(24, beta=2.0), 24, 32, 96, 51, prior_scale=1.0, out_gain=0.3),
    "both_masks": _both_masks,
    # unit mode variances: with 0.5 these trajectories amplify rounding so much that an fp32 reference is off by 1e-3
    "d16": lambda: _cmcd(many_modes(3, 16, var=1.0), 16, 24, 130, 52),
    "d17": lambda: _cmcd(many_modes(3, 17, var=1.0), 17, 24, 130, 53),
    "k1": _k1,
}


def _built(case, device, precision, method="kl"):
    from tests.product_builders import Built
    built = Built(case, device, precision)
    built.loss.method = method
    return built


def worst(got: dict, want: dict):
    assert set(got) == set(want), set(got) ^ set(want)
    return max(((got[k] - want[k]).abs().max() / want[k].abs().max().clamp(min=1e-12)).item() for k in want)


def _cotangents(built, x0, noise, seed=0):
    """ubar from the rollout of the very plan the training step used, and the status counters of that adjoint."""
    from sde_sampler_lrds_b200 import pack
    from sde_sampler_lrds_b200 import train as TR
    dev = built.device
    (plan,) = [h[0] for h in built.loss._plans.values()]
    x_dev = x0.to(dev)
    z_dev = None if noise is None else noise.to(dev)
    x_T, rnd, xs = pack.run_rollout(plan, x_dev, z_dev, seed, 0, True)
    rnd = rnd - built.prior.log_prob(x_dev).reshape(rnd.shape)
    _, w, _ = TR._loss_weights(built.loss, rnd, x_T)
    pack.read_status(dev)
    cot = TR.adjoint_cmcd(plan, xs, w, seed, z_dev)
    return cot, pack.read_status(dev)


@pytest.mark.parametrize("precision", ["fp32", "tf32x3", "f16x3"])
@pytest.mark.parametrize("name", list(CASES))
def test_cmcd_kl_gradient_matches_oracle(name, precision, device):
    case = CASES[name]()
    x0, noise = initial_state(case), noise_for(case)
    built = _built(case, device, precision)
    loss, metrics = built.train_loss(x0, noise)
    assert loss.requires_grad and loss.ndim == 0 and "train/n_filtered_cumulative" in metrics
    loss.backward()
    got = {n: p.grad.detach().cpu() for n, p in built.ctrl.named_parameters() if p.grad is not None}
    # the reference in fp64: over these trajectories an fp32 reference is itself off by up to ~1e-3 in places
    lo, du, go, _ = CKO.kl_loss_and_grads(case["problem"], x0, noise, dtype=torch.float64)
    assert abs(loss.item() - lo.item()) <= 1e-4 * max(1.0, abs(lo.item())), (loss.item(), lo.item())
    assert worst(got, go) < 1e-3, worst(got, go)
    cot, status = _cotangents(built, x0, noise)
    assert cot.shape == du.shape
    err = ((cot.cpu() - du).abs().amax(dim=(1, 2)) / du.abs().amax(dim=(1, 2)).clamp(min=1e-30)).max().item()
    assert err < 1e-3, err
    assert status["nonfinite"] == 0


def test_both_masks_fire_in_the_clipped_case():
    """The drift clip and the control clip of the 'both_masks' case are active along the oracle's trajectory."""
    from oracle import rollout_oracle as O
    case = _both_masks()
    p = case["problem"]
    x0, noise = initial_state(case), noise_for(case)
    xs = O.rollout(p, x0, noise, return_traj=True)[2]
    ts, _, _, drift, _ = CKO._parts(dict(p, clip_score=None), torch.float32)
    raw = torch.stack([drift(ts[j], xs[j]) for j in range(len(ts))])
    assert 0.01 < (raw.abs() > p["clip_score"]).float().mean() < 0.99
    net = O.make_ctrl(dict(p["ctrl"], clip_model=None), None)
    u = torch.stack([net(ts[j], xs[j]) for j in range(len(ts))])
    assert 0.01 < (u.abs() > p["ctrl"]["clip_model"]).float().mean() < 0.99


@pytest.mark.parametrize("name", ["gmm", "many_modes"])
def test_cmcd_kl_with_generated_noise_equals_recorded_noise(name, device):
    """Without recorded increments the rollout draws its noise in the kernel and the adjoint regenerates it: loss and
    gradient equal the run that is handed those increments as a recorded array."""
    from sde_sampler_lrds_b200 import train as TR
    case = CASES[name]()
    x0 = initial_state(case)
    K, B, d = noise_for(case).shape
    out = []
    for recorded in (False, True):
        built = _built(case, device, "f16x3")
        z = TR.normals(11, 0, K, B, d, device) if recorded else None
        loss, _ = built.train_loss(x0, z, seed=11)
        loss.backward()
        out.append((loss.item(), {n: p.grad.detach().clone() for n, p in built.ctrl.named_parameters() if p.grad is not None}))
    (l0, g0), (l1, g1) = out
    assert abs(l0 - l1) <= 1e-6 * max(1.0, abs(l1))
    assert worst(g0, g1) < 5e-4


@pytest.mark.parametrize("precision", ["fp32", "f16x3"])
def test_cmcd_adjoint_is_deterministic(precision, device):
    case = CASES["many_modes"]()
    x0 = initial_state(case)
    built = _built(case, device, precision)
    loss, _ = built.train_loss(x0, None, seed=5)
    assert math.isfinite(loss.item())
    a, sa = _cotangents(built, x0, None, seed=5)
    b, sb = _cotangents(built, x0, None, seed=5)
    assert torch.equal(a, b)
    assert sa["nonfinite"] == 0 and sb["nonfinite"] == 0


def test_cmcd_kl_training_steps_through_make_model(device):
    """make_model(solver_type='cmcd', model_type='base_zero_init', loss_type='kl') over many_modes: three optimiser
    steps through TrainableWrapper.run, every loss finite and every parameter of the control moved."""
    from sde_sampler_lrds_b200 import benchmark_utils as BU
    from sde_sampler_lrds_b200.additions.hacking import TrainableWrapper
    from tests.test_solver_api_gpu import TRAIN, _gmm_ref, _randomise_last_layers
    d, M = 6, 5
    model = BU.make_model(solver_type="cmcd", loss_type="kl", model_type="base_zero_init", force_base_zero_init=True,
                          solver_details={"sigma": 1.0, **_gmm_ref(d, M)},
                          target_details=BU.make_target_details("many_modes", dim=d, n_modes=M),
                          training_details=dict(TRAIN, train_steps=3), n_steps=24, device=str(device),
                          ref_type="default", integrator_type="em", time_type="uniform")
    _randomise_last_layers(model)
    before = {n: p.detach().clone() for n, p in model.generative_ctrl.named_parameters()}
    res, hist = TrainableWrapper(model, verbose=False).run(keep_training_metrics=True)
    assert len(hist["train/loss"]) == 3 and all(math.isfinite(v) for v in hist["train/loss"])
    assert hist["train/no_grad"][-1] == 0 and hist["train/skipped_steps"][-1] == 0
    moved = [n for n, p in model.generative_ctrl.named_parameters() if not torch.equal(p.detach(), before[n])]
    assert len(moved) == len(before)
    assert math.isfinite(res.metrics["eval/elbo"])


def test_cmcd_kl_training_form_of_simulate(device):
    """simulate(train=True) with method 'kl' returns the log-weights of the training form: the evaluation rollout's minus
    the prior log-density of x_0."""
    case = CASES["gmm"]()
    x0, noise = initial_state(case), noise_for(case)
    built = _built(case, device, "fp32")
    _, rnd_eval, _ = built.simulate(x0, noise)
    _, rnd_train, _ = built.loss.simulate(built.ts, x0.to(device), *built.args, train=True, noise=noise.to(device))
    want = rnd_eval - built.prior.log_prob(x0.to(device)).reshape(rnd_eval.shape)
    assert torch.allclose(rnd_train, want, rtol=0, atol=1e-5 * want.abs().max().item())
    _, _, _, rnd_o = CKO.kl_loss_and_grads(case["problem"], x0, noise)
    assert torch.allclose(rnd_train.cpu(), rnd_o, rtol=1e-4, atol=1e-4)


def test_score_ctrl_cmcd_kl_still_raises(device):
    case = case_cmcd_many_modes("score")
    built = _built(case, device, "f16x3")
    with pytest.raises(NotImplementedError):
        built.train_loss(initial_state(case), noise_for(case))


@pytest.mark.parametrize("precision, kernel", [("f16x3", "adjoint_cmcd_tc_kernel"), ("tf32x3", "adjoint_cmcd_simt_kernel"),
                                               ("fp32", "adjoint_cmcd_simt_kernel")])
def test_cmcd_adjoint_kernel_choice(precision, kernel, device):
    """F16X3 specs inside the weight-gradient kernel's envelope run the tensor-core adjoint; the others the fp32 anchor."""
    from torch.profiler import ProfilerActivity, profile
    case = CASES["many_modes"]()
    x0, noise = initial_state(case), noise_for(case)
    built = _built(case, device, precision)
    built.train_loss(x0, noise)[0].backward()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _cotangents(built, x0, noise)
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages() if "adjoint_cmcd" in e.key]
    assert len(names) == 1 and kernel in names[0], names
