"""GPU: the pathwise training objective (method 'kl' / 'kl_ito') of ClippedCtrl samplers - fused rollout, reverse-time
adjoint kernel (lrds_adjoint), parameter pass - against the CPU reference tests/kl_oracle.py on identical increments;
then training steps through make_model.

Tolerances as for the 'lv' objective (test_train_gpu.py): loss within 1e-4 relative; every cotangent step and every
parameter-gradient tensor within 1e-3 of its largest entry (2e-2 for the logistic-regression target, whose clamp mask
flips for a few particles)."""
import math

import pytest
import torch

from tests import kl_oracle as KO
from tests.cases import (case_ddpm_snr, case_dds_many_modes, case_dis, case_ei_many_modes_clipped, case_ei_pbm,
                         case_pis_logreg, case_pis_many_modes, case_pis_phi4, ctrl, initial_state, noise_for)

pytestmark = pytest.mark.gpu


def _clipped(case, out_gain=0.5):
    """The case with a ClippedCtrl drift (base_zero_init) of the same dimension."""
    p = dict(case["problem"])
    d = p["ctrl"]["sd"]["base_model.input_embed.weight"].shape[1]
    p["ctrl"] = ctrl(d, "clipped", seed=case["seed"], out_gain=out_gain)
    return dict(case, problem=p)


KL_CASES = {
    "pis_many_modes": lambda: _clipped(case_pis_many_modes()),
    "pis_phi4": lambda: _clipped(case_pis_phi4(K=64, B=64), out_gain=0.3),
    "pis_logreg": lambda: _clipped(case_pis_logreg()),
    "ei_many_modes_clipped": case_ei_many_modes_clipped,
    "ei_pbm": case_ei_pbm,
    "ddpm_snr": lambda: _clipped(case_ddpm_snr()),
    "dds_many_modes": lambda: _clipped(case_dds_many_modes(True)),
    "dis_many_modes": lambda: _clipped(case_dis("many_modes", False)),
}
RUNS = [(n, "kl") for n in KL_CASES] + [("dds_many_modes", "kl_ito")]


def _tol(case):
    return 2e-2 if case["problem"]["target"]["kind"] == "logreg" else 1e-3


def _built(case, device, precision, method):
    from tests.product_builders import Built
    built = Built(case, device, precision)
    built.loss.method = method
    return built


def worst(got: dict, want: dict):
    assert set(got) == set(want), set(got) ^ set(want)
    return max(((got[k] - want[k]).abs().max() / want[k].abs().max().clamp(min=1e-12)).item() for k in want)


@pytest.mark.parametrize("precision", ["fp32", "f16x3"])
@pytest.mark.parametrize("name, method", RUNS)
def test_kl_gradient_matches_oracle(name, method, precision, device):
    from sde_sampler_lrds_b200 import pack
    from sde_sampler_lrds_b200 import train as TR
    case = KL_CASES[name]()
    x0, noise = initial_state(case), noise_for(case)
    built = _built(case, device, precision, method)
    loss, metrics = built.train_loss(x0, noise)
    assert loss.requires_grad and loss.ndim == 0 and "train/n_filtered_cumulative" in metrics
    loss.backward()
    got = {n: p.grad.detach().cpu() for n, p in built.ctrl.named_parameters() if p.grad is not None}
    lo, dg, go, _ = KO.kl_loss_and_grads(case["problem"], x0, noise, method)
    tol = _tol(case)
    assert abs(loss.item() - lo.item()) <= 1e-4 * max(1.0, abs(lo.item())), (loss.item(), lo.item())
    assert worst(got, go) < tol, worst(got, go)
    # the cotangents d loss / d g_k of the kernel, from the rollout of the very plan the training step used
    (plan,) = [h[0] for h in built.loss._plans.values()]
    x_dev, z_dev = x0.to(device), noise.to(device)
    x_T, rnd, xs = pack.run_rollout(plan, x_dev, z_dev, 0, 0, True)
    if case["problem"]["method"] == "dis":
        rnd = rnd - built.prior.log_prob(x_dev).reshape(rnd.shape)
    _, w, _ = TR._loss_weights(built.loss, rnd, x_T)
    cot = TR.adjoint(plan, xs, w, 0, z_dev).cpu()
    err = ((cot - dg).abs().amax(dim=(1, 2)) / dg.abs().amax(dim=(1, 2)).clamp(min=1e-30)).max().item()
    assert err < tol, err


@pytest.mark.parametrize("name", ["pis_many_modes", "ei_many_modes_clipped", "dis_many_modes"])
def test_kl_with_generated_noise_equals_recorded_noise(name, device):
    """Without recorded increments the rollout draws its noise in the kernel and the adjoint regenerates it: loss and
    gradient equal the run that is handed those increments as a recorded array."""
    from sde_sampler_lrds_b200 import train as TR
    case = KL_CASES[name]()
    x0 = initial_state(case)
    K, B, d = noise_for(case).shape
    out = []
    for recorded in (False, True):
        built = _built(case, device, "f16x3", "kl")
        z = TR.normals(11, 0, K, B, d, device) if recorded else None
        loss, _ = built.train_loss(x0, z, seed=11)
        loss.backward()
        out.append((loss.item(), {n: p.grad.detach().clone() for n, p in built.ctrl.named_parameters() if p.grad is not None}))
    (l0, g0), (l1, g1) = out
    assert abs(l0 - l1) <= 1e-6 * max(1.0, abs(l1))
    assert worst(g0, g1) < 5e-4


@pytest.mark.parametrize("solver_type, kw", [
    ("vp-ref", dict(ref_type="gmm", integrator_type="ei", time_type="snr")),
    ("pbm-ref", dict(ref_type="default", integrator_type="ei", time_type="snr")),
    ("pis_orig", dict(ref_type="default", integrator_type="em", time_type="uniform")),
    ("dds_orig", dict(ref_type="default", integrator_type="em", time_type="uniform")),
    ("dis_orig", dict(ref_type="default", integrator_type="em", time_type="uniform")),
])
def test_kl_training_steps_through_make_model(solver_type, kw, device):
    """make_model(..., model_type='base_zero_init', loss_type='kl'): three optimiser steps through TrainableWrapper.run,
    every loss finite and every parameter of the control moved."""
    from sde_sampler_lrds_b200 import benchmark_utils as BU
    from sde_sampler_lrds_b200.additions.hacking import TrainableWrapper
    from tests.test_solver_api_gpu import TRAIN, _gmm_ref, _randomise_last_layers
    d, M = 6, 5
    model = BU.make_model(solver_type=solver_type, loss_type="kl", model_type="base_zero_init", force_base_zero_init=True,
                          solver_details={"sigma": 1.0, **_gmm_ref(d, M)},
                          target_details=BU.make_target_details("many_modes", dim=d, n_modes=M),
                          training_details=dict(TRAIN, train_steps=3), n_steps=24, device=str(device), **kw)
    _randomise_last_layers(model)
    before = {n: p.detach().clone() for n, p in model.generative_ctrl.named_parameters()}
    res, hist = TrainableWrapper(model, verbose=False).run(keep_training_metrics=True)
    assert len(hist["train/loss"]) == 3 and all(math.isfinite(v) for v in hist["train/loss"])
    assert hist["train/no_grad"][-1] == 0 and hist["train/skipped_steps"][-1] == 0
    moved = [n for n, p in model.generative_ctrl.named_parameters() if not torch.equal(p.detach(), before[n])]
    assert len(moved) == len(before)
    assert math.isfinite(res.metrics["eval/elbo"])
