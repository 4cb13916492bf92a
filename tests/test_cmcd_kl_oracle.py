"""CPU: the reference of the pathwise CMCD objective (tests/cmcd_kl_oracle.py) against fp64 central finite differences
of its loss, and the reverse-time recursion of lrds_adjoint_cmcd against its autograd cotangents - on mixture targets
with a diagonal and an isotropic prior and on PhiFour, with and without an active drift clip."""
import pytest
import torch

from tests import cmcd_kl_oracle as CKO
from tests.cases import ctrl, many_modes, phi4, uniform_ts

D, K, B = 3, 6, 5
PROBES = [("base_model.out_layer.weight", (1, 7)), ("base_model.input_embed.weight", (11, 0)),
          ("base_model.hidden_layer.0.bias", (4,)), ("base_model.timestep_embed.out_layer.bias", (9,))]


def _problem(target, clip_score, iso):
    tgt = many_modes(2, D) if target == "gmm" else phi4(D, beta=2.0)
    g = torch.Generator().manual_seed(5)
    prior = ({"loc": torch.zeros(D), "scale": 2.0 * torch.ones(D), "isotropic": True} if iso else
             {"loc": 0.3 * torch.randn(D, generator=g), "scale": 1.5 + torch.rand(D, generator=g), "isotropic": False})
    return {"method": "cmcd", "sde": None, "diff": 1.0, "T": 1.0, "clip_score": clip_score, "ts": uniform_ts(1.0, K),
            "target": tgt, "ctrl": ctrl(D, "clipped", seed=5, out_gain=1.0, num_hidden=1), "prior": prior}


def _inputs():
    gen = torch.Generator().manual_seed(3)
    return torch.randn(B, D, generator=gen, dtype=torch.float64) * 2, torch.randn(K, B, D, generator=gen, dtype=torch.float64)


CASES = [("gmm", 1e5, False), ("gmm", 0.8, False), ("gmm", 1e5, True), ("gmm", 0.8, True), ("phi4", 1e5, False),
         ("phi4", 0.8, False)]


@pytest.mark.parametrize("target, clip_score, iso", CASES)
def test_cmcd_kl_gradient_matches_finite_differences(target, clip_score, iso):
    p = _problem(target, clip_score, iso)
    x0, noise = _inputs()
    loss, du, grads, _ = CKO.kl_loss_and_grads(p, x0, noise, dtype=torch.float64)
    assert torch.isfinite(loss) and du.shape == (K + 1, B, D) and du.abs().max() > 0
    for name, idx in PROBES:
        vals = []
        for sgn in (1.0, -1.0):
            sd = {k: t.clone().double() for k, t in p["ctrl"]["sd"].items()}
            sd[name][idx] += sgn * 1e-6
            vals.append(CKO.kl_loss_and_grads(dict(p, ctrl=dict(p["ctrl"], sd=sd)), x0, noise, dtype=torch.float64)[0].item())
        fd = (vals[0] - vals[1]) / 2e-6
        assert abs(grads[name][idx].item() - fd) <= 1e-6 * max(1.0, abs(fd)), (name, grads[name][idx].item(), fd)


@pytest.mark.parametrize("target, clip_score, iso", CASES)
def test_cmcd_adjoint_recursion_matches_autograd(target, clip_score, iso):
    p = _problem(target, clip_score, iso)
    x0, noise = _inputs()
    _, du, _, rnd = CKO.kl_loss_and_grads(p, x0, noise, dtype=torch.float64)
    assert rnd.isfinite().all()
    ubar = CKO.adjoint_recursion(p, x0, noise, 1.0 / B)
    assert (ubar - du).abs().max() <= 1e-12 * du.abs().max()


def test_cmcd_drift_clip_is_active_in_the_clipped_cases():
    """The clipped cases above exercise the mask of the drift clip: some drift coordinates exceed it."""
    from oracle import rollout_oracle as O
    for target in ("gmm", "phi4"):
        p = _problem(target, 0.8, False)
        x0, _ = _inputs()
        _, _, _, drift, _ = CKO._parts(dict(p, clip_score=None), torch.float64)
        raw = drift(torch.tensor(0.5, dtype=torch.float64), x0)
        assert (raw.abs() > 0.8).any() and (raw.abs() < 0.8).any()
        assert O.clip(raw, 0.8).abs().max() <= 0.8


def test_cmcd_kl_and_kl_ito_are_the_same_objective():
    p = _problem("gmm", 0.8, False)
    x0, noise = _inputs()
    a = CKO.kl_loss_and_grads(p, x0, noise, "kl", dtype=torch.float64)
    b = CKO.kl_loss_and_grads(p, x0, noise, "kl_ito", dtype=torch.float64)
    assert a[0].item() == b[0].item() and torch.equal(a[1], b[1])
    assert all(torch.equal(a[2][k], b[2][k]) for k in a[2])
