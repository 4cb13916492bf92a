"""CPU: the pathwise-gradient reference (tests/kl_oracle.py) against fp64 central finite differences of its own loss, on
small problems of every linear loss class: the parameter gradients it returns are the derivative of the loss it returns."""
import pytest
import torch

from tests import kl_oracle as KO
from tests.cases import BM, VP10, ctrl, many_modes, uniform_ts

D, K, B = 3, 6, 5


def _problem(kind):
    tgt = many_modes(2, D)
    c = ctrl(D, "clipped", seed=5, out_gain=1.0, num_hidden=1)
    if kind == "ei_gmm":
        ref = {"kind": "gmm", "means": tgt["loc"] + 0.1, "variances": 1.3 * tgt["scale"] ** 2, "weights": tgt["weights"].clone()}
        return {"method": "ei", "sde": VP10, "ts": uniform_ts(1.0, K), "target": tgt, "ctrl": c, "ref": ref}
    if kind == "ddpm_gauss":
        ref = {"kind": "gauss", "mean": 0.2 * torch.ones(D), "var": 1.5 * torch.ones(D)}
        return {"method": "ddpm", "sde": VP10, "ts": uniform_ts(1.0 - 1e-3, K, start=1e-3), "target": tgt, "ctrl": c, "ref": ref}
    if kind == "em_pis":
        return {"method": "em", "sde": BM, "ts": uniform_ts(5.0, K), "target": tgt, "ctrl": c,
                "ref": {"kind": "pis", "loc": torch.zeros(D)}}
    if kind == "dds":
        return {"method": "dds", "sde": None, "alpha": 1.0, "sigma": 2.0, "ts": uniform_ts(2.0, K), "target": tgt, "ctrl": c,
                "ref": {"kind": "iso", "loc": 0.0, "scale": 2.0}}
    return {"method": "dis", "sde": VP10, "ts": uniform_ts(1.0, K), "target": tgt, "ctrl": c,
            "ref": {"kind": "iso", "loc": 0.0, "scale": 1.0}}


PROBES = [("base_model.out_layer.weight", (1, 7)), ("base_model.out_layer.bias", (2,)),
          ("base_model.hidden_layer.0.weight", (4, 9)), ("base_model.input_embed.weight", (11, 0)),
          ("base_model.timestep_embed.out_layer.weight", (3, 5)), ("base_model.timestep_embed.timestep_phase", (0, 6))]


@pytest.mark.parametrize("kind, method", [("ei_gmm", "kl"), ("ddpm_gauss", "kl"), ("em_pis", "kl"), ("dds", "kl"),
                                          ("dds", "kl_ito"), ("dis", "kl"), ("dis", "kl_ito")])
def test_pathwise_gradient_matches_finite_differences(kind, method):
    problem = _problem(kind)
    g = torch.Generator().manual_seed(3)
    x0 = torch.randn(B, D, generator=g, dtype=torch.float64)
    if kind == "em_pis":
        x0 = torch.zeros(B, D, dtype=torch.float64)
    noise = torch.randn(K, B, D, generator=g, dtype=torch.float64)
    loss, dg, grads, _ = KO.kl_loss_and_grads(problem, x0, noise, method, dtype=torch.float64)
    assert dg.shape == (K, B, D) and torch.isfinite(dg).all() and dg.abs().max() > 0
    eps = 1e-6
    for name, idx in PROBES:
        vals = []
        for sign in (1.0, -1.0):
            sd = {k: v.clone().double() for k, v in problem["ctrl"]["sd"].items()}
            sd[name][idx] += sign * eps
            p = dict(problem, ctrl=dict(problem["ctrl"], sd=sd))
            vals.append(KO.kl_loss_and_grads(p, x0, noise, method, dtype=torch.float64)[0].item())
        fd = (vals[0] - vals[1]) / (2 * eps)
        got = grads[name][idx].item()
        assert abs(got - fd) <= 1e-6 * max(1.0, abs(fd)), (name, got, fd)


def test_dis_kl_ito_differs_from_kl_only_by_the_ito_term():
    """'kl' leaves the Ito integral out of the DIS training log-weight, 'kl_ito' keeps it: with zero increments the two
    coincide."""
    problem = _problem("dis")
    x0 = torch.randn(B, D, generator=torch.Generator().manual_seed(4), dtype=torch.float64)
    zero = torch.zeros(K, B, D, dtype=torch.float64)
    a = KO.kl_loss_and_grads(problem, x0, zero, "kl", dtype=torch.float64)
    b = KO.kl_loss_and_grads(problem, x0, zero, "kl_ito", dtype=torch.float64)
    assert torch.allclose(a[3], b[3]) and torch.allclose(a[1], b[1])
    noise = torch.randn(K, B, D, generator=torch.Generator().manual_seed(5), dtype=torch.float64)
    assert not torch.allclose(KO.kl_loss_and_grads(problem, x0, noise, "kl", dtype=torch.float64)[3],
                              KO.kl_loss_and_grads(problem, x0, noise, "kl_ito", dtype=torch.float64)[3])
