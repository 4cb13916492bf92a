"""CPU: lrds_adjoint_cmcd validates its spec without a GPU - what it is not built for is LRDS_ERR_UNSUPPORTED (or
LRDS_ERR_INVALID for malformed arguments) with a message, never a silent fallback."""
import ctypes as C

from sde_sampler_lrds_b200 import _native as N

P = 256  # a pointer value that is never dereferenced on the validation path


def _spec():
    """A CMCD ClippedCtrl spec over a mixture target with a diagonal Gaussian prior."""
    s = N.Spec()
    s.abi_version, s.kind, s.ctrl_kind, s.precision = N.ABI_VERSION, N.ROLLOUT_CMCD, N.CTRL_CLIPPED, N.PRECISION_F16X3
    s.B, s.d, s.K = 8, 4, 3
    s.mlp.d, s.mlp.d_pad, s.mlp.num_hidden = 4, 8, 2
    s.mlp.w_in_t = s.mlp.w_hid_t = s.mlp.b_hid = s.mlp.w_out_t = s.mlp.b_out = P
    s.steps = P
    s.cmcd_diff = 1.0
    s.target.kind = N.DISTR_GMM
    g = s.target.gmm
    g.M, g.logc, g.mu, g.ivar, g.sn = 3, P, P, P, P
    s.ref_0.M, s.ref_0.logc, s.ref_0.mu, s.ref_0.ivar, s.ref_0.sn = 1, P, P, P, P
    return s


def _call(spec, traj=P, row_w=P, cot=P):
    return N.lib().lrds_adjoint_cmcd(None if spec is None else C.byref(spec), traj, None, 0, 0, row_w, cot, None)


def _err():
    return N.lib().lrds_last_error()


def test_adjoint_cmcd_rejects_malformed_arguments_without_a_gpu():
    assert _call(None) == -1 and b"NULL" in _err()
    for kw in (dict(traj=None), dict(row_w=None), dict(cot=None)):
        assert _call(_spec(), **kw) == -1 and b"required" in _err(), kw
    s = _spec()
    s.abi_version = 99
    assert _call(s) == -1 and b"abi_version" in _err()
    s = _spec()
    s.K = 0
    assert _call(s) == -1 and b"K must be" in _err()
    s = _spec()
    s.precision = 17
    assert _call(s) == -1 and b"precision" in _err()


def test_adjoint_cmcd_rejects_what_it_is_not_built_for_without_a_gpu():
    for field, value, words in (("kind", N.ROLLOUT_LINEAR, b"CMCD"), ("kind", N.ROLLOUT_EUBO_CMCD, b"CMCD"),
                                ("kind", N.ROLLOUT_EUBO_LINEAR, b"CMCD"), ("ctrl_kind", N.CTRL_SCORE, b"ClippedCtrl"),
                                ("precision", N.PRECISION_BF16, b"reduced-precision"),
                                ("precision", N.PRECISION_TF32, b"reduced-precision")):
        s = _spec()
        setattr(s, field, value)
        assert _call(s) == -2, (field, value)
        assert words in _err(), (field, value, _err())
    # the other controls (CancelDriftCtrl / LerpCtrl: LerpCtrl passes the common validation with its Gaussian prior)
    for kind in (N.CTRL_CANCEL_DRIFT, N.CTRL_LERP):
        s = _spec()
        s.ctrl_kind = kind
        assert _call(s) == -2 and b"ClippedCtrl" in _err(), kind
    # the logistic-regression target
    s = _spec()
    s.target.kind = N.DISTR_LOGREG
    lr = s.target.logreg
    lr.N, lr.p, lr.n_pad, lr.X, lr.Xt, lr.y = 5, 3, 8, P, P, P
    assert _call(s) == -2 and b"logistic-regression" in _err()
    # full-covariance blocks: the prior and the target
    s = _spec()
    s.ref_0.layout, s.ref_0.ivar = N.GMM_FULL, None
    assert _call(s) == -2 and b"full-covariance" in _err()
    s = _spec()
    s.target.gmm.layout, s.target.gmm.ivar = N.GMM_FULL, None
    assert _call(s) == -2 and b"full-covariance" in _err()
    # a mixture prior
    s = _spec()
    s.ref_0.M = 2
    assert _call(s) == -2 and b"Gaussian prior" in _err()
    # no target
    s = _spec()
    s.target.kind = N.DISTR_NONE
    assert _call(s) == -1 and b"target" in _err()


def test_adjoint_cmcd_accepts_the_phi4_target_up_to_the_launch():
    """A PhiFour spec passes validation: without a device the call fails at the launch (a CUDA error, not a refusal)."""
    import pytest
    import torch
    if torch.cuda.is_available():
        pytest.skip("with a device the call would launch: acceptance on a GPU is covered by tests/test_cmcd_kl_train_gpu.py")
    s = _spec()
    s.target.kind = N.DISTR_PHI4
    s.target.phi4.a, s.target.phi4.beta = 0.1, 20.0
    assert _call(s) not in (0, -1, -2)


def test_lrds_adjoint_still_refuses_cmcd_and_points_to_the_new_entry():
    s = _spec()
    assert N.lib().lrds_adjoint(C.byref(s), P, None, 0, 0, P, P, None) == -2
    assert b"LINEAR" in _err() and b"lrds_adjoint_cmcd" in _err()
