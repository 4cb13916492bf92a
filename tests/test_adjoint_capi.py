"""CPU: lrds_adjoint validates its spec without a GPU - what it is not built for is LRDS_ERR_UNSUPPORTED, never a silent
fallback."""
import ctypes as C

from sde_sampler_lrds_b200 import _native as N


def _spec(p=256):
    """A LINEAR ClippedCtrl spec over a PhiFour target whose pointers are never dereferenced on the validation path."""
    s = N.Spec()
    s.abi_version, s.kind, s.ctrl_kind, s.precision = N.ABI_VERSION, N.ROLLOUT_LINEAR, N.CTRL_CLIPPED, N.PRECISION_F16X3
    s.B, s.d, s.K = 8, 4, 3
    s.mlp.d, s.mlp.d_pad, s.mlp.num_hidden = 4, 8, 2
    s.mlp.w_in_t = s.mlp.w_hid_t = s.mlp.b_hid = s.mlp.w_out_t = s.mlp.b_out = p
    s.steps = p
    s.target.kind = N.DISTR_PHI4
    s.ref_0.M, s.ref_0.logc, s.ref_0.mu, s.ref_0.ivar, s.ref_0.sn = 1, p, p, p, p
    return s


def test_adjoint_rejects_what_it_is_not_built_for_without_a_gpu():
    lib = N.lib()
    p = 256

    def call(spec):
        return lib.lrds_adjoint(None if spec is None else C.byref(spec), p, None, 0, 0, p, p, None)

    assert call(None) == N.lib().lrds_adjoint(None, None, None, 0, 0, None, None, None) == -1
    assert b"NULL" in lib.lrds_last_error()
    s = _spec()
    assert lib.lrds_adjoint(C.byref(s), None, None, 0, 0, p, p, None) == -1  # no trajectory
    for field, value, words in (("ctrl_kind", N.CTRL_SCORE, b"ClippedCtrl"), ("precision", N.PRECISION_BF16, b"reduced-precision"),
                                ("precision", N.PRECISION_TF32, b"reduced-precision"), ("kind", N.ROLLOUT_CMCD, b"LINEAR"),
                                ("kind", N.ROLLOUT_EUBO_LINEAR, b"LINEAR")):
        s = _spec()
        setattr(s, field, value)
        assert call(s) == -2, (field, value)
        assert words in lib.lrds_last_error()
    s = _spec()
    s.ref_0.layout, s.ref_0.ivar = N.GMM_FULL, None
    assert call(s) == -2 and b"full-covariance" in lib.lrds_last_error()
