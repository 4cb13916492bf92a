"""CPU: the C-ABI library builds, loads, and exports every symbol include/lrds_b200.h declares; argument
validation answers without a GPU."""
import ctypes as C
import math
import os
import re

from sde_sampler_lrds_b200 import _native as N

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol():
    N.build()
    lib = N.lib()
    header = open(os.path.join(ROOT, "include", "lrds_b200.h")).read()
    declared = set(re.findall(r"^(?:int|int64_t|const char\*)\s+(lrds_[a-z_0-9]+)\s*\(", header, flags=re.M))
    assert declared == set(N.EXPORTS), declared ^ set(N.EXPORTS)
    for name in declared:
        assert hasattr(lib, name), name
    assert lib.lrds_abi_version() == N.ABI_VERSION


def test_struct_sizes_match_header():
    # field-by-field mirror of include/lrds_b200.h (natural alignment, no packing pragmas)
    assert C.sizeof(N.Mlp) == 16 + 6 * 8
    assert C.sizeof(N.Gmm) == 8 + 4 * 8 + 24 + 16
    assert C.sizeof(N.Phi4) == 16
    assert C.sizeof(N.LogReg) == 16 + 24 + 24 + 8
    assert C.sizeof(N.Distr) == 8 + C.sizeof(N.Gmm) + C.sizeof(N.Phi4) + C.sizeof(N.LogReg)
    assert C.sizeof(N.Spec) == 40 + 24 + 8 + 8 + C.sizeof(N.Mlp) + C.sizeof(N.Distr) + 2 * C.sizeof(N.Gmm) + 8  # + status


def test_invalid_arguments_are_rejected_without_a_gpu():
    lib = N.lib()
    assert lib.lrds_rollout(None, None, None, 0, 0, None, None, None, None) == -1
    assert b"NULL" in lib.lrds_last_error()
    spec = N.Spec()
    spec.abi_version = 99
    assert lib.lrds_rollout(C.byref(spec), None, None, 0, 0, None, None, None, None) == -1
    assert b"got 99" in lib.lrds_last_error()
    assert lib.lrds_estimator_blocks(1) == 1 and lib.lrds_estimator_blocks(8193) == 2
    assert lib.lrds_estimator_partials(None, 0, None, None, None) == -1

    # the bare-distribution entry points: arguments, then the distribution (no pointer is dereferenced on these paths)
    p = 256  # dummy device pointer
    d = 4

    def distr_eval(distr, B=8, x=p):
        return lib.lrds_distr_eval(C.byref(distr) if distr else None, d, x, B, p, None, None)

    def mala(distr, C_=8, sampler=N.MCMC_MALA):
        return lib.lrds_mala(C.byref(distr) if distr else None, d, C_, 0, 4, 0, sampler, p, p, None, None, 0, p, None, None)

    def score_cot(distr, S=2):
        return lib.lrds_score_cot_scratch_floats(C.byref(distr) if distr else None, d, S, 8)

    good = N.Distr()
    good.kind = N.DISTR_PHI4
    for call, who in ((lambda: distr_eval(None), b"distr_eval"), (lambda: distr_eval(good, B=0), b"distr_eval"),
                      (lambda: distr_eval(good, x=None), b"distr_eval"), (lambda: mala(None), b"mala"),
                      (lambda: mala(good, C_=0), b"mala"), (lambda: score_cot(None), b"score_cot"),
                      (lambda: score_cot(good, S=0), b"score_cot")):
        assert call() == -1 and who in lib.lrds_last_error()
    none = N.Distr()
    none.kind = N.DISTR_NONE
    assert distr_eval(none) == -2 and mala(none) == -2 and score_cot(none) == -2
    full = N.Distr()
    full.kind = N.DISTR_GMM
    full.gmm.M, full.gmm.layout, full.gmm.logc, full.gmm.mu, full.gmm.sn = 2, N.GMM_FULL, p, p, p
    for call, who in ((lambda: score_cot(full), b"score_cot"), (lambda: mala(full), b"mala")):
        assert call() == -2 and who in lib.lrds_last_error()
    assert mala(good, sampler=7) == -1


def test_mixture_tensor_core_image_layout():
    """lrds_gmm.mix_tc (include/lrds_b200.h): B[n][m] with rows n = 16 c + i (i < 8: -1/var, i >= 8: mu/var of dim
    8 c + i % 8), power-of-two scaled, fp16 hi | lo parts in the K-major [m/8][n][m%8] layout, un-scale in the tail."""
    import torch
    from sde_sampler_lrds_b200.distr.base import gmm_mix_tc_image
    torch.manual_seed(0)
    S, M, d, dp = 3, 5, 11, 16
    loc, var = torch.randn(S, M, d) * 7, torch.rand(S, M, d) * 2 + 0.05
    w = torch.rand(M) + 0.1
    logc = -0.5 * d * math.log(2 * math.pi) - 0.5 * torch.log(var).sum(-1) + torch.log(w / w.sum())
    img = gmm_mix_tc_image(loc, var, dp, logc)
    lib = N.lib()
    lib.lrds_gmm_mix_tc_bytes.restype = C.c_int64
    nbytes = lib.lrds_gmm_mix_tc_bytes(M, dp)
    assert img.shape == (S, nbytes) and img.dtype == torch.uint8 and nbytes % 16 == 0
    Kin, Mp = 16 * ((dp + 15) // 16), 16
    lpart = Mp * Kin * 2
    contr = nbytes - (2 * lpart + 4 * Mp + 16)
    part = (contr - 16) // 2
    for s in range(S):
        unscale = img[s, 2 * part:2 * part + 4].view(torch.float32).item()
        assert unscale > 0 and math.log2(unscale) == round(math.log2(unscale))
        hi = img[s, :part].view(torch.float16).float().reshape(2, 2 * dp, 8)      # [m/8][n][m%8], M padded to 16
        lo = img[s, part:2 * part].view(torch.float16).float().reshape(2, 2 * dp, 8)
        Bm = ((hi + lo) * unscale).permute(0, 2, 1).reshape(16, 2 * dp)            # [m][n]
        assert hi.abs().max() < 2 ** 15 and hi.abs().max() >= 2 ** 14
        for m in range(16):
            for n in range(2 * dp):
                c, i = divmod(n, 16)
                j = 8 * c + i % 8
                want = 0.0 if (m >= M or j >= d) else (-1.0 / var[s, m, j] if i < 8 else loc[s, m, j] / var[s, m, j]).item()
                assert abs(Bm[m, n].item() - want) <= 2.0 ** -20 * max(abs(want), 2.0 ** -10), (s, m, n)
        # the logit image behind it: wc[j/8][m][j%8] hi | lo, c_m, {un-scale, max |wc_m|, max |c_m|, shared}
        L = img[s, contr:]
        tail = L[2 * lpart + 4 * Mp:].view(torch.float32)
        us = tail[0].item()
        assert us > 0 and math.log2(us) == round(math.log2(us)) and tail[3].item() == 0.0  # per-mode variances: not shared
        hi = L[:lpart].view(torch.float16).float().reshape(Kin // 8, Mp, 8)
        lo = L[lpart:2 * lpart].view(torch.float16).float().reshape(Kin // 8, Mp, 8)
        Wc = ((hi + lo) * us).permute(1, 0, 2).reshape(Mp, Kin)                       # [m][j]
        wfull = (loc[s].double() / var[s].double())
        want_w = wfull - wfull.mean(0, keepdim=True)
        assert (Wc[:M, :d].double() - want_w).abs().max() <= 2.0 ** -19 * want_w.abs().max()
        assert Wc[M:].abs().max() == 0 and Wc[:, d:].abs().max() == 0
        cm = L[2 * lpart:2 * lpart + 4 * Mp].view(torch.float32)
        want_c = logc[s].double() - 0.5 * (loc[s].double() ** 2 / var[s].double()).sum(-1)
        want_c = want_c - want_c.max()  # shifted by its maximum (softmax-invariant)
        assert (cm[:M].double() - want_c).abs().max() <= 1e-6 * want_c.abs().max() and torch.isinf(cm[M:]).all()
        assert abs(tail[1].item() - want_w.pow(2).sum(-1).sqrt().max().item()) <= 1e-5 * tail[1].item()
        assert abs(tail[2].item() - want_c.abs().max().item()) <= 1e-5 * tail[2].item()
    # a mixture whose modes share their variances sets the flag
    var_sh = (torch.rand(1, d) * 2 + 0.05).expand(M, d)
    logc_sh = -0.5 * torch.log(var_sh).sum(-1) + torch.log(w / w.sum())
    img2 = gmm_mix_tc_image(loc[0], var_sh, dp, logc_sh)
    assert img2[-16:].view(torch.float32)[3].item() == 1.0


def test_gradient_kernel_size_queries_without_a_gpu():
    """lrds_mlp_grad_floats / _scratch_floats are host-only queries: the layout of lrds_mlp's weight blocks, and
    LRDS_ERR_UNSUPPORTED (-2) for shapes the kernel is not built for (d > 64, more than two hidden layers)."""
    from sde_sampler_lrds_b200 import _native as N
    from sde_sampler_lrds_b200.train import pow2_scale
    L = N.lib()
    assert L.lrds_mlp_grad_floats(50, 2) == 50 * 64 + 2 * 64 * 64 + 2 * 64 + 64 * 56 + 56
    assert L.lrds_mlp_grad_floats(2, 0) == 2 * 64 + 64 * 8 + 8
    assert L.lrds_mlp_grad_floats(65, 2) == -2 and L.lrds_mlp_grad_floats(50, 3) == -2
    assert L.lrds_mlp_grad_scratch_floats(65, 2, 4, 4) == -2
    # power-of-two operand scale: bound * scale in (2, 4]
    for b in (1e-6, 0.3, 4.0, 777.0):
        s = pow2_scale(b)
        assert 2.0 < b * s <= 4.0 and s == 2.0 ** round(__import__("math").log2(s))
    assert pow2_scale(0.0) == 1.0 and pow2_scale(float("inf")) == 1.0
