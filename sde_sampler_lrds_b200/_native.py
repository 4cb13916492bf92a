"""ctypes binding of liblrds_b200.so (C ABI in include/lrds_b200.h) and its in-tree build.

There is no CPU fallback: importing this module without the built library, or calling into it with
tensors that are not on a CUDA device, raises.  The library is built in-tree by ``build()`` (nvcc,
sm_100a) so that it travels with the repository snapshot to the GPU box.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import threading

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
CSRC = os.path.join(HERE, "csrc")
# LRDS_B200_LIB: another build of the same library (A/B timing of kernel variants by the tools; same C ABI)
LIB_PATH = os.environ.get("LRDS_B200_LIB") or os.path.join(CSRC, "liblrds_b200.so")
INCLUDE = os.path.join(os.path.dirname(HERE), "include")

ABI_VERSION = 11
CHANNELS = 64
STEP_STRIDE = 80
(STEP_A, STEP_B, STEP_C, STEP_DT, STEP_SQRT_DT, STEP_W_COST, STEP_W_ITO, STEP_GAMMA, STEP_FRAC, STEP_SIGU,
 STEP_EU_A, STEP_EU_B, STEP_EU_C, STEP_CX, STEP_LERP, STEP_GSCALE) = range(16)
STEP_BIAS1 = 16

ROLLOUT_LINEAR, ROLLOUT_CMCD, ROLLOUT_EUBO_LINEAR, ROLLOUT_EUBO_CMCD = range(4)
UPDATE_AXPY, UPDATE_EM = range(2)
ITO_NONE, ITO_SCALED, ITO_EM, ITO_DDS = range(4)
CTRL_CLIPPED, CTRL_SCORE, CTRL_CANCEL_DRIFT, CTRL_LERP = range(4)
DISTR_NONE, DISTR_GMM, DISTR_PHI4, DISTR_LOGREG = range(4)
GMM_DIAG, GMM_FULL = range(2)
MCMC_MALA, MCMC_RWMH = 0, 1
PRECISION_FP32_SIMT, PRECISION_TF32X3, PRECISION_BF16, PRECISION_TF32, PRECISION_F16X3 = range(5)
PRECISIONS = {"fp32": PRECISION_FP32_SIMT, "tf32x3": PRECISION_TF32X3, "bf16": PRECISION_BF16, "tf32": PRECISION_TF32,
              "f16x3": PRECISION_F16X3}

FP = C.c_void_p  # device pointers travel as integers


class Mlp(C.Structure):
    _fields_ = [("d", C.c_int32), ("d_pad", C.c_int32), ("num_hidden", C.c_int32), ("reserved", C.c_int32),
                ("w_in_t", FP), ("w_hid_t", FP), ("b_hid", FP), ("w_out_t", FP), ("b_out", FP), ("tc_image", FP)]


class Gmm(C.Structure):
    _fields_ = [("M", C.c_int32), ("layout", C.c_int32), ("logc", FP), ("mu", FP), ("ivar", FP), ("sn", FP),
                ("step_stride_logc", C.c_int64), ("step_stride_param", C.c_int64), ("step_stride_sn", C.c_int64),
                ("mix_tc", FP), ("step_stride_mix_tc", C.c_int64)]


class Phi4(C.Structure):
    _fields_ = [("a", C.c_float), ("b", C.c_float), ("beta", C.c_float), ("reserved", C.c_float)]


class LogReg(C.Structure):
    _fields_ = [("N", C.c_int32), ("p", C.c_int32), ("n_pad", C.c_int32), ("reserved", C.c_int32),
                ("X", FP), ("Xt", FP), ("y", FP),
                ("weight_scale", C.c_float), ("intercept_mean", C.c_float), ("intercept_scale", C.c_float),
                ("threshold", C.c_float), ("eps", C.c_float), ("reserved2", C.c_float), ("x_tc", FP)]


class Distr(C.Structure):
    _fields_ = [("kind", C.c_int32), ("reserved", C.c_int32), ("gmm", Gmm), ("phi4", Phi4), ("logreg", LogReg)]


class Spec(C.Structure):
    _fields_ = [("abi_version", C.c_int32), ("kind", C.c_int32), ("update_form", C.c_int32), ("ito_form", C.c_int32),
                ("ctrl_kind", C.c_int32), ("precision", C.c_int32), ("B", C.c_int32), ("d", C.c_int32),
                ("K", C.c_int32), ("has_ref_ctrl", C.c_int32),
                ("clip_model", C.c_float), ("clip_score", C.c_float), ("scale_score", C.c_float),
                ("clip_target", C.c_float), ("cmcd_diff", C.c_float), ("cmcd_clip", C.c_float),
                ("init_cost", C.c_int32), ("rnd_offset", C.c_float),
                ("steps", FP), ("mlp", Mlp), ("target", Distr), ("ref_t", Gmm), ("ref_0", Gmm), ("status", FP)]


EXPORTS = ["lrds_rollout", "lrds_adjoint", "lrds_adjoint_cmcd", "lrds_tc_image_bytes", "lrds_gmm_mix_tc_bytes", "lrds_pack_gmm_mix_tc", "lrds_logreg_tc_bytes",
           "lrds_pack_logreg_tc", "lrds_pack_mlp_tc", "lrds_estimator_blocks", "lrds_estimator_partials", "lrds_estimator_merge", "lrds_ctrl_forward",
           "lrds_distr_eval", "lrds_axpy_step", "lrds_normals", "lrds_mala", "lrds_mlp_grad", "lrds_mlp_grad_floats",
           "lrds_mlp_grad_scratch_floats", "lrds_score_cot_sums", "lrds_score_cot_scratch_floats",
           "lrds_last_error", "lrds_abi_version",
           "lrds_launch_count"]

COMPILE_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-O3", "-lineinfo", "-std=c++17",
                 "-Xcompiler", "-fPIC"]
LINK_FLAGS = ["-gencode", "arch=compute_100a,code=sm_100a", "-shared", "-Xcompiler", "-fPIC"]


def build(force: bool = False, verbose: bool = False, extra_flags=(), out: str | None = None) -> str:
    """Compiles csrc/*.cu into csrc/liblrds_b200.so for sm_100a (cross-compiles without a GPU).
    ``extra_flags`` / ``out``: instrumented builds of the tools (e.g. -DLRDS_MIX_TIMING) under another file name."""
    srcs = [os.path.join(CSRC, f) for f in sorted(os.listdir(CSRC)) if f.endswith((".cu", ".cuh", ".h"))]
    srcs.append(os.path.join(INCLUDE, "lrds_b200.h"))
    lib_path = out or os.path.join(CSRC, "liblrds_b200.so")
    if not force and os.path.exists(lib_path) and all(os.path.getmtime(lib_path) >= os.path.getmtime(s) for s in srcs):
        return lib_path
    units = [f for f in sorted(os.listdir(CSRC)) if f.endswith(".cu")]
    objs, procs = [], []
    tag = "" if out is None else "." + os.path.basename(out)
    for u in units:  # one nvcc per translation unit, in parallel
        obj = os.path.join(CSRC, u[:-3] + tag + ".o")
        cmd = ["nvcc", *COMPILE_FLAGS, *extra_flags, "-I", INCLUDE, "-c", "-o", obj, os.path.join(CSRC, u)]
        if verbose:
            cmd.insert(1, "-Xptxas=-v")
        procs.append((u, subprocess.Popen(cmd, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True)))
        objs.append(obj)
    log = ""
    for u, p in procs:
        out, _ = p.communicate()
        log += out
        if p.returncode != 0:
            raise RuntimeError(f"nvcc failed on {u}:\n" + out)
    res = subprocess.run(["nvcc", *LINK_FLAGS, "-o", lib_path, *objs], capture_output=True, text=True)
    if res.returncode != 0:
        raise RuntimeError("link failed:\n" + res.stdout + res.stderr)
    for o in objs:  # only the .so travels with the repository snapshot
        os.remove(o)
    if verbose:
        print(log)
    return lib_path


_lib = None
_lock = threading.Lock()


def lib():
    """The loaded library; raises if it has not been built (no fallback of any kind)."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise RuntimeError(
                        f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                        "(sde_sampler_lrds_b200 has no CPU or PyTorch fallback for the rollout).")
                L = C.CDLL(LIB_PATH)
                L.lrds_last_error.restype = C.c_char_p
                L.lrds_launch_count.restype = C.c_int64
                L.lrds_rollout.argtypes = [C.POINTER(Spec), FP, FP, C.c_uint64, C.c_uint64, FP, FP, FP, FP]
                L.lrds_adjoint.argtypes = [C.POINTER(Spec), FP, FP, C.c_uint64, C.c_uint64, FP, FP, FP]
                L.lrds_adjoint_cmcd.argtypes = [C.POINTER(Spec), FP, FP, C.c_uint64, C.c_uint64, FP, FP, FP]
                L.lrds_tc_image_bytes.restype = C.c_int64
                L.lrds_tc_image_bytes.argtypes = [C.c_int32, C.c_int32, C.c_int32]
                L.lrds_pack_mlp_tc.argtypes = [C.POINTER(Mlp), C.c_int32, FP, FP]
                L.lrds_estimator_blocks.argtypes = [C.c_int32]
                L.lrds_estimator_partials.argtypes = [FP, C.c_int32, FP, FP, FP]
                L.lrds_gmm_mix_tc_bytes.restype = C.c_int64
                L.lrds_gmm_mix_tc_bytes.argtypes = [C.c_int32, C.c_int32]
                L.lrds_pack_gmm_mix_tc.argtypes = [C.POINTER(Gmm), C.c_int32, C.c_int32, C.c_int32, FP, FP]
                L.lrds_logreg_tc_bytes.restype = C.c_int64
                L.lrds_logreg_tc_bytes.argtypes = [C.c_int32, C.c_int32]
                L.lrds_pack_logreg_tc.argtypes = [C.POINTER(LogReg), C.c_int32, FP, FP]
                L.lrds_estimator_merge.argtypes = [FP, C.c_int32, FP, FP]
                L.lrds_ctrl_forward.argtypes = [C.POINTER(Spec), C.c_int32, FP, C.c_int32, FP, FP]
                L.lrds_distr_eval.argtypes = [C.POINTER(Distr), C.c_int32, FP, C.c_int32, FP, FP, FP]
                L.lrds_axpy_step.argtypes = [FP, FP, FP, C.c_float, C.c_float, C.c_float, FP, C.c_int64, FP]
                L.lrds_mala.argtypes = [C.POINTER(Distr), C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, C.c_int32, FP, FP, FP, FP,
                                        C.c_uint64, FP, FP, FP]
                L.lrds_normals.argtypes = [C.c_uint64, C.c_uint64, C.c_int32, C.c_int32, C.c_int32, C.c_int32, FP, FP]
                L.lrds_mlp_grad_floats.restype = C.c_int64
                L.lrds_mlp_grad_floats.argtypes = [C.c_int32, C.c_int32]
                L.lrds_mlp_grad_scratch_floats.restype = C.c_int64
                L.lrds_mlp_grad_scratch_floats.argtypes = [C.c_int32, C.c_int32, C.c_int32, C.c_int32]
                L.lrds_mlp_grad.argtypes = [C.POINTER(Mlp), FP, FP, FP, FP, FP, C.c_float, C.c_float, FP, C.c_int32, C.c_int32,
                                            FP, FP, FP, FP]
                L.lrds_score_cot_scratch_floats.restype = C.c_int64
                L.lrds_score_cot_scratch_floats.argtypes = [C.POINTER(Distr), C.c_int32, C.c_int32, C.c_int32]
                L.lrds_score_cot_sums.argtypes = [C.POINTER(Distr), C.c_int32, FP, FP, FP, FP, C.c_float, C.c_int32, C.c_int32,
                                                  FP, FP, FP]
                if L.lrds_abi_version() != ABI_VERSION:
                    raise RuntimeError("liblrds_b200.so ABI version mismatch; rebuild")
                _lib = L
    return _lib


class LrdsError(RuntimeError):
    pass


def check(code: int):
    if code != 0:
        msg = lib().lrds_last_error().decode()
        if code == -2:
            raise NotImplementedError(f"lrds_b200: {msg}")
        raise LrdsError(f"lrds_b200 error {code}: {msg}")


def ptr(t: torch.Tensor | None):
    """Device pointer of a contiguous float32 (or float64 for partials) CUDA tensor; None -> NULL."""
    if t is None:
        return None
    if not t.is_cuda:
        raise LrdsError("sde_sampler_lrds_b200 runs on CUDA tensors only (no CPU fallback); got a CPU tensor")
    if not t.is_contiguous():
        raise LrdsError("tensor must be contiguous")
    return C.c_void_p(t.data_ptr())


def seed_arg(seed: int):
    """A Philox seed as the ABI's uint64 (taken modulo 2^64)."""
    return C.c_uint64(seed & (2 ** 64 - 1))


def stream_ptr(device=None):
    return C.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def launch_count() -> int:
    return int(lib().lrds_launch_count())
