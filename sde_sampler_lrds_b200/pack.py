"""Host-side packing of a rollout into the C ABI's ``lrds_spec``: introspection of the reference-style Python
objects (control module, SDE, target / reference distributions), the per-step coefficient table and the
weight buffers.  Everything here is O(K) or O(#weights) host work; per-particle arithmetic lives in csrc/.

Objects that have no kernel raise NotImplementedError - there is no silent CPU / PyTorch fallback
(BASELINE.json north_star; SURVEY.md 8b).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import torch

from . import _native as N
from .distr.base import Distribution, fill_gmm, gmm_block
from .distr.gauss import GMM, GMMFull
from .models.mlp import FourierMLP, TimeEmbed
from .models.reparam import CancelDriftCtrl, ClippedCtrl, LerpCtrl, ScoreCtrl

_DEFAULT_PRECISION = "f16x3"


def set_default_precision(name: str):
    """'f16x3' (default: tcgen05 with the 3-pass fp16 split, fp32-grade), 'tf32x3' (the same with tf32 operands),
    'fp32' (SIMT parity anchor), or the reduced-precision fast modes 'tf32' / 'bf16'."""
    global _DEFAULT_PRECISION
    if name not in N.PRECISIONS:
        raise ValueError(f"unknown precision {name!r}")
    _DEFAULT_PRECISION = name


def default_precision() -> str:
    return _DEFAULT_PRECISION


# --------------------------------------------------------------------------------------------------------------
# introspection
# --------------------------------------------------------------------------------------------------------------
@dataclass
class CtrlInfo:
    kind: int
    base: FourierMLP
    score_model: TimeEmbed | None = None
    target: Distribution | None = None
    clip_model: float | None = None
    clip_score: float | None = None
    scale_score: float = 1.0
    sde: object | None = None              # CancelDriftCtrl / LerpCtrl: the OU SDE of their time-only coefficients
    prior: Distribution | None = None      # LerpCtrl: the prior whose score is interpolated


def resolve_ctrl(ctrl) -> CtrlInfo:
    """Accepts FourierMLP, ClippedCtrl, ScoreCtrl (optionally wrapped in an EMA AveragedModel)."""
    if isinstance(ctrl, torch.optim.swa_utils.AveragedModel):
        ctrl = ctrl.module
    if isinstance(ctrl, FourierMLP):
        return CtrlInfo(N.CTRL_CLIPPED, ctrl)
    if isinstance(ctrl, ScoreCtrl):
        target = getattr(ctrl.target_score, "__self__", None)
        if not isinstance(target, Distribution):
            raise NotImplementedError("ScoreCtrl.target_score must be the bound .score of a kernel-backed Distribution")
        if not isinstance(ctrl.base_model, FourierMLP):
            raise NotImplementedError(f"drift backbone {type(ctrl.base_model).__name__} has no B200 kernel")
        if ctrl.score_model is not None and not (isinstance(ctrl.score_model, TimeEmbed) and ctrl.score_model.dim_out == 1):
            raise NotImplementedError("score_model must be a TimeEmbed with dim_out=1 (conf/model/score.yaml)")
        info = CtrlInfo(N.CTRL_SCORE, ctrl.base_model, ctrl.score_model, target, ctrl.clip_model, ctrl.clip_score,
                        float(ctrl.scale_score))
        if isinstance(ctrl, CancelDriftCtrl):
            info.kind, info.sde = N.CTRL_CANCEL_DRIFT, ctrl.sde
        elif isinstance(ctrl, LerpCtrl):
            prior = getattr(ctrl.prior_score, "__self__", None)
            if not isinstance(prior, GMM) or prior.loc.shape[0] != 1:
                raise NotImplementedError("LerpCtrl.prior_score must be the bound .score of a diagonal Gaussian prior")
            info.kind, info.sde, info.prior = N.CTRL_LERP, ctrl.sde, prior
        elif type(ctrl) is not ScoreCtrl:
            raise NotImplementedError(f"control of type {type(ctrl).__name__} has no B200 kernel (no fallback is provided)")
        return info
    if isinstance(ctrl, ClippedCtrl):
        if not isinstance(ctrl.base_model, FourierMLP):
            raise NotImplementedError(f"drift backbone {type(ctrl.base_model).__name__} has no B200 kernel")
        return CtrlInfo(N.CTRL_CLIPPED, ctrl.base_model, clip_model=ctrl.clip_model)
    raise NotImplementedError(f"control of type {type(ctrl).__name__} has no B200 kernel (no fallback is provided)")


def resolve_log_prob(fn):
    """(Distribution, clip) behind a log-density callable: a bound ``unnorm_log_prob`` / ``log_prob`` of a
    Distribution, or a solver's ``clipped_target_unnorm_log_prob`` (solver/oc.py:80-87)."""
    owner = getattr(fn, "__self__", None)
    if isinstance(owner, Distribution):
        if fn.__name__ == "log_prob" and owner.log_norm_const not in (0, 0.0):
            raise NotImplementedError("log_prob with a non-zero log_norm_const is not used by the rollout solvers")
        return owner, None
    if owner is not None and hasattr(owner, "target") and isinstance(owner.target, Distribution):
        return owner.target, getattr(owner, "clip_target", None)
    raise NotImplementedError("log-density callable must be a bound method of a kernel-backed Distribution")


def time_columns(table: torch.Tensor, info: CtrlInfo, taus: torch.Tensor):
    """Writes the parameter-dependent time-only columns of the control for times ``taus`` into the step table, evaluated
    on the table's device: bias1 [S][64] = input_embed.bias + TimeEmbed(tau) and gamma [S] = the clipped score-model
    factor (1 without one)."""
    dev = table.device
    table[:, N.STEP_BIAS1:N.STEP_BIAS1 + N.CHANNELS] = info.base.bias_rows(taus, dev)
    if info.kind != N.CTRL_CLIPPED and info.score_model is not None:
        gamma = info.score_model.rows(taus, dev).reshape(-1)
        table[:, N.STEP_GAMMA] = gamma if info.clip_model is None else gamma.clip(-info.clip_model, info.clip_model)
    else:
        table[:, N.STEP_GAMMA] = 1.0


def dis_ctrl_rows(info: CtrlInfo, taus: torch.Tensor, table: torch.Tensor):
    """Time-only coefficients of CancelDriftCtrl / LerpCtrl (models/reparam.py:131-147, 189-199) in the reference's
    float32 scalar formulas: columns STEP_CX, STEP_LERP, STEP_GSCALE of the per-step table."""
    if info.kind not in (N.CTRL_CANCEL_DRIFT, N.CTRL_LERP):
        return
    sde = info.sde.host()
    for k, t in enumerate(taus.detach().to("cpu", torch.float32).reshape(-1)):
        sig = sde.diff(t)
        if info.kind == N.CTRL_CANCEL_DRIFT:
            table[k, N.STEP_CX], table[k, N.STEP_GSCALE] = sde.drift_coeff_t(t) / sig, 0.5 * sig
        else:
            table[k, N.STEP_LERP], table[k, N.STEP_GSCALE] = t / sde.terminal_t, sig


def fill_ctrl(spec: N.Spec, info: CtrlInfo, device, keep: list, prior: Distribution | None = None):
    """Fills the control's fields of the spec and returns the keepalive of the weight block spec.mlp points into
    (Plan.weights).  ``prior`` = the distribution that fills spec.ref_0 when it is the rollout's prior (DIS); LerpCtrl
    needs it."""
    if info.kind == N.CTRL_LERP and prior is not info.prior:
        raise NotImplementedError("LerpCtrl runs in the DIS rollout from the prior whose score it interpolates "
                                  "(TimeReversalLoss with initial_log_prob = that prior's log_prob)")
    spec.ctrl_kind = info.kind
    spec.clip_model = float(info.clip_model) if info.clip_model is not None else 0.0
    spec.clip_score = float(info.clip_score) if info.clip_score is not None else 0.0
    spec.scale_score = float(info.scale_score)
    mlp, weights = info.base.lrds_mlp(device, spec.precision)
    spec.mlp = mlp
    spec.d = info.base.dim
    if info.target is not None:
        if info.target.dim != info.base.dim:
            raise ValueError("target and drift network dimensions differ")
        distr, k2 = info.target.lrds_distr(device)
        spec.target = distr
        keep.append(k2)
    return weights


def new_spec(precision: str | None = None) -> N.Spec:
    s = N.Spec()
    s.abi_version = N.ABI_VERSION
    s.precision = N.PRECISIONS[precision or _DEFAULT_PRECISION]
    return s


def ctrl_forward(module, t: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
    """u = module(t, x) for a drift model (FourierMLP / ClippedCtrl / ScoreCtrl) through lrds_ctrl_forward."""
    if not x.is_cuda:
        raise N.LrdsError("drift models run on CUDA tensors only (no CPU fallback)")
    info = resolve_ctrl(module)
    keep: list = []
    spec = new_spec("fp32")
    keep.append(fill_ctrl(spec, info, x.device, keep, prior=info.prior))
    if info.kind == N.CTRL_LERP:
        fill_ref0(spec, info.prior, x.device, keep)
    t = torch.as_tensor(t)
    if t.numel() != 1:
        if not bool((t.reshape(-1) == t.reshape(-1)[0]).all()):
            raise NotImplementedError("drift models are evaluated at one time per call (as every solver does)")
        t = t.reshape(-1)[0]
    table = finish_table(torch.zeros(1, N.STEP_STRIDE), info, t.reshape(1), x.device)
    spec.steps = table.data_ptr()
    lead = x.shape[:-1]
    xf = x.detach().reshape(-1, spec.d).to(torch.float32).contiguous()
    spec.B, spec.K = xf.shape[0], 1
    out = torch.empty_like(xf)
    with torch.cuda.device(x.device):
        N.check(N.lib().lrds_ctrl_forward(C.byref(spec), 0, N.ptr(xf), xf.shape[0], N.ptr(out), N.stream_ptr(x.device)))
    return out.reshape(*lead, spec.d)


# --------------------------------------------------------------------------------------------------------------
# a packed rollout
# --------------------------------------------------------------------------------------------------------------
@dataclass
class Plan:
    spec: N.Spec
    keep: list                          # the further buffers the spec points into (target, reference and prior blocks)
    weights: object                     # the weight block / tensor-core image spec.mlp points into (fill_ctrl, refresh_ctrl)
    steps: torch.Tensor                 # [rows, STEP_STRIDE] device: the step table spec.steps points at (finish_table)
    rows: int = 0
    noise_steps: int = 0
    taus: torch.Tensor | None = None    # [rows] host: the time the control is evaluated at in row k (finish_table, train.py)
    ito_w: torch.Tensor | None = None   # [K] host: the weight of <g, z> in the log-weight of step k
    dev_cache: dict = field(default_factory=dict)  # device copies of host-side rows, made once per plan (on_device)


def on_device(plan: "Plan", name: str, device, make=None) -> torch.Tensor:
    """Device copy of a host tensor of the plan (``plan.<name>`` or ``make()``), cached: a pageable host-to-device copy
    synchronises the stream, which a training step must not do once per step."""
    key = (name, str(device))
    if key not in plan.dev_cache:
        src = getattr(plan, name) if make is None else make()
        plan.dev_cache[key] = src.to(device)
    return plan.dev_cache[key]


def ito_weights(table: torch.Tensor, ito_form: int) -> torch.Tensor:
    """Per-step weight of sum(g z) in rnd for the LINEAR loops (include/lrds_b200.h, lrds_ito_form)."""
    if ito_form == N.ITO_SCALED:
        return table[:, N.STEP_W_ITO].clone()
    if ito_form == N.ITO_EM:
        return table[:, N.STEP_SQRT_DT].clone()
    if ito_form == N.ITO_DDS:
        return table[:, N.STEP_SIGU] * table[:, N.STEP_W_ITO]
    return torch.zeros(table.shape[0])


def _scalar_rows(ts: torch.Tensor):
    ts = ts.detach().to("cpu", torch.float32)
    return ts, list(zip(ts[:-1], ts[1:]))


def fill_ref0(spec: N.Spec, distr: Distribution, device, keep: list, single_gaussian: str | None = None):
    """Fills spec.ref_0 (the RDS / DDS reference term, the CMCD / DIS prior, LerpCtrl's prior) from the (logc, mu, ivar)
    block of a diagonal Gaussian / mixture Distribution, or the FullBlock of a full-covariance one (GaussFull / GMMFull:
    the RDS reference term; the CMCD / DIS priors and LerpCtrl are refused for it by the library).
    ``single_gaussian``: the refusal raised when ``distr`` has more than one component."""
    if isinstance(distr, GMMFull):
        blk = distr.block(device)
    elif isinstance(distr, GMM):
        blk = gmm_block(distr.loc, torch.square(distr.scale), distr.mixture_weights, device)
    else:
        raise NotImplementedError(f"{type(distr).__name__} cannot serve as a Gaussian reference / prior here")
    if single_gaussian is not None and blk[1].shape[0] != 1:
        raise NotImplementedError(single_gaussian)
    fill_gmm(spec.ref_0, blk)
    keep.append(blk)


def finish_table(table: torch.Tensor, info: CtrlInfo, taus: torch.Tensor, device) -> torch.Tensor:
    """The host step table with the control's time-only columns for times ``taus`` written in, copied to ``device``."""
    time_columns(table, info, taus)
    dis_ctrl_rows(info, taus, table)
    return table.contiguous().to(device)


def refresh_ctrl(plan: "Plan", info: CtrlInfo, device):
    """Re-packs what depends on the control's parameters into a cached plan: the weight block / tensor-core image and
    the TimeEmbed columns of the device table (bias rows, gamma) at the plan's times, in place and ordered on the
    current stream behind earlier launches that read them.  The rows are evaluated on the device here (no parameter
    round trip through the host in a training step); a freshly built plan evaluates them with the same torch ops on the
    host, which agrees to float32 rounding."""
    plan.spec.mlp, plan.weights = info.base.lrds_mlp(device, plan.spec.precision)
    time_columns(plan.steps, info, on_device(plan, "taus", plan.steps.device))


_status: dict = {}


def status_counters(device) -> torch.Tensor:
    """The device's two rollout status counters (lrds_spec.status): [0] particle threads whose fp16 tensor-core operands
    saturated (f16x3: |coordinate| > 65504 or a hidden pre-activation > 1023), [1] particles with a non-finite result.
    Every rollout launched from this process ADDS to them; ``read_status`` returns and optionally clears them."""
    dev = torch.device(device)
    key = (dev.type, dev.index if dev.index is not None else torch.cuda.current_device())
    if key not in _status:
        _status[key] = torch.zeros(2, dtype=torch.int32, device=dev)
    return _status[key]


def read_status(device, reset: bool = True) -> dict:
    """{'saturated': n, 'nonfinite': n} accumulated by the rollouts on ``device`` since the last reset (synchronises)."""
    t = status_counters(device)
    sat, nf = (int(v) for v in t.cpu())
    if reset:
        t.zero_()
    return {"saturated": sat, "nonfinite": nf}


def run_rollout(plan: Plan, x0: torch.Tensor, noise: torch.Tensor | None, seed: int, particle_offset: int,
                return_traj: bool):
    """Launches lrds_rollout for ``plan`` on x0's device; returns (x_T, rnd (B,1), xs | None)."""
    if not x0.is_cuda:
        raise N.LrdsError("the rollout runs on CUDA tensors only (no CPU fallback)")
    dev = x0.device
    xf = x0.detach().to(torch.float32).contiguous()
    B, d = xf.shape
    if d != plan.spec.d:
        raise ValueError(f"x has dimension {d}, the model expects {plan.spec.d}")
    spec = N.Spec.from_buffer_copy(plan.spec)  # the cached plan is shared between calls (and threads): never mutated here
    spec.B = B
    status = status_counters(dev)
    spec.status = status.data_ptr()
    if noise is not None:
        noise = noise.detach().to(dev, torch.float32).contiguous()
        if tuple(noise.shape) != (plan.noise_steps, B, d):
            raise ValueError(f"noise must have shape {(plan.noise_steps, B, d)}, got {tuple(noise.shape)}")
    x_out = torch.empty_like(xf)
    rnd = torch.empty(B, device=dev, dtype=torch.float32)
    traj = torch.empty(spec.K + 1, B, d, device=dev, dtype=torch.float32) if return_traj else None
    with torch.cuda.device(dev):
        N.check(N.lib().lrds_rollout(C.byref(spec), N.ptr(xf), N.ptr(noise), N.seed_arg(seed),
                                     C.c_uint64(particle_offset), N.ptr(x_out), N.ptr(rnd), N.ptr(traj),
                                     N.stream_ptr(dev)))
    return x_out, rnd.unsqueeze(-1), traj
