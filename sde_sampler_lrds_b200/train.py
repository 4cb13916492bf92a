"""Training objective through the fused rollout: ``loss(ts, x, ...)`` of the linear rollout losses with
method 'lv' / 'lv_traj' (sde_sampler/losses/oc.py:364-394, 1240-1272, 1399-1431 -> compute_loss 105-131), the first
version of SURVEY.md 8f item 1.

With these methods the SDE follows the DETACHED control (generative_and_sde_ctrl, oc.py:83-103), so no gradient flows
along a trajectory: the states x_k are constants and

    d rnd_b / d theta = sum_k  c_k <z_bk, d g(t_k, x_bk) / d theta>          (c_k = the Ito weight of step k)

because the running cost g (sde_ctrl - g / 2) has a vanishing derivative at sde_ctrl = g.  The reference obtains this
by autograd through K sequential steps (~40-150 eager ops each).  Here

  1. the rollout is ONE fused kernel launch (csrc/), fed with the generator's own increments z (lrds_normals) and
     returning the trajectory;
  2. d loss / d rnd comes from the reference's loss formula on the B log-weights;
  3. the parameter gradient is ONE batched pass over all K x B stored states with the cotangent
     (d loss / d rnd_b) c_k z_bk: the hand-written weight-gradient kernel lrds_mlp_grad (csrc/lrds_mlp_grad.cu: the
     activations are recomputed from the stored states on the tensor cores, the weight gradients accumulate in TMEM)
     for the backbone; what remains for autograd is K rows wide (TimeEmbed under the kernel's bias cotangent, the
     time-only score factor of ScoreCtrl).  The kernel serves the default precision "f16x3" (its weight-gradient operands
     are single fp16 roundings: gradient tensors agree with autograd to ~5e-4 of their norm, far below the Monte-Carlo
     noise of the estimate).  Shapes it is not built for (d > 64, more than 2 hidden layers) and the precisions chosen
     for fp32-grade arithmetic throughout ("tf32x3", "fp32") take the same pass through torch autograd (large library
     GEMMs) - stated, not hidden.

With method 'kl' / 'kl_ito' (kl_objective, ClippedCtrl) the SDE follows the non-detached control and the gradient runs
through the trajectory: step 3 takes the cotangents d loss / d g_k that the reverse-time adjoint kernel lrds_adjoint
computes from the stored trajectory (csrc/lrds_adjoint.cuh); everything else is shared with the LV objective.

Nothing here runs on the CPU or imports the oracle.
"""
from __future__ import annotations

import ctypes as C

import torch
import torch.nn.functional as F

from . import _native as N
from . import pack


def time_embed_rows(m, t: torch.Tensor) -> torch.Tensor:
    """Differentiable TimeEmbed.forward for a 1-D tensor of times (sde_sampler/models/mlp.py:85-96)."""
    arg = m.timestep_coeff * t.reshape(-1, 1) + m.timestep_phase
    e = torch.cat([torch.sin(arg), torch.cos(arg)], dim=1)
    for layer in m.hidden_layer:
        e = F.gelu(layer(e))
    return m.out_layer(e)


def _clip(v, bound):
    return v if bound is None else v.clip(-bound, bound)


def control_rows(info: pack.CtrlInfo, taus: torch.Tensor, xs: torch.Tensor, score: torch.Tensor | None,
                 coef: torch.Tensor | None = None) -> torch.Tensor:
    """g(t_s, x_sb) for times taus [S] and states xs [S, B, d], differentiable in the parameters of the control:
    FourierMLP.forward (models/mlp.py:135-143) under ClippedCtrl / ScoreCtrl / CancelDriftCtrl / LerpCtrl.forward
    (models/reparam.py:33-43, 112-117, 131-147, 189-199).  ``score`` = the (for LerpCtrl: interpolated) target score at
    xs, a constant because the states carry no gradient; ``coef`` [S, 16] = the time-only table columns of the two DIS
    models (pack.dis_ctrl_rows)."""
    base = info.base
    emb = base.input_embed(xs) + time_embed_rows(base.timestep_embed, taus)[:, None, :]
    for layer in base.hidden_layer:
        emb = layer(F.gelu(emb))
    g = _clip(base.out_layer(F.gelu(emb)), info.clip_model)
    if info.kind == N.CTRL_CLIPPED:
        return g
    sc = info.scale_score * _clip(score, info.clip_score)
    if info.score_model is not None:
        sc = sc * _clip(time_embed_rows(info.score_model, taus), info.clip_model)[:, None, :]
    if info.kind == N.CTRL_CANCEL_DRIFT:  # ctrl + drift / diff + 0.5 diff score
        return g + coef[:, N.STEP_CX, None, None] * xs + coef[:, N.STEP_GSCALE, None, None] * sc
    if info.kind == N.CTRL_LERP:          # ctrl + diff score
        return g + coef[:, N.STEP_GSCALE, None, None] * sc
    return g + sc


def mlp_grad_applicable(base) -> bool:
    """The weight-gradient kernel (lrds_mlp_grad) is built for the FourierMLP shapes d <= 64, at most 2 hidden layers."""
    return hasattr(base, "lrds_mlp") and N.lib().lrds_mlp_grad_floats(base.dim, len(base.hidden_layer)) > 0


def pow2_scale(bound: float, target: float = 4.0) -> float:
    """Power of two s with bound * s in (target / 2, target] (1 for a zero / non-finite bound)."""
    import math
    if not (bound > 0.0) or math.isinf(bound):
        return 1.0
    return 2.0 ** math.floor(math.log2(target / bound))


def mlp_grad(base, bias1: torch.Tensor, xs: torch.Tensor, cot: torch.Tensor, clip, step_w=None, row_w=None,
             cot_bound=None):
    """Gradient of  sum_{s,b} <cot_sb * step_w_s * row_w_b, clip(FourierMLP(t_s, x_sb))>  in the backbone's parameters,
    by the hand-written kernel: returns ({parameter: gradient} for input_embed.weight, hidden_layer.*, out_layer.*,
    dbias1 [S, 64]) where dbias1 is the cotangent of ``bias1`` = input_embed.bias + TimeEmbed(t_s) (the caller carries it
    through TimeEmbed with autograd: S rows).  ``cot_bound`` >= max |cot * step_w * row_w| sets the fp16 operand scale: a
    float, or a 0-dim DEVICE tensor (the scale is then formed on the device: no host synchronisation)."""
    dev = xs.device
    S, B, d = xs.shape
    nh = len(base.hidden_layer)
    mlp, keep = base.lrds_mlp(dev, N.PRECISION_F16X3)
    xs, cot = xs.contiguous(), cot.contiguous()
    bias1 = bias1.detach().to(dev, torch.float32).contiguous()
    if cot_bound is None:
        cot_bound = cot.abs().max()
        if step_w is not None:
            cot_bound = cot_bound * step_w.abs().max().to(dev)
        if row_w is not None:
            cot_bound = cot_bound * row_w.abs().max()
    scale, scale_dev = 1.0, None
    if torch.is_tensor(cot_bound):  # 2^floor(log2(4 / bound)) on the device; 1 for a zero / non-finite bound
        bnd = cot_bound.detach().to(dev, torch.float32).reshape(())
        scale_dev = torch.exp2(torch.floor(torch.log2(4.0 / bnd)))
        scale_dev = torch.where(torch.isfinite(scale_dev) & (scale_dev > 0), scale_dev, torch.ones_like(scale_dev)).reshape(1)
    else:
        scale = pow2_scale(float(cot_bound))
    L = N.lib()
    flat = torch.empty(int(L.lrds_mlp_grad_floats(d, nh)), device=dev, dtype=torch.float32)
    dbias1 = torch.empty(S, N.CHANNELS, device=dev, dtype=torch.float32)
    scratch = torch.empty(int(L.lrds_mlp_grad_scratch_floats(d, nh, S, B)), device=dev, dtype=torch.float32)
    sw = None if step_w is None else step_w.detach().to(dev, torch.float32).contiguous()
    rw = None if row_w is None else row_w.detach().to(dev, torch.float32).reshape(-1).contiguous()
    with torch.cuda.device(dev):
        N.check(L.lrds_mlp_grad(C.byref(mlp), N.ptr(bias1), N.ptr(xs), N.ptr(cot), N.ptr(sw), N.ptr(rw),
                                float(clip) if clip is not None else 0.0, scale, N.ptr(scale_dev), S, B, N.ptr(flat),
                                N.ptr(dbias1), N.ptr(scratch), N.stream_ptr(dev)))
    Cc, dp = N.CHANNELS, mlp.d_pad
    w_in_t, w_hid_t, b_hid, w_out_t, b_out = flat.split([d * Cc, nh * Cc * Cc, nh * Cc, Cc * dp, dp])
    grads = {base.input_embed.weight: w_in_t.view(d, Cc).t(),
             base.out_layer.weight: w_out_t.view(Cc, dp)[:, :d].t(), base.out_layer.bias: b_out[:d]}
    for i, layer in enumerate(base.hidden_layer):
        grads[layer.weight] = w_hid_t.view(nh, Cc, Cc)[i].t()
        grads[layer.bias] = b_hid.view(nh, Cc)[i]
    return grads, dbias1


def score_cot_sums(distr, xs: torch.Tensor, cot: torch.Tensor, clip, step_w=None, row_w=None) -> torch.Tensor:
    """M[s, j] = sum_b step_w[s] row_w[b] cot[s, b, j] clip(distr.score(xs[s, b]))[j]  by one fused launch
    (lrds_score_cot_sums): the scores are evaluated and reduced in the kernel instead of being written out."""
    dev = xs.device
    S, B, d = xs.shape
    block, _keep = distr.lrds_distr(dev)
    L = N.lib()
    n = int(L.lrds_score_cot_scratch_floats(C.byref(block), d, S, B))
    if n < 0:
        N.check(n)
    out = torch.empty(S, d, device=dev, dtype=torch.float32)
    scratch = torch.empty(n, device=dev, dtype=torch.float32)
    sw = None if step_w is None else step_w.detach().to(dev, torch.float32).contiguous()
    rw = None if row_w is None else row_w.detach().to(dev, torch.float32).reshape(-1).contiguous()
    with torch.cuda.device(dev):
        N.check(L.lrds_score_cot_sums(C.byref(block), d, N.ptr(xs.contiguous()), N.ptr(cot.contiguous()), N.ptr(sw), N.ptr(rw),
                                      float(clip) if clip is not None else 0.0, S, B, N.ptr(out), N.ptr(scratch),
                                      N.stream_ptr(dev)))
    return out


def control_param_grads(info: pack.CtrlInfo, params, taus, xs, cot, step_w, row_w, coef, score_of, max_rows: int,
                        cot_max: float | None = None):
    """Gradients (a list aligned with ``params``) of  sum_{s,b} <cot_sb step_w_s row_w_b, control_rows(...)_sb>  with the
    backbone's part taken by the weight-gradient kernel (mlp_grad) over all S x B states at once.  What is left for
    autograd is S rows wide: TimeEmbed + input bias under the kernel's cotangent dbias1, and the time-only factor
    clip(TimeEmbed_score(t)) of ScoreCtrl / CancelDriftCtrl / LerpCtrl (models/reparam.py:112-117, 131-147, 189-199)
    under  M[s] = sum_b cot_sb (x) scale_score clip(score(x_sb))  (``score_of(k0, k1)`` -> the constant scores)."""
    base = info.base
    S, B, d = xs.shape
    by_param = {}
    with torch.enable_grad():
        bias1 = time_embed_rows(base.timestep_embed, taus) + base.input_embed.bias
    bound = cot.abs().max() if cot_max is None else torch.full((), float(cot_max), device=xs.device)  # device scalars:
    if step_w is not None:                                                                            # no host round trip
        bound = bound * step_w.abs().max()
    if row_w is not None:
        bound = bound * row_w.abs().max()
    kernel_grads, dbias1 = mlp_grad(base, bias1, xs, cot, info.clip_model, step_w, row_w, cot_bound=bound)
    by_param.update(kernel_grads)
    tp = [p for p in [*base.timestep_embed.parameters(), base.input_embed.bias] if p.requires_grad]
    if tp:
        for p, g in zip(tp, torch.autograd.grad(bias1, tp, grad_outputs=dbias1, allow_unused=True)):
            by_param[p] = g
    sp = [] if info.kind == N.CTRL_CLIPPED or info.score_model is None else \
        [p for p in info.score_model.parameters() if p.requires_grad]
    if sp:
        if info.kind != N.CTRL_LERP and hasattr(info.target, "lrds_distr"):  # scores evaluated and reduced in one kernel
            M = info.scale_score * score_cot_sums(info.target, xs, cot, info.clip_score, step_w, row_w)
            if info.kind == N.CTRL_CANCEL_DRIFT:
                M = M * coef[:S, N.STEP_GSCALE, None]
        else:  # LerpCtrl clips the INTERPOLATED score (models/reparam.py:170-183): two distributions, elementwise here
            M = xs.new_empty(S, d)
            rows = max(1, max_rows // B)
            with torch.no_grad():
                for k0 in range(0, S, rows):
                    k1 = min(S, k0 + rows)
                    sc = info.scale_score * _clip(score_of(k0, k1), info.clip_score)
                    if info.kind in (N.CTRL_CANCEL_DRIFT, N.CTRL_LERP):
                        sc = sc * coef[k0:k1, N.STEP_GSCALE, None, None]
                    c = cot[k0:k1]
                    if step_w is not None:
                        c = c * step_w[k0:k1, None, None]
                    if row_w is not None:
                        c = c * row_w.reshape(1, B, 1)
                    M[k0:k1] = (c * sc).sum(1)
        with torch.enable_grad():
            gam = _clip(time_embed_rows(info.score_model, taus), info.clip_model)
            for p, g in zip(sp, torch.autograd.grad((gam * M).sum(), sp, allow_unused=True)):
                by_param[p] = g
    return [by_param.get(p) for p in params]


class _InjectGrads(torch.autograd.Function):
    """loss value whose backward hands the precomputed parameter gradients to autograd."""

    @staticmethod
    def forward(ctx, value, grads, *params):
        ctx.grads = grads
        return value.clone()

    @staticmethod
    def backward(ctx, grad_out):
        return (None, None, *[None if g is None else grad_out * g for g in ctx.grads])


def normals(seed: int, particle_offset: int, K: int, B: int, d: int, device) -> torch.Tensor:
    """The increments z [K, B, d] the production-mode rollout would draw in-kernel (lrds_normals, stream 0)."""
    z = torch.empty(K, B, d, device=device, dtype=torch.float32)
    with torch.cuda.device(device):
        N.check(N.lib().lrds_normals(C.c_uint64(seed & (2 ** 64 - 1)), C.c_uint64(particle_offset), 0, K, B, d, N.ptr(z),
                                     N.stream_ptr(device)))
    return z


def lv_weights(rnd: torch.Tensor, mask: torch.Tensor, group=None):
    """(loss, d loss / d rnd) of loss = Var(rnd[mask]) (unbiased) over the GLOBAL batch when the particles are sharded
    over the ranks of ``group``: three fp64 sums (sum, count, sum of squares) travel through ONE all_reduce - the
    training-side counterpart of the estimator exchange (DESIGN.md section 6).  Runs on whatever device ``rnd`` lives on
    (NCCL on the GPUs, gloo in the CPU tests)."""
    import torch.distributed as dist
    r = rnd.detach().double()
    m = mask.to(r.dtype)
    stats = torch.stack([(r * m).sum(), m.sum(), (r * r * m).sum()])
    if group is not None and dist.is_available() and dist.is_initialized():
        dist.all_reduce(stats, op=dist.ReduceOp.SUM, group=group)
    s, n, s2 = stats
    mean = s / n
    var = (s2 - n * mean * mean) / (n - 1.0)
    w = 2.0 * (r - mean) / (n - 1.0) * m
    return var.to(rnd.dtype), w.to(rnd.dtype)


def _loss_weights(loss_obj, rnd: torch.Tensor, x_T: torch.Tensor):
    """(loss, d loss / d rnd_b, metrics) of the reference's loss formula (compute_loss) on the B log-weights."""
    rnd_leaf = rnd.detach().clone().requires_grad_(True)
    with torch.enable_grad():
        value, metrics = loss_obj.compute_loss(rnd_leaf, samples=x_T)
        (w,) = torch.autograd.grad(value, rnd_leaf)  # zero for filtered particles
    return value, w, metrics


def _param_grads(loss_obj, plan: pack.Plan, info: pack.CtrlInfo, xs: torch.Tensor, cot: torch.Tensor, weights,
                 max_rows: int, cot_max: float | None = None):
    """Gradients (aligned with the control's trainable parameters) of  sum_{k,b} <c_kb, g(t_k, x_kb)>  over the K stored
    states xs [K, B, d], with c = cot, or (step_w_k row_w_b) cot for ``weights`` = (step_w [K], row_w [B]): the
    weight-gradient kernel (lrds_mlp_grad) where it is built, else autograd over ``control_rows`` in slices of
    ``max_rows`` rows.  ``cot_max`` >= max |cot| when known (saves a reduction)."""
    dev = xs.device
    K, B, d = xs.shape
    params = [p for p in loss_obj.generative_ctrl.parameters() if p.requires_grad]
    grads: list = [None] * len(params)
    taus = pack.on_device(plan, "taus", dev)
    step_w, row_w = weights if weights is not None else (None, None)

    def dis_rows():  # time-only table columns of the DIS drift models (they do not depend on the parameters)
        c = torch.zeros(K, N.STEP_BIAS1)
        pack.dis_ctrl_rows(info, plan.taus, c)
        return c
    coef = pack.on_device(plan, "coef", dev, dis_rows)
    step_rows = max(1, max_rows // B)

    def score_of(k0, k1):  # the constant score factor of the control at the stored states of steps k0 .. k1 - 1
        flat = xs[k0:k1].reshape(-1, d)
        score = info.target.score(flat).reshape(k1 - k0, B, d)
        if info.kind == N.CTRL_LERP:  # clipped_interpolated_score, models/reparam.py:170-183
            score = torch.lerp(info.prior.score(flat).reshape(k1 - k0, B, d), score, coef[k0:k1, N.STEP_LERP, None, None])
        return score

    use_kernel = mlp_grad_applicable(info.base) and plan.spec.precision == N.PRECISION_F16X3
    if use_kernel:  # the backbone's gradient by lrds_mlp_grad: one launch over all K x B stored states
        grads = control_param_grads(info, params, taus[:K], xs, cot, step_w, None if row_w is None else row_w.reshape(-1),
                                    coef, score_of, max_rows, cot_max=cot_max)
    for k0 in range(0, K if not use_kernel else 0, step_rows):
        k1 = min(K, k0 + step_rows)
        xs_c = xs[k0:k1]
        score = None
        if info.kind != N.CTRL_CLIPPED:
            score = info.target.score(xs_c.reshape(-1, d)).reshape(k1 - k0, B, d)
            if info.kind == N.CTRL_LERP:  # clipped_interpolated_score, models/reparam.py:170-183
                prior = info.prior.score(xs_c.reshape(-1, d)).reshape(k1 - k0, B, d)
                score = torch.lerp(prior, score, coef[k0:k1, N.STEP_LERP, None, None])
        c = cot[k0:k1] if weights is None else (step_w[k0:k1, None, None] * row_w.reshape(1, B, 1)) * cot[k0:k1]
        with torch.enable_grad():
            surrogate = (c * control_rows(info, taus[k0:k1], xs_c, score, coef[k0:k1])).sum()
        _accumulate(grads, params, surrogate)
    return params, grads


def lv_objective(loss_obj, plan: pack.Plan, info: pack.CtrlInfo, x: torch.Tensor, seed: int, noise=None,
                 particle_offset: int = 0, max_rows: int = 1 << 20, group=None):
    """(loss, metrics) like ``BaseOCLoss.__call__``: ``loss`` is a scalar whose ``backward()`` leaves the LV gradient in
    the ``.grad`` of the control's parameters.  With ``group`` (a torch.distributed group; method 'lv') the batch is the
    union of the ranks' shards (``particle_offset`` = this rank's first global particle index): the variance and its
    weights are global (lv_weights) and the parameter gradients are summed over the ranks, so every rank returns the
    loss and gradient of the whole batch."""
    dev = x.device
    B, d = x.shape
    K = plan.noise_steps
    # without recorded increments the rollout draws its own (in-kernel Philox, no read of a [K, B, d] array); lrds_normals
    # reproduces exactly those for the cotangents below
    z = normals(seed, particle_offset, K, B, d, dev) if noise is None else noise.detach().to(dev, torch.float32).contiguous()
    with torch.no_grad():
        x_T, rnd, xs = pack.run_rollout(plan, x, None if noise is None else z, seed, particle_offset, True)
    if group is not None:
        if loss_obj.method != "lv":
            raise NotImplementedError("sharded training is built for method 'lv'")
        mask = loss_obj.filter(rnd, samples=x_T)
        loss_obj.n_filtered += (mask.numel() - mask.sum()).item()
        value, w = lv_weights(rnd, mask, group)
        metrics = {"train/n_filtered_cumulative": loss_obj.n_filtered}
    else:
        value, w, metrics = _loss_weights(loss_obj, rnd, x_T)
    ito_w = pack.on_device(plan, "ito_w", dev)
    # the generator's normals are bounded: Box-Muller on at most 32-bit uniforms, |z| <= sqrt(2 * 32 * ln 2) < 6.7
    params, grads = _param_grads(loss_obj, plan, info, xs[:K], z, (ito_w[:K], w), max_rows,
                                 cot_max=7.0 if noise is None else None)
    if group is not None:  # one all_reduce over the flattened gradients
        import torch.distributed as dist
        flat = torch.cat([(g if g is not None else torch.zeros_like(p)).reshape(-1) for g, p in zip(grads, params)])
        dist.all_reduce(flat, op=dist.ReduceOp.SUM, group=group)
        grads = [c.reshape(p.shape) for c, p in zip(flat.split([p.numel() for p in params]), params)]
    return _InjectGrads.apply(value.detach(), grads, *params), metrics


def adjoint(plan: pack.Plan, xs: torch.Tensor, w: torch.Tensor, seed: int, noise=None, particle_offset: int = 0):
    """gbar [K, B, d] = d loss / d g_k of the pathwise ('kl' / 'kl_ito') gradient by the reverse-time kernel lrds_adjoint:
    ``xs`` [K + 1, B, d] = the trajectory the rollout of ``plan`` wrote, ``w`` [B] = d loss / d rnd_b, ``noise`` = the
    increments that rollout consumed (None: the kernel regenerates the in-kernel Philox draws of ``seed``)."""
    dev = xs.device
    K1, B, d = xs.shape
    spec = N.Spec.from_buffer_copy(plan.spec)  # the cached plan is shared: never mutated here
    spec.B = B
    spec.status = pack.status_counters(dev).data_ptr()
    cot = torch.empty(K1 - 1, B, d, device=dev, dtype=torch.float32)
    rw = w.detach().to(dev, torch.float32).reshape(-1).contiguous()
    z = None if noise is None else noise.detach().to(dev, torch.float32).contiguous()
    with torch.cuda.device(dev):
        N.check(N.lib().lrds_adjoint(C.byref(spec), N.ptr(xs.contiguous()), N.ptr(z), C.c_uint64(seed & (2 ** 64 - 1)),
                                     C.c_uint64(particle_offset), N.ptr(rw), N.ptr(cot), N.stream_ptr(dev)))
    return cot


def kl_objective(loss_obj, plan: pack.Plan, info: pack.CtrlInfo, x: torch.Tensor, seed: int, noise=None,
                 particle_offset: int = 0, max_rows: int = 1 << 20, rnd_start=None):
    """(loss, metrics) of method 'kl' / 'kl_ito' (the SDE follows the non-detached control, oc.py:83-103; loss =
    mean(rnd[mask])): the fused rollout with its trajectory, d loss / d rnd from compute_loss, the reverse-time adjoint
    (lrds_adjoint) for the cotangents gbar_k = d loss / d g_k, and the same parameter pass as lv_objective with
    cot = gbar.  ``rnd_start`` [B]: subtracted from the rollout's log-weights (the DIS training form starts at 0, the
    rollout at the prior log-density)."""
    if rnd_start is not None and plan.spec.rnd_offset != 0.0:  # the training plans start at log p_prior(x_0) exactly
        raise ValueError("rnd_start assumes a rollout whose initial cost has no state-independent offset (train=True)")
    noise = None if noise is None else noise.detach().to(x.device, torch.float32).contiguous()
    with torch.no_grad():
        x_T, rnd, xs = pack.run_rollout(plan, x, noise, seed, particle_offset, True)
        if rnd_start is not None:
            rnd = rnd - rnd_start.reshape(rnd.shape)
    value, w, metrics = _loss_weights(loss_obj, rnd, x_T)
    cot = adjoint(plan, xs, w, seed, noise, particle_offset)
    params, grads = _param_grads(loss_obj, plan, info, xs[:-1], cot, None, max_rows)
    return _InjectGrads.apply(value.detach(), grads, *params), metrics


def _accumulate(grads, params, surrogate):
    for i, g in enumerate(torch.autograd.grad(surrogate, params, allow_unused=True)):
        if g is not None:
            grads[i] = g if grads[i] is None else grads[i] + g


def cmcd_lv_objective(loss_obj, plan: pack.Plan, info: pack.CtrlInfo, x: torch.Tensor, seed: int, noise=None,
                      particle_offset: int = 0, max_rows: int = 1 << 20):
    """The same for ControlledLangevinSDELoss (oc.py:666-755, 830-860) with method 'lv'.  Every trajectory point
    (ts[j], xs[j]) enters the log-weight twice - as the start of step j (control u_s) and as the end of step j - 1
    (control u_t) - through cost_k = (drift_s + drift_t) / sigma + u_s - u_t:

        d rnd_b / d theta = sum_j < [j < K] db_j  -  [j >= 1] (cost_{j-1} dt_{j-1} + db_{j-1}),  d g(ts[j], xs[j]) / d theta >

    (the term cost (sde_ctrl - u_s) dt of oc.py:739 removes the cost dt contribution of the start point).  One batched
    pass over the K + 1 stored states evaluates the controls and the tempered drifts for the costs, a second one carries
    the cotangents back."""
    dev = x.device
    B, d = x.shape
    K = plan.noise_steps
    z = normals(seed, particle_offset, K, B, d, dev) if noise is None else noise.detach().to(dev, torch.float32).contiguous()
    with torch.no_grad():
        x_T, rnd, xs = pack.run_rollout(plan, x, z, seed, particle_offset, True)
    rnd_leaf = rnd.detach().clone().requires_grad_(True)
    with torch.enable_grad():
        value, metrics = loss_obj.compute_loss(rnd_leaf, samples=x_T)
        (w,) = torch.autograd.grad(value, rnd_leaf)
    params = [p for p in loss_obj.generative_ctrl.parameters() if p.requires_grad]
    grads: list = [None] * len(params)
    sde = loss_obj.sde
    ts = pack.on_device(plan, "taus", dev)      # [K + 1]
    dt = pack.on_device(plan, "dt", dev, lambda: plan.taus[1:] - plan.taus[:-1])
    sig = sde.diff_coeff.to(dev)
    frac = pack.on_device(plan, "frac", dev, lambda: plan.taus / sde.terminal_t.detach().cpu())
    target, prior = sde.target_score.__self__, sde.prior_score.__self__
    rows = max(1, max_rows // B)
    gd, drift, tscore = [], [], []
    with torch.no_grad():  # pass 1: controls and tempered drifts (eq/sdes.py:101-110) at every stored state
        for j0 in range(0, K + 1, rows):
            j1 = min(K + 1, j0 + rows)
            flat = xs[j0:j1].reshape(-1, d)
            tsc = target.score(flat).reshape(j1 - j0, B, d)
            dr = tsc * frac[j0:j1, None, None] + prior.score(flat).reshape(j1 - j0, B, d) * (1.0 - frac[j0:j1, None, None])
            dr = _clip(dr * (0.5 * sig ** 2), sde.clip_score)
            gd.append(control_rows(info, ts[j0:j1], xs[j0:j1], tsc if info.kind != N.CTRL_CLIPPED else None))
            drift.append(dr)
            tscore.append(tsc)
        gd, drift, tscore = torch.cat(gd), torch.cat(drift), torch.cat(tscore)
        db = dt.sqrt()[:, None, None] * z                                   # [K, B, d]
        cost = (drift[:-1] + drift[1:]) / sig + gd[:-1] - gd[1:]             # [K, B, d]
        cot = torch.zeros_like(xs)
        cot[:-1] += db
        cot[1:] -= cost * dt[:, None, None] + db
        cot *= w[None, :, :]
    use_kernel = mlp_grad_applicable(info.base) and plan.spec.precision == N.PRECISION_F16X3
    if use_kernel:  # pass 2 by lrds_mlp_grad: one launch over the (K + 1) x B stored states
        grads = control_param_grads(info, params, ts, xs, cot, None, None, None, lambda j0, j1: tscore[j0:j1], max_rows)
    for j0 in range(0, K + 1 if not use_kernel else 0, rows):  # pass 2 (shapes the kernel is not built for): autograd
        j1 = min(K + 1, j0 + rows)
        with torch.enable_grad():
            g = control_rows(info, ts[j0:j1], xs[j0:j1], tscore[j0:j1] if info.kind != N.CTRL_CLIPPED else None)
            _accumulate(grads, params, (cot[j0:j1] * g).sum())
    return _InjectGrads.apply(value.detach(), grads, *params), metrics
