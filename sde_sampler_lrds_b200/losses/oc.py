"""The integrate-and-weight loop behind RDS / PIS / DDS / CMCD with the reference's loss classes and method
signatures (sde_sampler/losses/oc.py): ``simulate`` / ``eval`` / ``compute_eubo`` pack the rollout into an
``lrds_spec`` and run ONE fused CUDA kernel for all K steps (csrc/), instead of ~40-150 eager ops per step.

    EMReferenceSDELoss            oc.py:203-428   (RDS-EM; PIS with reference_ctrl=None)
    EIReferenceSDELoss            oc.py:431-568
    DDPMLikeReferenceSDELoss      oc.py:571-651
    ControlledLangevinSDELoss     oc.py:654-894   (CMCD)
    ExponentialIntegratorSDELoss  oc.py:1310-1467 (DDS)
    TimeReversalLoss              oc.py:1105-1307 (DIS: inference_ctrl=None)
    DiscreteTimeReversalLossEI    oc.py:897-1103  (discrete-time DIS with the exponential integrator)

Extra keyword arguments (not in the reference, all optional): ``noise`` = recorded standard normals [K, B, d]
to consume instead of in-kernel Philox draws (validation mode), ``seed`` / ``particle_offset`` for the
counter-based generator (global particle index => results independent of the GPU count).
Training: ``loss(ts, x, ...)`` with method 'lv' / 'lv_traj' returns a scalar whose ``backward()`` fills the control's
parameter gradients (train.py: fused rollout + one batched gradient pass), for every loss class below; 'kl' / 'kl_ito'
(pathwise gradient through the trajectory: fused rollout + the reverse-time adjoint kernel + the same parameter pass) for
the linear losses and CMCD with a ClippedCtrl drift.
"""
from __future__ import annotations

import itertools
from typing import Callable

import torch

from .. import _native as N
from .. import pack
from ..distr.base import Distribution, fill_gmm
from ..eq.sdes import OU, ControlledLangevinSDE, MarginalReference
from ..estimators import estimator_partials, metrics_from_partials
from ..utils.common import Results


def _fid(fn):
    """Stable identity of a callable for the plan cache: a bound method is a fresh object at every attribute access
    (``solver.clipped_target_unnorm_log_prob``), so it is keyed by its owner and name."""
    owner = getattr(fn, "__self__", None)
    return (id(owner), getattr(fn, "__name__", "")) if owner is not None else id(fn)


def _terminal_target(fn):
    """The Distribution behind a terminal log-density callable (the object a plan is packed from; NOT the solver that
    owns ``clipped_target_unnorm_log_prob``, whose parameters change with every training step)."""
    try:
        return pack.resolve_log_prob(fn)[0]
    except NotImplementedError:
        return None


def _fid_clip(fn):
    owner = getattr(fn, "__self__", None)
    return getattr(owner, "clip_target", None) if owner is not None and not isinstance(owner, Distribution) else None


def _state(obj):
    """(identity, tensor versions) of an object a plan was packed from.  The identity is an ``id``: the cache entry keeps
    a strong reference to the object (``_cached``), so the address cannot be recycled while the entry lives; in-place
    edits of its parameters / buffers show up in the version counters."""
    if obj is None:
        return None
    if isinstance(obj, torch.nn.Module):
        return (id(obj),) + tuple((t.data_ptr(), t._version) for t in list(obj.parameters()) + list(obj.buffers()))
    tensors = tuple(v for v in vars(obj).values() if isinstance(v, torch.Tensor)) if hasattr(obj, "__dict__") else ()
    return (id(obj),) + tuple((t.data_ptr(), t._version) for t in tensors)


def _resolve_reference(ref_ctrl):
    if ref_ctrl is None:
        return None
    if isinstance(ref_ctrl, MarginalReference):
        return ref_ctrl
    owner = getattr(ref_ctrl, "__self__", None)
    cand = getattr(owner, "reference_score_t", None)
    if isinstance(cand, MarginalReference):
        return cand
    raise NotImplementedError("reference_ctrl must be a MarginalReference (gaussian / gmm reference); "
                              "neural references are a later row (SURVEY.md 8f item 3)")


class BaseOCLoss:
    """Base class: estimators and bookkeeping shared by every rollout loss."""

    def __init__(self, generative_ctrl: Callable, generative_ctrl_ema: Callable, sde: OU | None = None,
                 method: str = "kl", traj_per_sample: int = 1, filter_samples: Callable | None = None,
                 max_rnd: float | None = None, sde_ctrl_dropout: float | None = None,
                 sde_ctrl_noise: float | None = None, precision: str | None = None, **kwargs):
        self.generative_ctrl = generative_ctrl
        self.generative_ctrl_ema = generative_ctrl_ema
        self.sde = sde
        if method not in ["kl", "kl_ito", "lv", "lv_traj"]:
            raise ValueError("Unknown loss method.")
        self.method = method
        if traj_per_sample == 1 and self.method == "lv_traj":
            raise ValueError("Cannot compute variance over a single trajectory.")
        self.traj_per_sample = traj_per_sample
        self.filter_samples = filter_samples
        self.max_rnd = max_rnd
        self.sde_ctrl_noise = sde_ctrl_noise
        self.sde_ctrl_dropout = sde_ctrl_dropout
        self.n_filtered = 0
        self.precision = precision
        self._plans: dict = {}
        self._grids: dict = {}
        self._calls = itertools.count()

    # ---- estimators (oc.py:134-173) ---------------------------------------------------------------------------
    @staticmethod
    def compute_results(rnd: torch.Tensor, compute_weights: bool = False, ts=None, samples=None, xs=None,
                        group=None) -> Results:
        """ELBO, importance weights, log Z and LV from the log-weights; the reductions run in the estimator
        kernel (fp64 partials), merged across ranks when ``group`` is a torch.distributed group."""
        part = estimator_partials(rnd, group=group)
        m = metrics_from_partials(part)
        metrics = {"eval/elbo": m["elbo"]}
        if compute_weights:
            weights = torch.exp(-rnd.double() - part[0]).div(part[1]).to(rnd.dtype)  # softmax(-rnd, dim=0)
            log_norm_const_preds = {"log_norm_const_is": m["log_norm_const_is"]}
            metrics["eval/lv_loss"] = m["lv_loss"]
            # ESS of the importance weights, (sum w)^2 / sum w^2 (get_metrics, eval/metrics.py:134-140), from the same partials
            metrics["eval/effective_sample_size"] = m["effective_sample_size"]
            metrics["eval/norm_effective_sample_size"] = m["norm_effective_sample_size"]
        else:
            weights, log_norm_const_preds = None, {}
        return Results(samples=samples, weights=weights, log_norm_const_preds=log_norm_const_preds, ts=ts, xs=xs,
                       metrics=metrics)

    def filter(self, rnd, samples=None):
        mask = True
        if samples is not None and self.filter_samples is not None:
            mask = self.filter_samples(samples)
        if self.max_rnd is None:
            return mask & rnd.isfinite()
        return mask & (rnd < self.max_rnd)

    def compute_loss(self, rnd: torch.Tensor, samples: torch.Tensor | None = None):
        """The variational loss from the log-weights (oc.py:105-131): variance ('lv'), per-sample variance over the
        repeated trajectories ('lv_traj') or mean ('kl') of the particles that pass ``filter``."""
        mask = self.filter(rnd, samples=samples)
        assert mask.shape == rnd.shape
        if self.method == "lv_traj":
            rnd = rnd.reshape(self.traj_per_sample, -1, 1)
            mask = mask.reshape(self.traj_per_sample, -1, 1).all(dim=0)
            n_bad = (mask.numel() - mask.sum()).item()  # the one host round trip of the loss formula
            self.n_filtered += self.traj_per_sample * n_bad
            loss = (rnd if n_bad == 0 else rnd[:, mask]).var(dim=0).mean()
        else:
            n_bad = (mask.numel() - mask.sum()).item()
            self.n_filtered += n_bad
            kept = rnd if n_bad == 0 else rnd[mask]  # nothing filtered (the usual case): no boolean gather
            loss = kept.var() if self.method == "lv" else kept.mean()
        return loss, {"train/n_filtered_cumulative": self.n_filtered}

    def _train(self, make_plan, x, noise=None, seed=None, particle_offset: int = 0, group=None, initial_log_prob=None):
        """[TRAINING] shared by the ``__call__`` of the linear losses: repeat the initial values, run the fused rollout
        and return (loss, metrics) with the gradient attached (train.py): for 'lv' / 'lv_traj' the SDE follows the
        detached control (lv_objective), for 'kl' / 'kl_ito' the pathwise gradient through the trajectory
        (kl_objective, ClippedCtrl).  ``initial_log_prob`` (DIS): the prior log-density the rollout starts the log-weight
        at, which the 'kl' training form leaves out."""
        from .. import train
        x = self._train_batch(x)
        info = self._ctrl(False)
        if self.method in ("lv", "lv_traj"):
            return train.lv_objective(self, make_plan(x.device), info, x, self._seed(seed), noise=noise,
                                      particle_offset=particle_offset, group=group)
        if group is not None:
            raise NotImplementedError("sharded training is built for method 'lv'")
        _kl_ctrl_check(info)
        if getattr(self, "_init_cost", False):
            raise NotImplementedError("the discrete-time DIS loss has no 'kl' training rollout here (no shipped config uses it)")
        rnd_start = None if initial_log_prob is None else _kl_start(initial_log_prob, x)
        return train.kl_objective(self, make_plan(x.device), info, x, self._seed(seed), noise=noise,
                                  particle_offset=particle_offset, rnd_start=rnd_start)

    def _train_batch(self, x):
        """The training batch: ``x`` repeated ``traj_per_sample`` times; control noise / dropout are refused."""
        if self.sde_ctrl_noise is not None or self.sde_ctrl_dropout is not None:
            raise NotImplementedError("sde_ctrl_noise / sde_ctrl_dropout are not set by any shipped config")
        if self.traj_per_sample != 1:
            x = x.repeat(self.traj_per_sample, 1, 1).reshape(-1, x.shape[-1])
        return x

    def __call__(self, ts, x, *args, **kwargs):
        raise NotImplementedError("training through this loss is not built (SURVEY.md 8f item 1): the linear losses "
                                  "(EM / EI / DDPM-like reference losses, DDS, DIS) train with method 'lv' or 'kl'")

    def load_state_dict(self, state_dict: dict):
        self.n_filtered = state_dict["n_filtered"]

    def state_dict(self) -> dict:
        return {"n_filtered": self.n_filtered}

    # ---- shared plumbing ------------------------------------------------------------------------------------------
    def _ctrl(self, use_ema):
        return pack.resolve_ctrl(self.generative_ctrl_ema if use_ema else self.generative_ctrl)

    def _check_plain(self, change_sde_ctrl):
        if change_sde_ctrl and (self.sde_ctrl_noise is not None or self.sde_ctrl_dropout is not None
                                or torch.is_grad_enabled()):
            raise NotImplementedError("change_sde_ctrl with autograd / control noise is training-only (SURVEY.md 8f item 1)")

    def _seed(self, seed):
        if seed is not None:
            return int(seed)
        return (int(torch.initial_seed()) * 0x9E3779B97F4A7C15 + next(self._calls) * 0xD1B54A32D192ED03) & (2 ** 64 - 1)

    def _cached(self, key, build, info, device):
        """Plans are cached by everything that does not depend on the control's parameters (grid, schedule, reference and
        target blocks: O(K) host work, ~45 ms at K = 200); a parameter update (training step, EMA
        swap) only refreshes the weight images and the TimeEmbed rows of the cached plan (pack.refresh_ctrl)."""
        skey, vers, refs = key
        hit = self._plans.get(skey)
        if hit is None:
            if len(self._plans) >= 16:
                self._plans.pop(next(iter(self._plans)))
            hit = self._plans[skey] = [build(), vers, refs]  # refs: the keyed objects stay alive with the entry
        elif hit[1] != vers:
            pack.refresh_ctrl(hit[0], info, device)
            hit[1] = vers
        return hit[0]

    def clear_plans(self):
        """Drops every cached rollout plan (the solvers call this when they swap the reference or the prior)."""
        self._plans.clear()
        self._grids.clear()

    def _grid_bytes(self, ts):
        """The time grid as bytes for the plan key.  A device-resident grid is read back ONCE per (storage, version):
        ``ts.to('cpu')`` is a stream synchronisation, which must not sit in front of every ``simulate``."""
        if not ts.is_cuda:
            return ts.detach().to(torch.float32).numpy().tobytes()
        gkey = (ts.data_ptr(), ts._version, tuple(ts.shape), ts.dtype)
        hit = self._grids.get(gkey)
        if hit is None or hit[1] is not ts:
            if len(self._grids) >= 16:
                self._grids.pop(next(iter(self._grids)))
            hit = self._grids[gkey] = (ts.detach().to("cpu", torch.float32).numpy().tobytes(), ts)  # keeps the storage alive
        return hit[0]

    def _key(self, tag, ts, device, info, terminal_unnorm_log_prob, objs=()):
        """(static key, control-parameter versions, keyed objects).  ``objs``: further objects the plan is packed from
        (references, priors, the SDE) besides the terminal target."""
        vers = tuple((p.data_ptr(), p._version) for p in info.base.parameters())
        if info.score_model is not None:
            vers += tuple((p.data_ptr(), p._version) for p in info.score_model.parameters())
        refs = (info.target, info.sde, info.prior, _terminal_target(terminal_unnorm_log_prob)) + tuple(objs)
        fid = (_fid(terminal_unnorm_log_prob), _fid_clip(terminal_unnorm_log_prob))
        return ((tag, self._grid_bytes(ts), str(device), self.precision or pack.default_precision(), info.kind, fid,
                 tuple(_state(o) for o in refs)), vers, refs)

    def _build_plan(self, tag, ts, device, use_ema, terminal_unnorm_log_prob, ref0, steps, objs=(), prior=None,
                    single_gaussian=None):
        """The cached plan of one rollout.  Every loss packs the control, the terminal target, the step table with the
        control's time-only columns and spec.ref_0 (from ``ref0``: the reference term or the prior) the same way;
        ``steps(spec, keep, tsc, pairs)`` does the rest: it sets the loss's own spec fields and returns (table, taus),
        the step rows and the times the control is evaluated at in each row.  ``tag`` and ``objs`` join the cache key;
        ``prior`` and ``single_gaussian`` go to pack.fill_ctrl and pack.fill_ref0."""
        info = self._ctrl(use_ema)
        key = self._key(tag, ts, device, info, terminal_unnorm_log_prob, objs=(ref0,) + tuple(objs))

        def build():
            tsc, pairs = pack._scalar_rows(ts)
            spec = pack.new_spec(self.precision)
            keep: list = []
            weights = pack.fill_ctrl(spec, info, device, keep, prior=prior)
            _terminal(spec, keep, device, terminal_unnorm_log_prob, info)
            spec.K = len(pairs)
            table, taus = steps(spec, keep, tsc, pairs)
            spec_table = pack.finish_table(table, info, taus, device)
            spec.steps = spec_table.data_ptr()
            pack.fill_ref0(spec, ref0, device, keep, single_gaussian)
            linear = spec.kind in (N.ROLLOUT_LINEAR, N.ROLLOUT_EUBO_LINEAR)
            return pack.Plan(spec, keep, weights, spec_table, rows=table.shape[0], noise_steps=spec.K, taus=taus,
                             ito_w=pack.ito_weights(table, spec.ito_form) if linear else None)
        return self._cached(key, build, info, device)


def _terminal(spec, keep, device, terminal_unnorm_log_prob, info):
    """Fills spec.target / clip_target from the terminal log-density callable."""
    target, clip_t = pack.resolve_log_prob(terminal_unnorm_log_prob)
    if info.target is not None and target is not info.target:
        raise NotImplementedError("ScoreCtrl.target_score and terminal_unnorm_log_prob must belong to the same target")
    if target.dim != spec.d:
        raise ValueError("target dimension differs from the drift network's")
    distr, k = target.lrds_distr(device)
    spec.target = distr
    keep.append(k)
    spec.clip_target = float(clip_t) if clip_t is not None else 0.0


def _kl_ctrl_check(info):
    """'kl' / 'kl_ito' train ClippedCtrl drifts only."""
    if info.kind != N.CTRL_CLIPPED:
        raise NotImplementedError("method 'kl' / 'kl_ito' is built for ClippedCtrl (base_zero_init): the adjoint of the "
                                  "score-family controls also needs each target's Hessian-vector product (not built)")


def _kl_start(initial_log_prob, x):
    """log p_prior(x_0) [B], by lrds_distr_eval: the DIS rollout starts its log-weight there (the pre-pass of its train
    plan, rnd_offset = 0), the 'kl' training form at 0 (oc.py:1164-1165), so the kl form subtracts it."""
    return initial_log_prob(x.detach().to(torch.float32)).reshape(-1)


class EMReferenceSDELoss(BaseOCLoss):
    """RDS loss with the Euler-Maruyama integrator (also PIS when ``reference_ctrl`` is None)."""

    _variant = "em"
    _init_cost = False  # DiscreteTimeReversalLossEI: the second log-density is the PRIOR, taken at the start of the rollout

    def __init__(self, *args, reference_ctrl: Callable | None = None, use_rescaling: bool = True, **kwargs):
        super().__init__(*args, **kwargs)
        self.reference_ctrl = reference_ctrl
        self.use_rescaling = use_rescaling

    # per-step coefficients with the reference's own float32 scalar formulas ------------------------------------
    def _rows(self, sde, s, t, T, row):
        tau = T - s
        dt = t - s
        if self._variant == "em":  # oc.py:261-284
            sig = sde.diff(tau)
            row[N.STEP_A], row[N.STEP_B], row[N.STEP_C] = sde.drift_coeff_t(tau), sig, torch.square(sig)
            row[N.STEP_W_COST] = 0.5 * dt
        else:
            ei = self._variant == "ei"
            a, b, c = sde.ei_coeffs(s, t) if ei else sde.ddpm_coeffs(s, t)
            om = sde.omega(s, t) if ei else sde.omega_ddpm(s, t)
            row[N.STEP_A], row[N.STEP_B], row[N.STEP_C] = a, b, c
            row[N.STEP_W_COST], row[N.STEP_W_ITO] = 0.5 * om, torch.sqrt(om)
        row[N.STEP_DT], row[N.STEP_SQRT_DT] = dt, dt.sqrt()

    def _plan(self, ts, device, use_ema, terminal_unnorm_log_prob, reference_log_prob, eubo):
        if self._variant == "em" and not self.use_rescaling:
            raise NotImplementedError("use_rescaling=False is unreachable from the shipped configs (SURVEY.md App. B.4)")
        ref = _resolve_reference(self.reference_ctrl)
        if eubo and ref is None and not self._init_cost:
            raise NotImplementedError("compute_eubo needs a reference control (the reference calls it unconditionally)")

        def steps(spec, keep, tsc, pairs):
            sde = self.sde.host()
            T = tsc[-1]
            K = len(pairs)
            spec.kind = N.ROLLOUT_EUBO_LINEAR if eubo else N.ROLLOUT_LINEAR
            # DDPM-like compute_eubo is the EM formula without the 1/sigma rescaling of the control (oc.py:571-582, 343-346)
            em_formulas = self._variant == "em" or (eubo and self._variant == "ddpm")
            spec.update_form = N.UPDATE_EM if em_formulas else N.UPDATE_AXPY
            spec.ito_form = N.ITO_EM if self._variant == "em" else N.ITO_SCALED
            spec.has_ref_ctrl = int(ref is not None)
            spec.init_cost = int(self._init_cost)
            table = torch.zeros(K, N.STEP_STRIDE)
            if not eubo:
                taus = T - tsc[:-1]
                for k, (s, t) in enumerate(pairs):
                    self._rows(sde, s, t, T, table[k])
            else:  # rows in loop order: reversed time (oc.py:326-329, 541-544)
                times_s, times_t = tsc[:-1].flip((0,)), tsc[1:].flip((0,))
                mean, var = sde.transition_params(T - times_t, T - times_s)
                std = var.sqrt()
                taus = T - times_s
                for i, (s, t) in enumerate(zip(times_s, times_t)):
                    row = table[i]
                    dt = t - s
                    row[N.STEP_EU_A], row[N.STEP_EU_B] = mean[i], std[i]
                    if em_formulas:  # oc.py:343-359
                        sig = sde.diff(T - s)
                        row[N.STEP_B] = sig if self._variant == "em" else 1.0  # divisor of the control (use_rescaling)
                        row[N.STEP_W_COST] = dt * sig ** 2
                        row[N.STEP_EU_C] = 1.0 / mean[i] - 1.0 + sde.drift_coeff_t(T - s) * dt
                        row[N.STEP_W_ITO] = std[i] / mean[i]
                    else:  # oc.py:560-564
                        om = sde.omega(s, t)
                        row[N.STEP_W_COST], row[N.STEP_W_ITO] = om, torch.sqrt(om)
            if ref is not None:
                if ref.dim != spec.d:
                    raise ValueError("reference dimension differs from the model's")
                blk = ref.block_at(taus, device)
                fill_gmm(spec.ref_t, blk, stepped=True)
                keep.append(blk)
            return table, taus
        return self._build_plan((self._variant, eubo, self._init_cost), ts, device, use_ema, terminal_unnorm_log_prob,
                                pack.resolve_log_prob(reference_log_prob)[0], steps, objs=(ref, self.sde))

    def __call__(self, ts, x, terminal_unnorm_log_prob, reference_log_prob, **kw):
        """[TRAINING] (loss, metrics) of oc.py:364-394."""
        return self._train(lambda dev: self._plan(ts, dev, False, terminal_unnorm_log_prob, reference_log_prob, eubo=False),
                           x, **kw)

    def simulate(self, ts, x, terminal_unnorm_log_prob, reference_log_prob, change_sde_ctrl: bool = False,
                 return_traj: bool = False, use_ema: bool = False, noise=None, seed=None, particle_offset: int = 0):
        """Denoising rollout from prior samples x: returns (x_T (B,d), rnd (B,1), xs (K+1,B,d) | None)."""
        self._check_plain(change_sde_ctrl)
        plan = self._plan(ts, x.device, use_ema, terminal_unnorm_log_prob, reference_log_prob, eubo=False)
        return pack.run_rollout(plan, x, noise, self._seed(seed), particle_offset, return_traj)

    def compute_eubo(self, ts, x, terminal_unnorm_log_prob, reference_log_prob, use_ema: bool = False, noise=None,
                     seed=None, particle_offset: int = 0):
        """Noising rollout from target samples x -> rnd (B,1).  Like the reference (oc.py:336-337) the input
        tensor is overwritten with the noised samples."""
        plan = self._plan(ts, x.device, use_ema, terminal_unnorm_log_prob, reference_log_prob, eubo=True)
        x_end, rnd, _ = pack.run_rollout(plan, x, noise, self._seed(seed), particle_offset, False)
        if x.dtype == torch.float32 and x.is_contiguous():
            x.copy_(x_end)
        return rnd

    def eval(self, ts, x, terminal_unnorm_log_prob, reference_log_prob=None, compute_weights: bool = True,
             return_traj: bool = True, use_ema: bool = True, **kw) -> Results:
        samples, rnd, xs = self.simulate(ts, x, terminal_unnorm_log_prob=terminal_unnorm_log_prob,
                                         reference_log_prob=reference_log_prob, change_sde_ctrl=False,
                                         return_traj=return_traj, use_ema=use_ema, **kw)
        return BaseOCLoss.compute_results(rnd, compute_weights=compute_weights, ts=ts, samples=samples, xs=xs)


class EIReferenceSDELoss(EMReferenceSDELoss):
    """RDS loss with the exponential integrator."""

    _variant = "ei"

    def __init__(self, *args, reference_ctrl: Callable | None = None, **kwargs):
        kwargs.pop("use_rescaling", None)
        super().__init__(*args, reference_ctrl=reference_ctrl, use_rescaling=False, **kwargs)


class DDPMLikeReferenceSDELoss(EMReferenceSDELoss):
    """RDS loss with the DDPM-like transition kernel."""

    _variant = "ddpm"

    def __init__(self, *args, reference_ctrl: Callable | None = None, **kwargs):
        kwargs.pop("use_rescaling", None)
        super().__init__(*args, reference_ctrl=reference_ctrl, use_rescaling=False, **kwargs)



class DiscreteTimeReversalLossEI(EIReferenceSDELoss):
    """Discrete-time DIS loss (Appendix D.4 of the paper; oc.py:897-1103): the exponential-integrator rollout of
    EIReferenceSDELoss without a reference control, the log-weight starting at the prior log-density
    (``initial_log_prob(x_0)``) instead of ending with a reference term; ``compute_eubo`` (980-1036) ends with the
    prior log-density at the noised state."""

    _init_cost = True

    def __init__(self, *args, **kwargs):
        kwargs.pop("reference_ctrl", None)
        super().__init__(*args, reference_ctrl=None, **kwargs)

    def __call__(self, ts, x, terminal_unnorm_log_prob, initial_log_prob=None, **kw):
        return super().__call__(ts, x, terminal_unnorm_log_prob, initial_log_prob, **kw)

    def simulate(self, ts, x, terminal_unnorm_log_prob, initial_log_prob=None, train: bool = True,
                 change_sde_ctrl: bool = False, return_traj: bool = False, use_ema: bool = False, **kw):
        if train and self.method in ["kl", "kl_ito"]:
            raise NotImplementedError("the kl training rollout starts the log-weight at 0 (oc.py:926-927) and is "
                                      "differentiated through the trajectory: not built (SURVEY.md 8f item 1)")
        return super().simulate(ts, x, terminal_unnorm_log_prob, initial_log_prob, change_sde_ctrl=change_sde_ctrl,
                                return_traj=return_traj, use_ema=use_ema, **kw)

    def compute_eubo(self, ts, x, terminal_unnorm_log_prob, initial_log_prob=None, use_ema: bool = False, **kw):
        return super().compute_eubo(ts, x, terminal_unnorm_log_prob, initial_log_prob, use_ema=use_ema, **kw)

    def eval(self, ts, x, terminal_unnorm_log_prob, initial_log_prob=None, compute_weights: bool = True,
             return_traj: bool = True, use_ema: bool = True, **kw) -> Results:
        samples, rnd, xs = self.simulate(ts, x, terminal_unnorm_log_prob, initial_log_prob, train=False,
                                         return_traj=return_traj, use_ema=use_ema, **kw)
        return BaseOCLoss.compute_results(rnd, compute_weights=compute_weights, ts=ts, samples=samples, xs=xs)


class ExponentialIntegratorSDELoss(BaseOCLoss):
    """Original DDS loss (forward-time control, exponential integrator of Vargas et al.)."""

    def __init__(self, *args, alpha: float, sigma: float, **kwargs):
        super().__init__(*args, **kwargs)
        self.alpha = alpha
        self.sigma = sigma

    def _plan(self, ts, device, use_ema, terminal_unnorm_log_prob, reference_log_prob, compute_ito_int):
        def steps(spec, keep, tsc, pairs):
            spec.kind = N.ROLLOUT_LINEAR
            spec.update_form = N.UPDATE_AXPY
            spec.ito_form = N.ITO_DDS if compute_ito_int else N.ITO_NONE
            spec.has_ref_ctrl = 0
            table = torch.zeros(len(pairs), N.STEP_STRIDE)
            for k, (s, t) in enumerate(pairs):  # oc.py:1366-1383
                row = table[k]
                dt = t - s
                beta_k = torch.clip(self.alpha * dt.sqrt(), 0, 1)
                alpha_k = torch.sqrt(1.0 - beta_k ** 2)
                row[N.STEP_A] = alpha_k
                row[N.STEP_B] = (beta_k ** 2) * (self.sigma ** 2)
                row[N.STEP_C] = self.sigma * beta_k
                row[N.STEP_W_COST] = 0.5 * (beta_k ** 2 * self.sigma ** 2)
                row[N.STEP_W_ITO] = beta_k
                row[N.STEP_SIGU] = self.sigma
                row[N.STEP_DT], row[N.STEP_SQRT_DT] = dt, dt.sqrt()
            return table, tsc[:-1]
        return self._build_plan(("dds", bool(compute_ito_int), self.alpha, self.sigma), ts, device, use_ema,
                                terminal_unnorm_log_prob, pack.resolve_log_prob(reference_log_prob)[0], steps)

    def __call__(self, ts, x, terminal_unnorm_log_prob, reference_log_prob, **kw):
        """[TRAINING] (loss, metrics) of oc.py:1399-1431 (compute_ito_int = method != 'kl')."""
        ito = self.method != "kl"
        return self._train(lambda dev: self._plan(ts, dev, False, terminal_unnorm_log_prob, reference_log_prob, ito), x, **kw)

    def simulate(self, ts, x, terminal_unnorm_log_prob, reference_log_prob, compute_ito_int: bool = False,
                 change_sde_ctrl: bool = False, return_traj: bool = False, use_ema: bool = False, noise=None,
                 seed=None, particle_offset: int = 0):
        self._check_plain(change_sde_ctrl)
        plan = self._plan(ts, x.device, use_ema, terminal_unnorm_log_prob, reference_log_prob, compute_ito_int)
        return pack.run_rollout(plan, x, noise, self._seed(seed), particle_offset, return_traj)

    def eval(self, ts, x, terminal_unnorm_log_prob, reference_log_prob=None, compute_weights: bool = True,
             return_traj: bool = True, use_ema: bool = True, **kw) -> Results:
        samples, rnd, xs = self.simulate(ts, x, terminal_unnorm_log_prob=terminal_unnorm_log_prob,
                                         reference_log_prob=reference_log_prob, compute_ito_int=compute_weights,
                                         change_sde_ctrl=False, return_traj=return_traj, use_ema=use_ema, **kw)
        return BaseOCLoss.compute_results(rnd, compute_weights=compute_weights, ts=ts, samples=samples, xs=xs)


class TimeReversalLoss(BaseOCLoss):
    """Original DIS loss, evaluation side (Bridge with ``inference_ctrl=None``, solver/oc.py:185-262): Euler-Maruyama
    with the control taken at the loop time, log-weight = initial_log_prob(x_0) + running cost - divergence integral
    [+ Ito term] - target(x_T)  (oc.py:1164-1230)."""

    def __init__(self, *args, inference_ctrl: Callable | None = None, div_estimator: str | None = None,
                 use_rescaling: bool = True, **kwargs):
        super().__init__(*args, **kwargs)
        if inference_ctrl is not None:
            raise NotImplementedError("a learned inference control (the general bridge sampler, divergence through "
                                      "autograd) has no fused kernel; DIS uses inference_ctrl=None (SURVEY.md 8f item 2)")
        if not use_rescaling:
            raise ValueError("use_rescaling must be True for TimeReversalLoss.")
        self.inference_ctrl = None
        self.div_estimator = div_estimator
        self.use_rescaling = use_rescaling

    def _plan(self, ts, device, use_ema, terminal_unnorm_log_prob, initial_log_prob, compute_ito_int, train=False):
        prior, _ = pack.resolve_log_prob(initial_log_prob)

        def steps(spec, keep, tsc, pairs):
            sde = self.sde.host()
            spec.kind = N.ROLLOUT_LINEAR
            spec.update_form = N.UPDATE_EM
            spec.ito_form = N.ITO_EM if compute_ito_int else N.ITO_NONE
            spec.has_ref_ctrl = 0
            table = torch.zeros(len(pairs), N.STEP_STRIDE)
            div = torch.zeros(())
            for k, (s, t) in enumerate(pairs):  # oc.py:1171-1230
                row = table[k]
                dt = t - s
                sig = sde.diff(s)
                # the EM update of the kernel is x + ((-(A x)) + sig u) dt + sig z sqrt(dt): A = -drift_coeff_t(s) gives +drift
                row[N.STEP_A], row[N.STEP_B], row[N.STEP_C] = -sde.drift_coeff_t(s), sig, torch.square(sig)
                row[N.STEP_W_COST] = 0.5 * dt
                row[N.STEP_DT], row[N.STEP_SQRT_DT] = dt, dt.sqrt()
                div = div - sde.int_drift_coeff_t(s, t) * spec.d  # rnd -= sde.drift_div_int(s, t, x), train=False (1217-1218)
            # the training rollout leaves the divergence integral out (`if not train`, oc.py:1217)
            spec.init_cost, spec.rnd_offset = 1, 0.0 if train else float(div)
            return table, tsc[:-1]
        return self._build_plan(("dis", bool(compute_ito_int), bool(train)), ts, device, use_ema, terminal_unnorm_log_prob,
                                prior, steps, objs=(self.sde,), prior=prior,
                                single_gaussian="DIS needs a Gaussian prior (solver/oc.py:207-208)")

    def __call__(self, ts, x, terminal_unnorm_log_prob, initial_log_prob=None, **kw):
        """[TRAINING] (loss, metrics) of oc.py:1240-1272 (compute_ito_int = method != 'kl', train=True)."""
        ito = self.method != "kl"
        return self._train(lambda dev: self._plan(ts, dev, False, terminal_unnorm_log_prob, initial_log_prob, ito, train=True),
                           x, initial_log_prob=initial_log_prob, **kw)

    def simulate(self, ts, x, terminal_unnorm_log_prob, initial_log_prob=None, train: bool = True,
                 compute_ito_int: bool = False, change_sde_ctrl: bool = False, return_traj: bool = False,
                 use_ema: bool = False, noise=None, seed=None, particle_offset: int = 0):
        self._check_plain(change_sde_ctrl)
        plan = self._plan(ts, x.device, use_ema, terminal_unnorm_log_prob, initial_log_prob, compute_ito_int, train=train)
        x_T, rnd, xs = pack.run_rollout(plan, x, noise, self._seed(seed), particle_offset, return_traj)
        if train and self.method in ["kl", "kl_ito"]:
            rnd = rnd - _kl_start(initial_log_prob, x).reshape(rnd.shape)
        return x_T, rnd, xs

    def eval(self, ts, x, terminal_unnorm_log_prob, initial_log_prob=None, compute_weights: bool = True,
             return_traj: bool = True, use_ema: bool = True, **kw) -> Results:
        samples, rnd, xs = self.simulate(ts, x, terminal_unnorm_log_prob=terminal_unnorm_log_prob,
                                         initial_log_prob=initial_log_prob, compute_ito_int=compute_weights,
                                         train=False, return_traj=return_traj, use_ema=use_ema, **kw)
        return BaseOCLoss.compute_results(rnd, compute_weights=compute_weights, ts=ts, samples=samples, xs=xs)


class ControlledLangevinSDELoss(BaseOCLoss):
    """Discrete-time CMCD loss.  The (control, drift) pair evaluated at the end point of step k is reused as the
    start point of step k+1 (the reference recomputes it: 2 network + 2 score evaluations per step)."""

    def __init__(self, *args, use_rescaling: bool = True, **kwargs):
        super().__init__(*args, **kwargs)
        self.use_rescaling = use_rescaling

    def _plan(self, ts, device, use_ema, terminal_unnorm_log_prob, initial_log_prob, eubo):
        if not self.use_rescaling:
            raise NotImplementedError("use_rescaling=False is unreachable from the shipped configs (SURVEY.md App. B.4)")
        if not isinstance(self.sde, ControlledLangevinSDE):
            raise NotImplementedError("CMCD needs a ControlledLangevinSDE")
        prior, _ = pack.resolve_log_prob(initial_log_prob)

        def steps(spec, keep, tsc, pairs):
            sde = self.sde
            K = len(pairs)
            tgt = getattr(sde.target_score, "__self__", None)
            pri = getattr(sde.prior_score, "__self__", None)
            target, _ = pack.resolve_log_prob(terminal_unnorm_log_prob)
            if tgt is not target or pri is not prior:
                raise NotImplementedError("ControlledLangevinSDE scores must be the bound .score of the rollout's "
                                          "target and prior distributions")
            spec.kind = N.ROLLOUT_EUBO_CMCD if eubo else N.ROLLOUT_CMCD
            spec.cmcd_diff = float(sde.diff_coeff)
            spec.cmcd_clip = float(sde.clip_score) if sde.clip_score is not None else 0.0
            table = torch.zeros(K + 1, N.STEP_STRIDE)
            T = sde.terminal_t.detach().to("cpu")
            for k in range(K + 1):
                table[k, N.STEP_FRAC] = tsc[k] / T
                if k < K:
                    dt = tsc[k + 1] - tsc[k]
                    table[k, N.STEP_DT], table[k, N.STEP_SQRT_DT] = dt, dt.sqrt()
            return table, tsc
        return self._build_plan(("cmcd", eubo), ts, device, use_ema, terminal_unnorm_log_prob, prior, steps,
                                objs=(self.sde,),
                                single_gaussian="CMCD needs a (diagonal) Gaussian prior (solver/oc.py:276-277)")

    def __call__(self, ts, x, terminal_unnorm_log_prob, initial_log_prob=None, noise=None, seed=None,
                 particle_offset: int = 0):
        """[TRAINING] (loss, metrics) of oc.py:830-860: method 'lv' / 'lv_traj' (train.cmcd_lv_objective), or 'kl' /
        'kl_ito' for a ClippedCtrl drift (train.cmcd_kl_objective: the pathwise gradient through the trajectory; the Ito
        term is always part of the CMCD log-weight, so the two are the same objective)."""
        from .. import train
        x = self._train_batch(x)
        info = self._ctrl(False)
        if info.kind not in (N.CTRL_CLIPPED, N.CTRL_SCORE):
            raise NotImplementedError("CMCD trains ClippedCtrl / ScoreCtrl drift models")
        if self.method in ("kl", "kl_ito"):
            _kl_ctrl_check(info)
        plan = self._plan(ts, x.device, False, terminal_unnorm_log_prob, initial_log_prob, eubo=False)
        if self.method in ("kl", "kl_ito"):
            return train.cmcd_kl_objective(self, plan, info, x, self._seed(seed), _kl_start(initial_log_prob, x), noise=noise,
                                           particle_offset=particle_offset)
        return train.cmcd_lv_objective(self, plan, info, x, self._seed(seed), noise=noise, particle_offset=particle_offset)

    def simulate(self, ts, x, terminal_unnorm_log_prob, initial_log_prob=None, train: bool = True,
                 change_sde_ctrl: bool = False, return_traj: bool = False, use_ema: bool = False, noise=None,
                 seed=None, particle_offset: int = 0):
        self._check_plain(change_sde_ctrl)
        plan = self._plan(ts, x.device, use_ema, terminal_unnorm_log_prob, initial_log_prob, eubo=False)
        x_T, rnd, xs = pack.run_rollout(plan, x, noise, self._seed(seed), particle_offset, return_traj)
        if train and self.method in ["kl", "kl_ito"]:  # the training form starts the log-weight at 0 (oc.py:695-696)
            rnd = rnd - _kl_start(initial_log_prob, x).reshape(rnd.shape)
        return x_T, rnd, xs

    def compute_eubo(self, ts, x, terminal_unnorm_log_prob, initial_log_prob=None, use_ema: bool = False, noise=None,
                     seed=None, particle_offset: int = 0):
        plan = self._plan(ts, x.device, use_ema, terminal_unnorm_log_prob, initial_log_prob, eubo=True)
        return pack.run_rollout(plan, x, noise, self._seed(seed), particle_offset, False)[1]

    def eval(self, ts, x, terminal_unnorm_log_prob, initial_log_prob=None, compute_weights: bool = True,
             return_traj: bool = True, use_ema: bool = True, **kw) -> Results:
        samples, rnd, xs = self.simulate(ts, x, terminal_unnorm_log_prob=terminal_unnorm_log_prob,
                                         initial_log_prob=initial_log_prob, train=False, return_traj=return_traj,
                                         use_ema=use_ema, **kw)
        return BaseOCLoss.compute_results(rnd, compute_weights=compute_weights, ts=ts, samples=samples, xs=xs)
