"""Diffusion-based samplers with the reference's class names and evaluation entry points
(sde_sampler/solver/oc.py: TrainableDiff 22-182, Bridge 185-262 (DIS), CMCD 264-346, PIS 349-423, DDS 426-492, RDS 495-666; the parts of
sde_sampler/solver/base.py they rely on: seed 52-55, device 57-61, target 64-65).

The reference builds these objects from a Hydra config; Hydra / OmegaConf are not part of this image, so the
constructors take the same information as a plain nested ``dict`` with the YAML's keys and defaults
(``benchmark_utils.default_config``; SURVEY.md Appendix A).  What is kept: ``compute_results`` (two rollouts, the
second one timed as ``eval/sample_time``), ``_compute_results``, ``clipped_target_unnorm_log_prob``,
``RDS.change_reference_type`` / ``reference_ctrl``, ``CMCD.update_prior``, ``state_dict`` of the reference parameters.
Training: ``compute_loss`` / ``_compute_loss`` / ``step`` (solver/base.py:401-457: Adam, loss / gradient guards, gradient
clipping, EMA) drive the LV objective of train.py.  What is not: the run loop with its evaluation schedule,
checkpoints, wandb, plots (control plane; SURVEY.md section 2 rows 17-24).
Every rollout below is ONE fused CUDA kernel launch (losses/oc.py -> csrc/).
"""
from __future__ import annotations

import time
from functools import partial
from typing import Callable

import numpy as np
import torch

from ..distr.base import Distribution
from ..distr.delta import Delta
from ..distr.gauss import Gauss
from ..eq.integrator import EulerIntegrator
from ..eq.sdes import OU, VP, ControlledLangevinSDE, MarginalReference, PinnedBM
from ..losses.oc import BaseOCLoss
from ..utils.common import Results, clip_and_log


def build(cfg: dict | None, **extra):
    """``hydra.utils.instantiate`` for plain dicts: ``{"_target_": callable, "_partial_": bool, **kwargs}``."""
    if cfg is None:
        return None
    kw = {k: (build(v) if isinstance(v, dict) and "_target_" in v else v) for k, v in cfg.items()
          if k not in ("_target_", "_partial_")}
    kw.update(extra)
    target = cfg["_target_"]
    return partial(target, **kw) if cfg.get("_partial_") else target(**kw)


class TrainableDiff(torch.nn.Module):
    """Base class for the diffusion-based variational samplers (evaluation side)."""

    def __init__(self, cfg: dict):
        super().__init__()
        self.cfg = cfg
        if cfg.get("seed") is not None:
            torch.manual_seed(cfg["seed"])
            np.random.seed(cfg["seed"])
        self.device = torch.device(cfg.get("device") or "cuda")
        if self.device.type != "cuda":
            raise RuntimeError("sde_sampler_lrds_b200 solvers run on a CUDA device (no CPU fallback)")
        self.eval_device = self.device
        self.target: Distribution = build(cfg["target"]).to(self.device)
        self.use_ema: bool = bool(cfg.get("use_ema", False))
        self.train_batch_size: int = cfg.get("train_batch_size", 512)
        self.train_timesteps: Callable = build(cfg["train_timesteps"])
        self.train_ts = None
        self.clip_target = cfg.get("clip_target")
        self.eubo_available = True
        self.eval_timesteps: Callable = build(cfg.get("eval_timesteps") or cfg["train_timesteps"])
        self.eval_ts = None
        self.eval_batch_size: int = cfg.get("eval_batch_size", 6000)
        self.eval_integrator = EulerIntegrator()
        self.plot_results = False
        self.n_steps = 0
        self.n_steps_skip = 0
        self.train_steps = cfg.get("train_steps", 0)
        self.ema_steps = cfg.get("ema_steps", 10)
        self.max_grad, self.max_loss, self.scale_loss = cfg.get("max_grad"), cfg.get("max_loss"), cfg.get("scale_loss")
        self.grad_clip = build(cfg.get("grad_clip"))
        self.setup_models()
        self.to(self.device)
        self.optim = None

    # ---- models ---------------------------------------------------------------------------------------------------
    def setup_models(self, langevin_based: bool = False, skip_prior: bool = False):
        if not skip_prior:
            self.prior: Distribution = build(self.cfg["prior"]).to(self.device)
        if langevin_based:
            self.sde = build(self.cfg.get("sde"), prior_score=self.prior.score, target_score=self.target.score)
        else:
            self.sde = build(self.cfg.get("sde"))
        if self.sde is not None:
            self.sde.to(self.device)
        gen = dict(self.cfg["generative_ctrl"])
        extra = {"target_score": self.target.score} if gen.pop("_wants_target_score", False) else {}
        if gen.pop("_wants_sde", False):  # CancelDriftCtrl / LerpCtrl (the reference passes these to every control)
            extra["sde"] = self.sde
        if gen.pop("_wants_prior_score", False):
            extra["prior_score"] = self.prior.score
        self.generative_ctrl = build(gen, **extra).to(self.device)
        if self.use_ema:
            total = self.cfg["train_steps"] / (self.cfg["train_batch_size"] * self.cfg.get("ema_steps", 10))
            alpha = min(1.0, (1.0 - self.cfg.get("ema_decay", 0.995)) / total)
            self.generative_ctrl_ema = torch.optim.swa_utils.AveragedModel(
                self.generative_ctrl, multi_avg_fn=torch.optim.swa_utils.get_ema_multi_avg_fn(1.0 - alpha),
                device=self.device)
            # AveragedModel deep-copies the control, and with it the objects behind its bound target / prior scores and
            # its SDE; the averaged parameters are the control's own, everything else must stay the solver's objects
            for name in ("target_score", "prior_score", "sde"):
                if hasattr(self.generative_ctrl, name):
                    setattr(self.generative_ctrl_ema.module, name, getattr(self.generative_ctrl, name))
        else:
            self.generative_ctrl_ema = self.generative_ctrl

    def setup(self):
        """Reference: target.compute_stats() + checkpoint restore (solver/base.py:108-113)."""
        if hasattr(self.target, "compute_stats"):
            self.target.compute_stats()

    def clipped_target_unnorm_log_prob(self, x: torch.Tensor) -> torch.Tensor:
        return clip_and_log(self.target.unnorm_log_prob(x), max_norm=self.clip_target, name="target")

    # ---- evaluation -----------------------------------------------------------------------------------------------
    def _compute_results(self, ts, x, use_ema=True, compute_weights=True, return_traj=True) -> Results:
        raise NotImplementedError

    # ---- training (solver/oc.py:94-121, solver/base.py:289-300, 401-457) -----------------------------------------------
    def _compute_loss(self, ts, x):
        raise NotImplementedError("training through this solver's loss is not built (SURVEY.md 8f item 1)")

    def compute_loss(self):
        """[TRAINING] the variational loss over a fresh batch of prior samples."""
        x = self.prior.sample((self.train_batch_size,))
        if self.train_ts is None:
            self.train_ts = self.train_timesteps(device=x.device)
        else:
            self.train_ts = self.train_ts.to(x.device)
        return self._compute_loss(self.train_ts, x)

    def trainable_parameters(self):
        return (p for p in self.parameters() if p.requires_grad)

    def setup_optimizer(self):
        """conf/solver/basic_oc_base.yaml: Adam, lr 3e-4 (``cfg['optim']`` = {'_target_': ..., 'lr': ...} overrides)."""
        cfg = dict(self.cfg.get("optim") or {"_target_": torch.optim.Adam, "lr": 3e-4})
        target = cfg.pop("_target_", torch.optim.Adam)
        self.optim = target(list(self.trainable_parameters()), **cfg)

    def step(self, step_id: int = 0) -> dict:
        """One stochastic gradient step (solver/base.py:401-457; no lr schedulers: none is configured by default)."""
        if self.optim is None:
            self.setup_optimizer()
        torch.cuda.synchronize(self.device)
        start_t = time.time()
        self.optim.zero_grad()
        loss, metrics = self.compute_loss()
        if self.scale_loss is not None:
            loss = self.scale_loss * loss
        loss.backward()
        loss_ok = loss.isfinite() if self.max_loss is None else loss.abs() <= self.max_loss
        grads = [p.grad for p in self.trainable_parameters() if p.grad is not None]
        if self.max_grad is None:
            grad_ok = bool(torch.stack([g.isfinite().all() for g in grads]).all())  # one host synchronisation
        else:
            max_grad = torch.stack([g.abs().max() for g in grads]).max()
            grad_ok = max_grad <= self.max_grad
            metrics["train/max_grad"] = max_grad.item()
        if loss_ok and grad_ok:
            if self.grad_clip is not None:
                metrics["train/grad_clip_norm"] = self.grad_clip(self.trainable_parameters()).item()
            self.optim.step()
            if self.use_ema and (step_id % self.ema_steps == 0):
                self.generative_ctrl_ema.update_parameters(self.generative_ctrl)
        else:
            self.n_steps_skip += 1
        torch.cuda.synchronize(self.device)
        metrics.update({"train/time_per_step": time.time() - start_t, "train/loss": loss.item(),
                        "train/skipped_steps": self.n_steps_skip,
                        "train/no_grad": sum(p.grad is None for p in self.trainable_parameters())})
        self.n_steps += 1
        return metrics

    @torch.no_grad()
    def compute_results(self, use_ema=True) -> Results:
        """Two rollouts from the same prior samples, like the reference (solver/oc.py:129-161): the first with
        weights and the full trajectory, the second (timed as eval/sample_time) without."""
        x = self.prior.sample((self.eval_batch_size,))
        if self.eval_ts is None:
            self.eval_ts = self.eval_timesteps(device=x.device)
        else:
            self.eval_ts = self.eval_ts.to(x.device)
        ts = self.eval_ts
        results = self._compute_results(ts, x, use_ema=use_ema, compute_weights=True)
        assert results.xs.shape == (len(ts), *results.samples.shape)
        torch.cuda.synchronize(x.device)
        start_time = time.time()
        add_results = self._compute_results(ts, x, use_ema=use_ema, compute_weights=False, return_traj=False)
        torch.cuda.synchronize(x.device)
        results.metrics["eval/sample_time"] = time.time() - start_time
        results.metrics.update(add_results.metrics)
        results.log_norm_const_preds.update(add_results.log_norm_const_preds)
        return results

    evaluate = compute_results


class Bridge(TrainableDiff):
    """DIS (``inference_ctrl`` absent; solver/oc.py:185-262).  The general bridge sampler with a learned inference
    control needs the divergence of a network through autograd and has no fused kernel."""

    def setup_models(self):
        super().setup_models()
        if self.cfg.get("inference_ctrl") is not None:
            raise NotImplementedError("Bridge with a learned inference_ctrl has no B200 kernel (SURVEY.md 8f item 2); "
                                      "DIS (inference_ctrl=None) does")
        self.inference_ctrl = None
        self.inference_sde = build(self.cfg["sde"]).to(self.device)
        if not isinstance(self.prior, Gauss):
            raise ValueError("Can only be used with Gaussian prior.")
        self.loss: BaseOCLoss = build(self.cfg["loss"], generative_ctrl=self.generative_ctrl,
                                      generative_ctrl_ema=self.generative_ctrl_ema, sde=self.sde,
                                      inference_ctrl=self.inference_ctrl,
                                      filter_samples=getattr(self.target, "filter", None))

    def _compute_loss(self, ts, x):
        return self.loss(ts, x, self.clipped_target_unnorm_log_prob, initial_log_prob=self.prior.log_prob)

    def _compute_results(self, ts, x, use_ema=True, compute_weights=True, return_traj=True) -> Results:
        return self.loss.eval(ts, x, self.clipped_target_unnorm_log_prob, use_ema=use_ema,
                              initial_log_prob=self.prior.log_prob, compute_weights=compute_weights,
                              return_traj=return_traj)


class CMCD(TrainableDiff):
    def setup_models(self, skip_prior: bool = False):
        super().setup_models(langevin_based=True, skip_prior=skip_prior)
        if not isinstance(self.prior, Gauss):
            raise ValueError("Can only be used with gaussian prior.")
        self.inference_sde = build(self.cfg["sde"], prior_score=self.prior.score, target_score=self.target.score)
        self.loss: BaseOCLoss = build(self.cfg["loss"], generative_ctrl=self.generative_ctrl,
                                      generative_ctrl_ema=self.generative_ctrl_ema, sde=self.sde,
                                      filter_samples=getattr(self.target, "filter", None))

    def update_prior(self, mean, var):
        """Diagonal Gaussian base distribution with the given mean / variance (solver/oc.py:291-303)."""
        if var.ndim == 2:
            raise NotImplementedError("full-covariance priors are a later row (SURVEY.md 8f item 2)")
        self.prior = Gauss(dim=mean.shape[0], loc=mean, scale=var.sqrt()).to(self.device)
        self.setup_models(skip_prior=True)
        self.to(self.device)

    def _compute_loss(self, ts, x):
        return self.loss(ts, x, self.clipped_target_unnorm_log_prob, initial_log_prob=self.prior.log_prob)

    def _compute_results(self, ts, x, use_ema=True, compute_weights=True, return_traj=True) -> Results:
        return self.loss.eval(ts, x, self.clipped_target_unnorm_log_prob, use_ema=use_ema,
                              initial_log_prob=self.prior.log_prob, compute_weights=compute_weights,
                              return_traj=return_traj)


class PIS(TrainableDiff):
    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.eubo_available = False

    def setup_models(self):
        super().setup_models()
        if not isinstance(self.prior, Delta):
            raise ValueError("Can only be used with dirac delta prior.")
        host = self.sde.host()
        self.reference_distr = host.marginal_distr(t=host.terminal_t, x_init=self.prior.loc.detach().cpu()).to(self.device)
        self.loss: BaseOCLoss = build(self.cfg["loss"], generative_ctrl=self.generative_ctrl,
                                      generative_ctrl_ema=self.generative_ctrl_ema, sde=self.sde,
                                      filter_samples=getattr(self.target, "filter", None))

    def _compute_loss(self, ts, x):
        return self.loss(ts, x, self.clipped_target_unnorm_log_prob, self.reference_distr.log_prob)

    def _compute_results(self, ts, x, use_ema=True, compute_weights=True, return_traj=True) -> Results:
        return self.loss.eval(ts, x, self.clipped_target_unnorm_log_prob, self.reference_distr.log_prob, use_ema=use_ema,
                              compute_weights=compute_weights, return_traj=return_traj)


class DDS(TrainableDiff):
    def __init__(self, *args, **kwargs):
        super().__init__(*args, **kwargs)
        self.eubo_available = False

    def setup_models(self):
        super().setup_models()
        if not isinstance(self.prior, Gauss):
            raise ValueError("Can only be used with Gaussian prior.")
        self.reference_distr = self.prior
        self.loss: BaseOCLoss = build(self.cfg["loss"], generative_ctrl=self.generative_ctrl,
                                      generative_ctrl_ema=self.generative_ctrl_ema, sde=self.sde,
                                      filter_samples=getattr(self.target, "filter", None))

    def _compute_loss(self, ts, x):
        return self.loss(ts, x, self.clipped_target_unnorm_log_prob, self.reference_distr.log_prob)

    def _compute_results(self, ts, x, use_ema=True, compute_weights=True, return_traj=True) -> Results:
        return self.loss.eval(ts, x, self.clipped_target_unnorm_log_prob, self.reference_distr.log_prob, use_ema=use_ema,
                              compute_weights=compute_weights, return_traj=return_traj)


class RDS(TrainableDiff):
    def setup_models(self):
        super().setup_models()
        self.inference_sde = build(self.cfg["sde"]).to(self.device)
        self.change_reference_type(ref_type="default")
        # the loss keeps the BOUND METHOD: switching the reference later takes effect (SURVEY.md 3.4)
        self.loss: BaseOCLoss = build(self.cfg["loss"], generative_ctrl=self.generative_ctrl,
                                      generative_ctrl_ema=self.generative_ctrl_ema, sde=self.sde,
                                      reference_ctrl=self.reference_ctrl,
                                      filter_samples=getattr(self.target, "filter", None))

    def change_reference_type(self, ref_type="default", net=None, eps=None, mean=None, var=None, means=None,
                              variances=None, weights=None):
        """Reference distribution and its time marginals (solver/oc.py:513-588): 'default' (from prior and SDE),
        'gaussian' (mean, var = diagonal [d], full [d][d] or the eigen form (eigenvalues, eigenvectors)), 'gmm' (means,
        variances = diagonal [M][d], full [M][d][d] or the eigen form, weights).  'nn' is a later row (SURVEY.md 8f
        item 3)."""
        if ref_type == "default":
            loc = self.prior.loc.detach().flatten().cpu()
            if isinstance(self.sde, VP):
                var0 = torch.square(self.prior.scale.detach()).flatten().cpu()
            elif isinstance(self.sde, PinnedBM):
                h = self.sde.host()
                var0 = h.terminal_t * h.diff_coeff ** 2 * torch.ones_like(loc)
            else:
                raise ValueError(f"Default reference for SDE type {type(self.sde)} is not supported.")
            self.reference_distr_utils = {"x_init": loc, "var_init": var0}
            self.reference_score_t = MarginalReference(self.sde, "gaussian", x_init=loc, var_init=var0)
        elif ref_type == "gaussian":
            var = tuple(v.float().cpu() for v in var) if isinstance(var, tuple) else var.float().cpu()
            self.reference_distr_utils = {"x_init": mean.float().cpu(), "var_init": var}
            self.reference_score_t = MarginalReference(self.sde, "gaussian", **self.reference_distr_utils)
        elif ref_type == "gmm":
            variances = tuple(v.float().cpu() for v in variances) if isinstance(variances, tuple) else variances.float().cpu()
            self.reference_distr_utils = {"means_init": means.float().cpu(), "variances_init": variances,
                                          "weights_init": weights.float().cpu()}
            self.reference_score_t = MarginalReference(self.sde, "gmm", **self.reference_distr_utils)
        elif ref_type == "nn":
            raise NotImplementedError("neural references need the score network on the GPU path (SURVEY.md 8f item 3)")
        else:
            raise NotImplementedError(f"Reference type {ref_type} is unknown.")
        self.reference_distr = self.reference_score_t.distr_at(torch.tensor(0.0), self.device)
        self.ref_type = ref_type
        if isinstance(getattr(self, "loss", None), BaseOCLoss):
            self.loss.clear_plans()  # plans packed from the previous reference must not be served again

    def reference_ctrl(self, t: torch.Tensor, x: torch.Tensor) -> torch.Tensor:
        return self.reference_score_t(t, x)

    def _compute_loss(self, ts, x):
        return self.loss(ts, x, self.clipped_target_unnorm_log_prob, self.reference_distr.log_prob)

    def _compute_results(self, ts, x, use_ema=True, compute_weights=True, return_traj=True) -> Results:
        return self.loss.eval(ts, x, self.clipped_target_unnorm_log_prob, self.reference_distr.log_prob, use_ema=use_ema,
                              compute_weights=compute_weights, return_traj=return_traj)

    def state_dict(self, *args, **kwargs):
        sd = super().state_dict(*args, **kwargs)
        sd.update({f"ref_{k}": v for k, v in self.reference_distr_utils.items()})
        sd["ref_type"] = self.ref_type
        return sd

    def load_state_dict(self, state_dict, *args, **kwargs):
        state_dict = dict(state_dict)
        ref_type = state_dict.pop("ref_type", None)
        ref = {k[4:]: state_dict.pop(k) for k in list(state_dict) if k.startswith("ref_")}
        out = super().load_state_dict(state_dict, *args, **kwargs)
        if ref_type == "gaussian":
            self.change_reference_type("gaussian", mean=ref["x_init"], var=ref["var_init"])
        elif ref_type == "gmm":
            self.change_reference_type("gmm", weights=ref["weights_init"], means=ref["means_init"],
                                       variances=ref["variances_init"])
        return out
