"""``make_model`` and ``make_target_details`` with the reference's signatures, selectors and forbidden combinations
(experiments/benchmark_utils.py:22-265), without Hydra: ``default_config`` resolves the same YAML defaults
(conf/solver/*.yaml and the groups they pull in; SURVEY.md Appendix A) into a plain dict and ``make_model`` applies
the same patches in the same order (benchmark_utils.py:176-262).

Differences, all loud: the U-Net controls and 'nn' references raise NotImplementedError (rows of SURVEY.md 8f), sample-based metrics (Sinkhorn / MMD / KS) are not attached, and the
logistic-regression targets read ``<data_dir>/<name>.pkl`` (pass ``target_details['data_dir']`` or set
``LRDS_DATA_DIR``; the datasets are not redistributed here).
"""
from __future__ import annotations

import os
from functools import partial
from pathlib import Path

import torch

from .distr.delta import Delta
from .distr.gauss import BracketTwoModes, IsotropicGauss, ManyModes, TwoModes
from .distr.logistic_regression import LogisticRegression
from .distr.phi_four import PhiFour
from .eq.sdes import VP, ControlledLangevinSDE, CosineVP, PinnedBM, ScaledBM
from .losses import oc as L
from .models.mlp import FourierMLP, TimeEmbed
from .models.reparam import CancelDriftCtrl, ClippedCtrl, LerpCtrl, ScoreCtrl
from .models.utils import init_bias_uniform_constant, init_bias_uniform_zeros, kaiming_uniform_zeros_
from .solver import oc as S
from .utils.common import get_timesteps

solver_types = {"dds_orig": "dds", "pis_orig": "pis", "dis_orig": "dis", "cmcd": "cmcd", "vp-ref": "vp_rds",
                "pbm-ref": "pbm_rds"}
model_types = {"target_informed_zero_init": "score", "target_informed_unet_zero_init": "score_unet",
               "target_informed_langevin_init": "langevin_init", "target_informed_lerp_tempering": "lerp",
               "base_zero_init": "basic", "unet_zero_init": "basic_unet"}


def make_target_details(target_name, **kwargs):
    """experiments/benchmark_utils.py:41-93 (including its typo: 'ill_conditioned' always defaults to 'medium')."""
    assert target_name in ["two_modes", "bracket_two_modes", "two_modes_full", "many_modes", "rings", "checkerboard",
                           "phi_four", "mnist", "mnist_zero_one", "cancer", "credit", "ionosphere", "sonar"]
    if target_name in ["two_modes", "two_modes_full"]:
        return {"name": target_name, "dim": kwargs.get("dim", 5),
                "ill_conditioned": kwargs.get("ill_conditioned", "not" if target_name == "target_name" else "medium"),
                "a": kwargs.get("a", 1.0)}
    if target_name == "bracket_two_modes":
        return {"name": target_name, "dim": kwargs.get("dim", 5), "a": kwargs.get("a", 0.75)}
    if target_name == "many_modes":
        return {"name": "many_modes", "dim": kwargs.get("dim", 5), "n_modes": kwargs.get("n_modes", 4),
                "mixture_weight_factor": kwargs.get("mixture_weight_factor", 3.0), "var": kwargs.get("var", 0.5)}
    if target_name == "phi_four":
        return {"name": "phi_four", "dim": kwargs.get("dim", 100), "b": kwargs.get("b", 0.0)}
    return {"name": target_name}


# ---- YAML defaults as plain dicts ---------------------------------------------------------------------------------
def _target_cfg(details: dict) -> dict:
    name = details["name"]
    if name == "two_modes":  # conf/target/two_modes.yaml
        cfg = {"_target_": TwoModes, "dim": 5, "a": 1.0, "centered": False, "ill_conditioned": "not",
               "n_reference_samples": 16384}
    elif name == "bracket_two_modes":  # conf/target/bracket_two_modes.yaml
        cfg = {"_target_": BracketTwoModes, "dim": 5, "a": 1.0, "n_reference_samples": 16384}
    elif name == "many_modes":  # conf/target/many_modes.yaml
        cfg = {"_target_": ManyModes, "n_modes": 4, "dim": 8, "seed_loc": 42, "mixture_weight_factor": 3.0, "var": 0.5,
               "n_reference_samples": 10000}
    elif name == "phi_four":  # conf/target/phi_four.yaml
        cfg = {"_target_": PhiFour, "dim": 100, "a": 0.1, "b": 0.0, "dim_phys": 1, "beta": 20.0}
    elif name in ("sonar", "ionosphere", "cancer", "credit"):  # conf/target/{sonar,ionosphere,cancer,credit}.yaml
        prm = {"sonar": (61, -2.5, 0.5, 4.5), "ionosphere": (34, 4.25, 0.25, 5.25), "cancer": (31, 31.0, 2.0, 3.75),
               "credit": (25, 3.25, 0.5, 1.25)}[name]
        data_dir = details.get("data_dir") or os.environ.get("LRDS_DATA_DIR")
        cfg = {"_target_": LogisticRegression, "dim": prm[0], "data_type": name, "intercept_mean": prm[1],
               "intercept_scale": prm[2], "weight_scale": prm[3],
               "data_dir": Path(data_dir) if data_dir else None}
    else:
        raise NotImplementedError(f"target {name!r} has no B200 kernel (rows of SURVEY.md section 2 marked out of scope)")
    for k, v in details.items():
        if k not in ("name", "data_dir"):
            cfg[k] = v
    return cfg


def _fouriermlp(dim):  # conf/model/base/fouriermlp.yaml
    return {"_target_": FourierMLP, "dim": dim, "num_layers": 4, "channels": 64, "activation": {"_target_": torch.nn.GELU},
            "last_bias_init": {"_target_": init_bias_uniform_zeros, "_partial_": True},
            "last_weight_init": {"_target_": kaiming_uniform_zeros_, "_partial_": True}, "use_angle_encoding": False}


def _model_cfg(model_type: str, dim: int) -> dict:
    if model_types[model_type] == "basic":  # conf/model/basic.yaml
        return {"_target_": ClippedCtrl, "base_model": _fouriermlp(dim), "clip_model": 1e4}
    if model_types[model_type] == "score":  # conf/model/score.yaml + base/time_embed.yaml
        return {"_target_": ScoreCtrl, "_wants_target_score": True, "base_model": _fouriermlp(dim),
                "score_model": {"_target_": TimeEmbed, "dim_out": 1, "num_layers": 4, "channels": 64,
                                "activation": {"_target_": torch.nn.GELU},
                                "last_bias_init": {"_target_": init_bias_uniform_zeros, "_partial_": True},
                                "last_weight_init": {"_target_": kaiming_uniform_zeros_, "_partial_": True}},
                "detach_score": False, "clip_score": 1e4, "clip_model": 1e4, "scale_score": 1.0}
    if model_types[model_type] in ("langevin_init", "lerp"):  # conf/model/langevin_init.yaml, conf/model/lerp.yaml
        cfg = _model_cfg("target_informed_zero_init", dim)
        cfg["score_model"]["last_bias_init"] = {"_target_": init_bias_uniform_constant, "val": 1.0, "_partial_": True}
        cfg["_wants_sde"] = True
        if model_types[model_type] == "langevin_init":
            cfg.update({"_target_": CancelDriftCtrl, "langevin_init": True})
            del cfg["scale_score"]
        else:
            cfg.update({"_target_": LerpCtrl, "_wants_prior_score": True, "hard_constraint": False})
        return cfg
    raise NotImplementedError(f"model_type {model_type!r} has no B200 kernel yet (SURVEY.md 8f item 3)")


def default_config(solver_type: str, model_type: str, loss_type: str, target_details: dict, force_vp20=False,
                   force_vp_cosine=False) -> dict:
    """The resolved conf/solver/<solver>.yaml tree (before make_model's patches)."""
    target = _target_cfg(target_details)
    dim = target["dim"]
    base = {"seed": 1, "device": None, "train_steps": 10000, "train_batch_size": 512, "eval_batch_size": 6000,
            "use_ema": False, "ema_decay": 0.995, "ema_steps": 10, "clip_target": None, "target": target,
            "train_timesteps": {"_target_": get_timesteps, "_partial_": True, "start": 0.0, "end": None, "steps": 100},
            "generative_ctrl": _model_cfg(model_type, dim)}
    # every solver YAML pulls the *_lv loss file and make_model only overrides loss.method: max_rnd stays 1e8 for 'kl' too
    em_loss = {"_target_": L.EMReferenceSDELoss, "method": loss_type, "traj_per_sample": 1,
               "max_rnd": 1e8, "sde_ctrl_noise": None, "sde_ctrl_dropout": None}
    name = solver_types[solver_type]
    if name == "vp_rds":
        sde = {"_target_": VP, "diff_coeff_sq_min": 0.1, "diff_coeff_sq_max": 20.0 if force_vp20 else 10.0,
               "scale_diff_coeff": 1.0, "terminal_t": 1.0}
        if force_vp_cosine:  # conf/sde/vp_cos.yaml
            sde = {"_target_": CosineVP, "c": 0.008, "scale_diff_coeff": 1.0, "terminal_t": 1.0}
        base.update(solver=S.RDS, sde=sde, loss=em_loss, prior={"_target_": IsotropicGauss, "dim": dim, "scale": "${sde.scale_diff_coeff}"})
    elif name == "pbm_rds":
        sde = {"_target_": PinnedBM, "diff_coeff": 0.4472135954999579, "terminal_t": 5.0}
        base.update(solver=S.RDS, sde=sde, loss=em_loss, prior={"_target_": Delta, "dim": dim})
        base["train_timesteps"]["start"] = 1e-4
    elif name == "pis":
        sde = {"_target_": ScaledBM, "diff_coeff": 0.4472135954999579, "terminal_t": 5.0}
        base.update(solver=S.PIS, sde=sde, loss=em_loss, prior={"_target_": Delta, "dim": dim})
    elif name == "dds":
        loss = {"_target_": L.ExponentialIntegratorSDELoss, "method": loss_type, "traj_per_sample": 1,
                "max_rnd": 1e8, "alpha": 1.0, "sigma": 1.0}
        base.update(solver=S.DDS, sde=None, loss=loss, prior={"_target_": IsotropicGauss, "dim": dim, "scale": "${loss.sigma}"})
        base["train_timesteps"].update(rescale_t="cosine", steps=None, end=6.4, dt=0.05)
    elif name == "cmcd":
        sde = {"_target_": ControlledLangevinSDE, "diff_coeff": 1.0, "terminal_t": 1.0, "clip_score": 1e5}
        loss = {"_target_": L.ControlledLangevinSDELoss, "method": loss_type, "traj_per_sample": 1, "max_rnd": None,
                "sde_ctrl_noise": None, "sde_ctrl_dropout": None}
        base.update(solver=S.CMCD, sde=sde, loss=loss, prior={"_target_": IsotropicGauss, "dim": dim, "scale": 5.0})
    elif name == "dis":  # conf/solver/dis.yaml + conf/loss/time_reversal[_lv].yaml
        sde = {"_target_": VP, "diff_coeff_sq_min": 0.1, "diff_coeff_sq_max": 20.0 if force_vp20 else 10.0,
               "scale_diff_coeff": 1.0, "terminal_t": 1.0}
        if force_vp_cosine:  # conf/sde/vp_cos.yaml (make_model refuses it for DIS; the tree composes all the same)
            sde = {"_target_": CosineVP, "c": 0.008, "scale_diff_coeff": 1.0, "terminal_t": 1.0}
        loss = {"_target_": L.TimeReversalLoss, "method": loss_type, "traj_per_sample": 1,
                "max_rnd": 1e8, "sde_ctrl_noise": None, "sde_ctrl_dropout": None}
        base.update(solver=S.Bridge, sde=sde, loss=loss,
                    prior={"_target_": IsotropicGauss, "dim": dim, "scale": "${sde.scale_diff_coeff}"})
    else:
        raise NotImplementedError(f"solver {solver_type!r} is unknown")
    return base


def _resolve(cfg: dict):
    """The three interpolations the YAMLs use, resolved AFTER the patches like OmegaConf does (solver/base.py:38-39)."""
    if cfg["train_timesteps"].get("end") is None:
        cfg["train_timesteps"]["end"] = cfg["sde"]["terminal_t"]
    scale = cfg["prior"].get("scale")
    if scale == "${sde.scale_diff_coeff}":
        cfg["prior"]["scale"] = cfg["sde"]["scale_diff_coeff"]
    elif scale == "${loss.sigma}":
        cfg["prior"]["scale"] = cfg["loss"]["sigma"]
    cfg["eval_timesteps"] = dict(cfg["train_timesteps"])
    return cfg


def mcmc_sample(device, target, x_init, mcmc_type="mala", step_size=1e-3, n_chains_per_mode=4, dataset_length=50000,
                n_warmup_steps=512, skip_chain_per_mode=False, target_log_prob_and_grad=None, adapt_step_size=True,
                shuffle=True, verbose=False, seed=None):
    """experiments/benchmark_utils.py:268-333 with the chain loop in one kernel launch (additions/mcmc.py).  Returns the
    [n_mcmc_steps * n_chains, d] dataset on the CPU like the reference."""
    from .additions.mcmc import mala_chains
    if mcmc_type not in ("mala", "rwmh"):  # the reference runs rwmh_step for every other value (benchmark_utils.py:308-314)
        raise NotImplementedError("mcmc_type must be 'mala' or 'rwmh'")
    if target_log_prob_and_grad is not None:
        raise NotImplementedError("a custom target_log_prob_and_grad cannot run inside the kernel; pass a Distribution")
    x_init = x_init.to(device)
    if skip_chain_per_mode:
        y_init = x_init.clone()
    else:
        y_init = torch.concat([x_init[i].unsqueeze(0).expand((n_chains_per_mode, -1)) for i in range(x_init.shape[0])], dim=0)
    n_chains = y_init.shape[0]
    n_mcmc_steps = int(dataset_length / n_chains)
    ys, _ = mala_chains(target, y_init, step_size, n_warmup_steps, n_mcmc_steps, adapt_step_size=adapt_step_size, seed=seed,
                        mcmc_type=mcmc_type)
    ret = ys.cpu().view((-1, *x_init.shape[1:]))
    return ret[torch.randperm(ret.shape[0])] if shuffle else ret


def fit_gmm(n_components, dataset, means_init=None, em_type="diag", max_iter=1000):
    """experiments/benchmark_utils.py:336-365: sklearn's EM over the MCMC data set (host library code in the reference
    as well), tried over the reference's ladder of ``reg_covar`` values.  Returns (weights, means, variances) as the
    ``*_ref`` entries of ``solver_details``: variances [M][d] for em_type='diag', covariance matrices [M][d][d] for
    em_type='full' (the full-covariance reference, GMMFull)."""
    from sklearn.mixture import GaussianMixture
    if em_type not in ("diag", "full"):
        raise NotImplementedError(f"em_type {em_type!r}: the references are built for 'diag' and 'full' covariances")
    from .distr.gauss import GMM, GMMFull
    for reg_covar in [1e-6, 5e-5, 1e-5, 5e-4, 1e-4, 5e-3, 1e-3, 5e-2, 1e-2]:
        try:
            dim = dataset.shape[-1]
            gmm = GaussianMixture(n_components=n_components, covariance_type=em_type,
                                  means_init=means_init.cpu().numpy() if means_init is not None else None,
                                  reg_covar=reg_covar, max_iter=max_iter)
            gmm = gmm.fit(dataset.view((-1, dataset.shape[-1])).numpy())
            weights = torch.from_numpy(gmm.weights_).float()
            means = torch.from_numpy(gmm.means_).float()
            variances = torch.from_numpy(gmm.covariances_).float()
            if em_type == "full":
                GMMFull(dim=dim, loc=means, covariance_matrix=variances, mixture_weights=weights)
            else:
                GMM(dim=dim, loc=means, scale=variances.sqrt(), mixture_weights=weights)
            return weights, means, variances
        except Exception:  # noqa: BLE001  (the reference retries on any failure with the next regularisation)
            continue
    raise ValueError("Couldn't fit a GMM on this dataset.")


def make_model(solver_type, ref_type, loss_type, integrator_type, model_type, time_type, solver_details, target_details,
               training_details, optim_details=None, n_steps=100, force_base_zero_init=False, use_ema=False,
               force_vp20=False, force_vp_cosine=False, compute_samples_based_metrics=True, force_T_cosine=None,
               device=None, precision=None):
    """experiments/benchmark_utils.py:96-265.  ``device`` / ``precision`` are the only additions."""
    assert solver_type in solver_types
    assert ref_type in ["default", "gaussian", "gmm", "nn"]
    assert loss_type in ["kl", "lv"]
    assert integrator_type in ["em", "ei", "ddpm_like"]
    assert model_type in model_types
    assert time_type in ["uniform", "snr"]
    assert isinstance(solver_details, dict)
    assert isinstance(target_details, dict) and ("name" in target_details)
    assert isinstance(training_details, dict)

    # Exceptions for orig models (benchmark_utils.py:111-131)
    if ("orig" in solver_type) or ("dis" in solver_type) or ("cmcd" in solver_type):
        if not ((model_type == "base_zero_init") and force_base_zero_init):
            if (solver_type == "dds_orig") and (model_type not in ["target_informed_zero_init", "target_informed_unet_zero_init"]):
                raise ValueError("Only target_informed_zero_init model is supported.")
            if (solver_type == "pis_orig") and (model_type not in ["target_informed_zero_init", "target_informed_unet_zero_init"]):
                raise ValueError("Only target_informed_zero_init model is supported.")
            if ("dis" in solver_type) and (model_type == "base_zero_init"):
                raise ValueError("Model base_zero_init is not supported.")
            if (solver_type == "cmcd") and (model_type == "base_zero_init"):
                raise ValueError("Only base_zero_init is supported for CMCD.")
        if not (time_type == "uniform"):
            raise ValueError("Only uniform time discretisation is supported for orig/cmcd models.")
        if not (integrator_type == "em"):
            raise ValueError("Can't use EI or DDPM-like discretization with orig models.")
        if force_vp20 and (solver_type != "dis_orig"):
            raise ValueError("Can't use vp_20 for orig models other than DIS.")
        if force_vp_cosine:
            raise ValueError("Can't use vp_cosine for orig models.")
    # Exceptions for the reference-based models (133-143)
    if "ref" in solver_type:
        if model_type == "target_informed_lerp_tempering":
            raise ValueError("Model target_informed_lerp_tempering is not supported.")
        if (solver_type == "pbm-ref") and (time_type == "uniform"):
            raise ValueError("PBM schedule is unstable with uniform time discretization.")
        if (integrator_type == "ddpm_like") and (time_type == "uniform"):
            raise ValueError("Using the integration scheme from DDPM with uniform times is unstable.")
    if force_vp20 and force_vp_cosine:
        raise ValueError("Can't use vp_20 and vp_cosine at the same time.")
    if (solver_type == "pbm-ref") and (force_vp20 or force_vp_cosine):
        raise ValueError("Can't use vp_20 or vp_cosine with PBM.")
    if ((ref_type != "default") and ("ref" not in solver_type)) and (solver_type != "cmcd"):
        raise ValueError("Only ref models can use a non-default ref.")
    if (solver_type == "cmcd") and (ref_type not in ["default", "gaussian"]):
        raise ValueError("Can't use ref other than gaussian for CMCD.")
    if (model_type == "target_informed_langevin_init") and (integrator_type in ["ei", "ddpm_like"]):
        raise ValueError("Can't use EI or DDPM-like with Langevin score.")
    if (model_type == "target_informed_langevin_init") and ("ref" in solver_type):
        raise NotImplementedError("the reference wraps this control in RemoveReferenceCtrl(..., sde=None) whose forward "
                                  "dereferences the missing sde (benchmark_utils.py:261-262, models/reparam.py:58-64): "
                                  "there is no reference behaviour to reproduce")

    # Build the config and apply the reference's patches (162-210)
    cfg = default_config(solver_type, model_type, loss_type, target_details, force_vp20=force_vp20,
                         force_vp_cosine=force_vp_cosine)
    cfg["device"] = device
    cfg["use_ema"] = use_ema
    cfg["train_steps"] = training_details["train_steps"]
    cfg["train_batch_size"] = training_details["train_batch_size"]
    cfg["eval_batch_size"] = training_details["eval_batch_size"]
    if solver_type != "dds_orig":
        cfg["train_timesteps"]["steps"] = n_steps
    if time_type == "snr":
        cfg["train_timesteps"]["start"] = 1e-4
        cfg["train_timesteps"]["end"] = cfg["sde"]["terminal_t"] - 1e-4
    if force_vp_cosine:  # benchmark_utils.py:191-192
        cfg["train_timesteps"]["start"] = 1e-3
    if ("ref" in solver_type) and (integrator_type == "ei"):
        cfg["loss"]["_target_"] = L.EIReferenceSDELoss
    if ("ref" in solver_type) and (integrator_type == "ddpm_like"):
        cfg["loss"]["_target_"] = L.DDPMLikeReferenceSDELoss
    if solver_type == "dds_orig":
        cfg["loss"]["sigma"] = solver_details["sigma"]
        if force_T_cosine is not None:
            cfg["train_timesteps"]["end"] = force_T_cosine
    elif solver_type == "pis_orig":
        cfg["sde"]["diff_coeff"] = solver_details["sigma"]
    elif (solver_type == "dis_orig") or (solver_type == "dis_discrete"):
        cfg["sde"]["scale_diff_coeff"] = solver_details["sigma"]
    elif ("ref" in solver_type) and (ref_type == "default"):
        if "pbm" in solver_type:
            cfg["sde"]["diff_coeff"] = solver_details["sigma"]
        if "vp" in solver_type:
            cfg["sde"]["scale_diff_coeff"] = solver_details["sigma"]
    if precision is not None:
        cfg["loss"]["precision"] = precision
    _resolve(cfg)

    model = cfg["solver"](cfg)
    model.setup()

    # Change the reference distributions (229-253)
    if "ref" in solver_type:
        if ref_type == "gaussian":
            model.change_reference_type(ref_type="gaussian", mean=solver_details["mean_ref"], var=solver_details["var_ref"])
        elif ref_type == "gmm":
            model.change_reference_type(ref_type="gmm", weights=solver_details["weights_ref"],
                                        means=solver_details["means_ref"], variances=solver_details["variances_ref"])
        elif ref_type == "nn":
            model.change_reference_type(ref_type="nn", net=solver_details["net"],
                                        eps=torch.tensor(cfg["train_timesteps"]["start"]))
    if ("cmcd" in solver_type) and (ref_type == "gaussian"):
        model.update_prior(mean=solver_details["mean"], var=solver_details["var"])

    # Set the type of time (256-258)
    if time_type == "snr":
        model.train_timesteps = partial(get_timesteps, **model.train_timesteps.keywords, sde=model.sde)
        model.eval_timesteps = partial(get_timesteps, **model.eval_timesteps.keywords, sde=model.sde)
    return model
