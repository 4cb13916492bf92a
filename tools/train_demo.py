#!/usr/bin/env python
"""End-to-end training through the fused rollout: make_model(...) over TwoModes d=2, 200 Adam steps (batch 512, lr 3e-3,
K=50) per solver, evaluation log-variance / ELBO before and after, wall time per step:   python tools/train_demo.py"""
import os, sys, math, time; sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from sde_sampler_lrds_b200 import benchmark_utils as BU

# throwaway model: library loading, cuBLAS handles and the first launches stay out of the per-step times below
_w = BU.make_model(solver_type="vp-ref", ref_type="default", loss_type="lv", integrator_type="ei", model_type="target_informed_zero_init",
                   time_type="snr", solver_details={"sigma": 1.0}, target_details=BU.make_target_details("two_modes", dim=2),
                   training_details={"train_steps": 3, "train_batch_size": 512, "eval_batch_size": 512}, n_steps=50, device="cuda:0")
for _i in range(3):
    _w.step(_i)
for solver, kw in (("pis_orig", dict(integrator_type="em", time_type="uniform")),
                   ("vp-ref", dict(integrator_type="ei", time_type="snr")),
                   ("dis_orig", dict(integrator_type="em", time_type="uniform")),
                   ("cmcd", dict(integrator_type="em", time_type="uniform", model_type="target_informed_zero_init"))):
    torch.manual_seed(0)
    model = BU.make_model(solver_type=solver, ref_type="default", loss_type="lv", model_type=kw.pop("model_type", "target_informed_zero_init"),
                          solver_details={"sigma": 1.0}, target_details=BU.make_target_details("two_modes", dim=2),
                          training_details={"train_steps": 200, "train_batch_size": 512, "eval_batch_size": 4096},
                          optim_details=None, n_steps=50, device="cuda:0", **kw)
    model.cfg["optim"] = {"_target_": torch.optim.Adam, "lr": 3e-3}
    r0 = model.compute_results().metrics
    t0 = time.time()
    losses = [model.step(i)["train/loss"] for i in range(200)]
    dt = time.time() - t0
    r1 = model.compute_results().metrics
    print(f"{solver}: lv_loss {r0['eval/lv_loss']:.3f} -> {r1['eval/lv_loss']:.3f}; elbo {r0['eval/elbo']:.3f} -> {r1['eval/elbo']:.3f}; "
          f"train loss first/last 20: {sum(losses[:20])/20:.3f} / {sum(losses[-20:])/20:.3f}; {dt/200*1e3:.1f} ms/step", flush=True)
