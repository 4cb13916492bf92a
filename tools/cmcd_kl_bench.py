#!/usr/bin/env python
"""Time of one pathwise CMCD ('kl') training step - loss(ts, x, ...) and loss.backward(): fused rollout with trajectory,
reverse-time adjoint kernel (lrds_adjoint_cmcd), parameter pass over the K + 1 points - next to the 'lv' step of the same
model, the adjoint alone for the f16x3 plan and for the fp32 plan of the same shape, and the CPU oracle's autograd
through the K-step loop.  Workload: ManyModes d = 50, M = 16, isotropic prior N(0, 5^2), ClippedCtrl, K = 200.

    python tools/cmcd_kl_bench.py [--json out.json] [--batches 512,8192,65536] [--cpu-batch 512]

GPU times are CUDA events around warmed-up calls (best of three); the adjoint kernel's name is read once from
torch.profiler in a separate pass; the card's name and power limit are read in the same run and stored with the rows."""
import argparse
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from tests import cases as T  # noqa: E402
from tests import cmcd_kl_oracle as CKO  # noqa: E402  (CPU baseline leg only)
from tests.product_builders import Built  # noqa: E402
from tools.kl_train_bench import best_ms, card  # noqa: E402

D, M = 50, 16


def problem(K, B):
    return {"problem": {"method": "cmcd", "sde": None, "diff": 1.0, "T": 1.0, "clip_score": 1e5,
                        "ts": T.uniform_ts(1.0, K), "target": T.many_modes(M, D, var=0.5),
                        "ctrl": T.ctrl(D, "clipped", seed=12, out_gain=1.0),
                        "prior": {"loc": torch.zeros(D), "scale": 5.0 * torch.ones(D), "isotropic": True}},
            "B": B, "seed": 140, "prior": ("iso", 0.0, 5.0)}


def adjoint_setup(case, precision, x0, dev):
    """(plan, trajectory, row weights) of one rollout of the training plan at ``precision``."""
    from sde_sampler_lrds_b200 import pack
    built = Built(case, dev, precision)
    built.loss.method = "kl"
    loss, _ = built.train_loss(x0, None, seed=2)
    loss.backward()
    (plan,) = [h[0] for h in built.loss._plans.values()]
    _, _, xs = pack.run_rollout(plan, x0, None, 3, 0, True)
    w = torch.full((x0.shape[0],), 1.0 / x0.shape[0], device=dev)
    return built, plan, xs, w


def kernel_name(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = [e.key for e in prof.key_averages() if "adjoint" in e.key]
    return names[0] if names else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--json", default=None)
    ap.add_argument("--batches", default="512,8192,65536")
    ap.add_argument("--cpu-batch", type=int, default=512)
    ap.add_argument("--K", type=int, default=200)
    args = ap.parse_args()
    from sde_sampler_lrds_b200 import train as TR
    dev = torch.device("cuda:0")
    meta = card()
    shape = f"many_modes d={D} M={M} CMCD N(0,5^2) prior ClippedCtrl K={args.K}"
    rows = []
    names = {}
    for B in [int(b) for b in args.batches.split(",")]:
        case = problem(args.K, B)
        x0 = (5.0 * torch.randn(B, D, generator=torch.Generator().manual_seed(1))).to(dev)
        row = {"shape": shape + " f16x3", "B": B, **meta}
        built, plan, xs, w = adjoint_setup(case, "f16x3", x0, dev)
        params = list(built.ctrl.parameters())
        for method in ("kl", "lv"):
            built.loss.method = method

            def step(seed):
                with torch.no_grad():  # an optimiser step changes the weights: the cached plan refreshes its weight images
                    params[0].add_(0.0)
                for p in params:
                    p.grad = None
                loss, _ = built.train_loss(x0, None, seed=seed)
                loss.backward()
            for i in range(2):
                step(i)
            torch.cuda.synchronize()
            row[f"{method}_step_ms"] = best_ms(step)
        TR.adjoint_cmcd(plan, xs, w, 3)
        torch.cuda.synchronize()
        row["adjoint_cmcd_ms"] = best_ms(lambda s: TR.adjoint_cmcd(plan, xs, w, 3))
        _, plan32, xs32, w32 = adjoint_setup(case, "fp32", x0, dev)
        TR.adjoint_cmcd(plan32, xs32, w32, 3)
        torch.cuda.synchronize()
        row["adjoint_cmcd_fp32_spec_ms"] = best_ms(lambda s: TR.adjoint_cmcd(plan32, xs32, w32, 3))
        row["kl_particle_steps_per_s"] = B * args.K / (row["kl_step_ms"] * 1e-3)
        names[B] = (plan, xs, w, plan32, xs32, w32)
        rows.append(row)
        print(json.dumps(row), flush=True)
    # the kernels behind the two adjoint timings, read once per batch in a pass of its own (the profiler slows the host)
    for row in rows:
        plan, xs, w, plan32, xs32, w32 = names[row["B"]]
        row["adjoint_kernel"] = kernel_name(lambda: TR.adjoint_cmcd(plan, xs, w, 3))
        row["adjoint_kernel_fp32_spec"] = kernel_name(lambda: TR.adjoint_cmcd(plan32, xs32, w32, 3))
        print(json.dumps({"B": row["B"], "adjoint_kernel": row["adjoint_kernel"],
                          "adjoint_kernel_fp32_spec": row["adjoint_kernel_fp32_spec"]}), flush=True)
    # CPU: the oracle's autograd through the loop (what the reference's training step does), all host threads
    B = args.cpu_batch
    case = problem(args.K, B)
    x0, noise = T.initial_state(case), T.noise_for(case)
    CKO.kl_loss_and_grads(dict(case["problem"], ts=case["problem"]["ts"][:5]), x0, noise[:4])  # warm-up
    t0 = time.time()
    CKO.kl_loss_and_grads(case["problem"], x0, noise)
    sec = time.time() - t0
    row = {"shape": shape + " fp32", "B": B, "cpu_kl_step_ms": sec * 1e3, "cpu_threads": torch.get_num_threads(),
           "kind": "oracle (CPU autograd through the K steps)"}
    rows.append(row)
    print(json.dumps(row), flush=True)
    if args.json:
        with open(args.json, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
