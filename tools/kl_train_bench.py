#!/usr/bin/env python
"""Time of one pathwise ('kl') training step - loss(ts, x, ...) and loss.backward(): fused rollout with trajectory,
reverse-time adjoint kernel (lrds_adjoint), parameter pass - next to the 'lv' step of the same model, the adjoint kernel
alone, and the CPU oracle's autograd through the K-step loop (the reference's way of computing the same gradient).
Workload: ManyModes d = 50, M = 16, RDS-EI with the 16-component GMM reference, ClippedCtrl, K = 200.

    python tools/kl_train_bench.py [--json out.json] [--batches 512,8192,65536] [--cpu-batch 512]

GPU times are CUDA events around warmed-up steps (best of three); the card's name and power limit are read in the same
run and stored with the rows."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

from tests import cases as T  # noqa: E402
from tests import kl_oracle as KO  # noqa: E402  (CPU baseline leg only)
from tests.product_builders import Built  # noqa: E402


def problem(K, B):
    case = T.case_ei_many_modes(K=K, B=B)
    case["problem"] = dict(case["problem"], ctrl=T.ctrl(50, "clipped", seed=12, out_gain=1.0))
    return case


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clock = (v.strip() for v in out[0].split(","))
    return {"gpu": name, "power_limit": power, "max_sm_clock": clock}


def best_ms(fn, reps=3):
    ev = [(torch.cuda.Event(True), torch.cuda.Event(True)) for _ in range(reps)]
    for i, (a, b) in enumerate(ev):
        a.record()
        fn(10 + i)
        b.record()
    torch.cuda.synchronize()
    return min(a.elapsed_time(b) for a, b in ev)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--json", default=None)
    ap.add_argument("--batches", default="512,8192,65536")
    ap.add_argument("--cpu-batch", type=int, default=512)
    ap.add_argument("--K", type=int, default=200)
    args = ap.parse_args()
    from sde_sampler_lrds_b200 import pack
    from sde_sampler_lrds_b200 import train as TR
    dev = torch.device("cuda:0")
    meta = card()
    shape = f"many_modes d=50 M=16 RDS-EI GMM ref ClippedCtrl K={args.K} f16x3"
    rows = []
    for B in [int(b) for b in args.batches.split(",")]:
        case = problem(args.K, B)
        x0 = torch.randn(B, 50, generator=torch.Generator().manual_seed(1)).to(dev)
        built = Built(case, dev, "f16x3")
        params = list(built.ctrl.parameters())
        row = {"shape": shape, "B": B, **meta}
        for method in ("kl", "lv"):
            built.loss.method = method

            def step(seed):
                with torch.no_grad():  # an optimiser step changes the weights: the cached plan refreshes its weight images
                    params[0].add_(0.0)
                for p in params:
                    p.grad = None
                loss, _ = built.train_loss(x0, None, seed=seed)
                loss.backward()
            for w in range(2):
                step(w)
            torch.cuda.synchronize()
            row[f"{method}_step_ms"] = best_ms(step)
        (plan,) = [h[0] for h in built.loss._plans.values()]
        _, _, xs = pack.run_rollout(plan, x0, None, 3, 0, True)
        w = torch.full((B,), 1.0 / B, device=dev)
        TR.adjoint(plan, xs, w, 3)
        torch.cuda.synchronize()
        row["adjoint_kernel_ms"] = best_ms(lambda s: TR.adjoint(plan, xs, w, 3))
        row["kl_particle_steps_per_s"] = B * args.K / (row["kl_step_ms"] * 1e-3)
        rows.append(row)
        print(json.dumps(row), flush=True)
    # CPU: the oracle's autograd through the loop (what the reference's training step does), all host threads
    B = args.cpu_batch
    case = problem(args.K, B)
    x0, noise = T.initial_state(case), T.noise_for(case)
    KO.kl_loss_and_grads(dict(case["problem"], ts=case["problem"]["ts"][:5]), x0, noise[:4])  # warm-up
    t0 = time.time()
    KO.kl_loss_and_grads(case["problem"], x0, noise)
    sec = time.time() - t0
    row = {"shape": shape.replace(" f16x3", "") + " fp32", "B": B, "cpu_kl_step_ms": sec * 1e3,
           "cpu_threads": torch.get_num_threads(), "kind": "oracle (CPU autograd through the K steps)"}
    rows.append(row)
    print(json.dumps(row), flush=True)
    if args.json:
        with open(args.json, "w") as f:
            json.dump(rows, f, indent=1)


if __name__ == "__main__":
    main()
