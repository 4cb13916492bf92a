#!/usr/bin/env python
"""RDS with a fitted full-covariance reference against the fitted diagonal one: EI, ManyModes d = 50 with 16 modes,
K = 200, f16x3 network, production-mode noise, at B = 8192 and 65536.

Both references are fitted by EM (fit_gmm, em_type 'full' / 'diag') to the same exact target samples.  Times are CUDA
events around one simulate() each, after warm-up, alternating the two references; the table reports the median ms per
rollout, particle-steps/s and the ELBO / log Z of each reference.  Writes profiles/<out> (JSON) with the card name and
its power limit."""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from sde_sampler_lrds_b200.benchmark_utils import fit_gmm  # noqa: E402
from tests import cases as T  # noqa: E402
from tests.product_builders import Built  # noqa: E402
from tests.test_full_cov_gpu import built_full  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else torch.cuda.get_device_name(0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--batches", default="8192,65536")
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--samples", type=int, default=16000, help="target samples the references are fitted to")
    ap.add_argument("--out", default="r03_full_cov_bench.json")
    args = ap.parse_args()
    dev = torch.device("cuda:0")
    K, d, M = 200, 50, 16
    base = T.case_ei_many_modes(K=K, B=8, d=d, M=M)
    tgt = base["problem"]["target"]
    g = torch.Generator().manual_seed(0)
    w = tgt["weights"] / tgt["weights"].sum()
    comp = torch.multinomial(w, args.samples, replacement=True, generator=g)
    data = tgt["loc"][comp] + tgt["scale"][comp] * torch.randn(args.samples, d, generator=g)
    wf, mf, cf = fit_gmm(M, data, means_init=tgt["loc"], em_type="full")
    wd, md, vd = fit_gmm(M, data, means_init=tgt["loc"], em_type="diag")
    refs = {"full": {"kind": "gmm_full", "means": mf, "cov": cf, "weights": wf},
            "diag": {"kind": "gmm", "means": md, "variances": vd, "weights": wd}}
    rows = []
    for B in (int(b) for b in args.batches.split(",")):
        builts = {}
        for name, ref in refs.items():
            case = dict(base, B=B, problem=dict(base["problem"], ref=ref))
            builts[name] = built_full(case, dev, "f16x3") if name == "full" else Built(case, dev, "f16x3")
        x0 = torch.randn(B, d, generator=torch.Generator().manual_seed(1)).to(dev)
        times = {n: [] for n in builts}
        res = {}
        for n, b in builts.items():  # warm-up: plan packing, module load
            for i in range(2):
                b.simulate(x0, None, seed=i)
        torch.cuda.synchronize()
        for r in range(args.reps):
            for n, b in builts.items():
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                _, rnd, _ = b.simulate(x0, None, seed=100 + r)
                e1.record()
                e1.synchronize()
                times[n].append(e0.elapsed_time(e1))
                if r == 0:
                    lw = -rnd.double().reshape(-1)
                    res[n] = {"elbo": lw.mean().item(),
                              "log_norm_const_is": (torch.logsumexp(lw, 0) - torch.log(torch.tensor(float(B)))).item()}
        for n in builts:
            ms = statistics.median(times[n])
            rows.append({"ref": n, "B": B, "K": K, "ms_per_rollout": ms, "spread_ms": [min(times[n]), max(times[n])],
                         "particle_steps_per_s": B * K / (ms * 1e-3), **res[n]})
            print(json.dumps(rows[-1]))
    out = {"card": card(), "workload": "RDS EI ManyModes d=50 M=16 K=200, f16x3, production-mode noise, fitted refs",
           "timing": "CUDA events around simulate(), median of %d alternating reps after 2 warm-ups" % args.reps,
           "rows": rows}
    with open(os.path.join(ROOT, "profiles", args.out), "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({"card": out["card"]}))


if __name__ == "__main__":
    main()
