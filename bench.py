#!/usr/bin/env python
"""Benchmark of the fused trajectory rollout (BASELINE.json metric: particle-steps/s).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision f16x3|tf32x3|fp32|tf32|bf16]
                    [--dump-outputs DIR]

The headline number is measured in the fp32-grade mode f16x3 (drift network, mixture logits AND mixture-score
contractions on tcgen05 tensor cores with the 3-pass fp16 (hi, lo) split of power-of-two scaled operands; parity-tested to
the north-star tolerance like tf32x3 and the fp32 SIMT anchor).  --fast-mode additionally times the reduced-precision bf16
kernel and reports it separately with its tolerance.

A "step" is one complete rollout of the workload's particle batch through all grid times (the quantity the
reference times as eval/sample_time, solver/oc.py:148-158) followed by the estimator reduction; under
torchrun every rank integrates its own shard of particles (weak scaling: 65536 per GPU, RNG counter = global
particle index) and the only exchange is the all_gather of 8 doubles per rank, merged on the device.  `value` times the
step on device-resident inputs; `e2e` times it through sde_sampler_lrds_b200.streaming.HostRolloutStream with pinned HOST
buffers in and out (the copies of neighbouring steps overlap the kernel); `workloads` times the other BASELINE.json shapes
on the device in the same run (single-GPU runs); `--impl reference` runs the CPU port of the reference's loop on the same
config, exactly --warmup + --steps rollouts of a 4096-particle sample.

Workload = BASELINE.json configs[1]: ManyModes d=50 (16 modes), RDS vp-ref (VP beta 0.1..20), diagonal-GMM
reference, target_informed (ScoreCtrl) drift, EI integrator, 200 steps, batch 65536, synthetic weights.
Prints ONE JSON line (see DESIGN.md "Measurement" for every field).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOAD = "many_modes_d50_M16_rds_gmmref_scorectrl_ei_K200_B65536"
B_PER_GPU, K_STEPS, DIM, MODES = 65536, 200, 50, 16
# algorithmic tensor FLOPs per particle-step (SURVEY.md 8d): MLP 256 d + 16384, two diag-GMM scores 8 M d each
FLOPS_PER_PARTICLE_STEP = (256 * DIM + 16384) + 2 * 8 * MODES * DIM
METRIC, UNIT = "particle_steps_per_sec", "particle-steps/s"
CPU_SAMPLE_B = 16384
REFERENCE_SAMPLE_B = 4096  # --impl reference: particles per timed step (CPU throughput is flat in B beyond ~4k)
# ALGORITHMIC budget of the work that is not a GEMM at fp32 parity, in FMA-class lane-operations per particle-step
# (DESIGN.md 5; a constant of the algorithm, NOT an executed-instruction count): erf-GELU 192 x 9 = 1730, 50 Gaussian
# draws (13 Philox4x32-10 blocks + Box-Muller) 560, integrator update / costs 500; a mixture whose modes do NOT share
# their variances adds its exact quadratic forms (2 FMA per mode and dim: 2 x 16 x 52 x 2 = 3328).  The bench workload's
# mixtures share their variances (logits on tcgen05), so the first figure is the one that applies; both are reported.
SIMT_LANE_OPS = {"shared_variance_mixtures": 1730 + 560 + 500, "general_diagonal_mixtures": 1730 + 560 + 500 + 3328}
FFMA_LANE_INSTR_PER_CLK_SM = 115.0  # measured on B200 (profiles/r01_ubench.txt); 128 nominal
# dram__bytes_read.sum + dram__bytes_write.sum of one launch of the benchmark kernel (profiles/r02_mix_summary.md)
DRAM_BYTES_PER_LAUNCH = {"f16x3": 17_147_136 + 768}
# the other BASELINE.json shapes, timed on the device in the same run (parity cases, not the headline): name in
# tools/shape_bench.py -> algorithmic tensor FLOPs per particle-step (BASELINE.md 3)
WORKLOADS = {
    "cfg1_two_modes_d2_em_K100_B2048": ("cfg1 two_modes", 16896 + 32 + 16),
    "cfg3_phi4_d100_pis_K256_B131072": ("cfg3 phi4 d=100 PIS", 41984),
    "cfg3_phi4_d100_dds_K256_B131072": ("cfg3 phi4 d=100 DDS", 41984),
    "cfg4_logreg_sonar_cmcd_K100_B262144": ("cfg4 logreg sonar", 71800),
    "cfg4_logreg_iono_cmcd_K100_B262144": ("cfg4 logreg iono", 62000),
    "cfg2_compute_eubo_K200_B65536": ("eubo cfg2", (256 * DIM + 16384) + 2 * 8 * MODES * DIM),
}
FAST_MODE_TOLERANCE = "log Z within 5e-2 abs, 99% of log-weights within 1e-2 rel (tests/test_rollout_parity_gpu.py)"


def measured_peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            p = json.load(f)
        return p, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock and throttle reasons through NVML while the timed region runs."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.max_mhz, self._stop_evt = index, [], set(), None, threading.Event()
        self.ready, self.recording = threading.Event(), False  # NVML init happens BEFORE the timed region

    def run(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self.index)
            self.max_mhz = nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM)
            names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                     nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                     nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
            nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)  # first calls are slow: make them before the timed region
            nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
            self.ready.set()
            while not self._stop_evt.is_set():
                # polled continuously from before the warm-up (a first NVML query inside the timed region stalls the
                # launch path for tens of ms); only samples taken while `recording` are reported
                mhz = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                if self.recording:
                    self.samples.append(mhz)
                    for bit, name in names.items():
                        if r & bit:
                            self.reasons.add(name)
                time.sleep(0.05)
        except Exception as e:  # pragma: no cover
            self.reasons.add(f"nvml_unavailable:{type(e).__name__}")
            self.ready.set()

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons)}


def build_case(B):
    from tests.cases import case_ei_many_modes
    return case_ei_many_modes(K=K_STEPS, B=B, d=DIM, M=MODES)


def cpu_port_throughput(B_sample, threads, steps=1, warmup=0):
    """Times the oracle (torch-on-CPU restatement of the reference's loop, pinned to the reference by tests/golden)
    on a bounded sample of the workload: B_sample particles through all K_STEPS grid times."""
    import torch
    from oracle import rollout_oracle as O
    torch.set_num_threads(threads)
    case = build_case(B_sample)
    g = torch.Generator().manual_seed(0)
    x0 = torch.randn(B_sample, DIM, generator=g)
    noise = torch.randn(K_STEPS, B_sample, DIM, generator=g)
    times = []
    for i in range(warmup + steps):
        t0 = time.perf_counter()
        O.rollout(case["problem"], x0, noise)
        if i >= warmup:
            times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    return B_sample * K_STEPS / dt, dt


def bench_config(world, precision):
    """The workload description both arms print (the reference arm runs the same workload on the host cores)."""
    return {"workload": WORKLOAD, "particles_per_gpu": B_PER_GPU, "grid_steps": K_STEPS, "dim": DIM, "modes": MODES,
            "precision": precision, "noise": "in-kernel Philox4x32-10", "l2": "flushed between timed iterations",
            "parallelism": f"particles sharded over {world} GPU(s), no data-path collective"}


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path.  The reference is Python/torch and its
    source tree does not travel to the GPU box, so the arm runs the oracle port (oracle/rollout_oracle.py, pinned
    to the reference by tests/golden) with all host threads.  It does exactly --warmup untimed and --steps timed steps;
    a step is one rollout of a bounded sample (REFERENCE_SAMPLE_B particles through all K_STEPS grid times) of the
    workload, so that the whole run ends within a few minutes."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    threads = os.cpu_count() or 1
    value, dt = cpu_port_throughput(REFERENCE_SAMPLE_B, threads, steps=max(1, args.steps), warmup=max(0, args.warmup))
    sample = (f"each step = B={REFERENCE_SAMPLE_B} of {B_PER_GPU} particles through all K={K_STEPS} grid times, d={DIM}; "
              f"torch {torch.__version__} CPU threads={threads}")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": max(1, args.steps), "warmup": max(0, args.warmup), "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": bench_config(args.gpus, args.precision),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def run_ours(args):
    import torch
    import torch.distributed as dist
    from sde_sampler_lrds_b200 import _native as N
    from sde_sampler_lrds_b200.estimators import gather_and_merge, metrics_from_partials
    from sde_sampler_lrds_b200.streaming import HostRolloutStream
    from tests.product_builders import Built

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # The contract is ONE JSON line on stdout: libraries that print there (NCCL's version banner at communicator
    # creation) are sent to stderr; the line is written to the saved descriptor at the end.
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the rollout has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    group = dist.group.WORLD if world > 1 else None

    B = B_PER_GPU
    case = build_case(B)
    built = Built(case, dev, args.precision)
    g = torch.Generator().manual_seed(1 + rank)
    x0_host = torch.randn(B, DIM, generator=g).pin_memory()
    x0 = x0_host.to(dev)
    offset = rank * B
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2
    blocks = N.lib().lrds_estimator_blocks(B)
    scratch = torch.empty(8 * (blocks + 1), device=dev, dtype=torch.float64)

    def step(seed):
        """One step on device-resident inputs: the fused rollout, the estimator partials and - the one exchange of the
        path - the all_gather of 8 doubles per rank with its merge, everything on the device (no host round trip)."""
        x, rnd, _ = built.simulate(x0, None, seed=seed, particle_offset=offset)
        r = rnd.reshape(-1)
        out = torch.empty(8, device=dev, dtype=torch.float64)
        N.check(N.lib().lrds_estimator_partials(N.ptr(r), r.numel(), N.ptr(out), N.ptr(scratch), N.stream_ptr(dev)))
        return x, rnd, (gather_and_merge(out, group, on_device=True) if group is not None else out)

    def barrier():
        if group is not None:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def max_over_ranks(v):
        t = torch.tensor([v], device=dev, dtype=torch.float64)
        if group is not None:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sampler = ClockSampler(local)
    sampler.start()
    sampler.ready.wait(timeout=10)
    prev = None
    for w in range(args.warmup):
        # two generations of outputs stay alive, as in the timed loop: the caching allocator then owns every buffer
        # the timed iterations need (a cudaMalloc inside the timed region would stall the launch path for milliseconds)
        cur = step(1000 + w)
        prev = cur
    barrier()
    del prev, cur

    # ---- device-resident timing (value) + the dominant kernel alone (roofline) -----------------------------------
    sampler.recording = True
    launches0 = N.launch_count()
    ev = [(torch.cuda.Event(True), torch.cuda.Event(True), torch.cuda.Event(True)) for _ in range(args.steps)]
    last = None
    for i in range(args.steps):
        flush.fill_(i & 0xFF)  # evict L2 between timed iterations (not timed)
        a, b, c = ev[i]
        a.record()
        x, rnd, _ = built.simulate(x0, None, seed=2000 + i, particle_offset=offset)
        b.record()
        r = rnd.reshape(-1)
        out = torch.empty(8, device=dev, dtype=torch.float64)
        N.check(N.lib().lrds_estimator_partials(N.ptr(r), r.numel(), N.ptr(out), N.ptr(scratch), N.stream_ptr(dev)))
        last = gather_and_merge(out, group, on_device=True) if group is not None else out
        c.record()
    barrier()
    launches = N.launch_count() - launches0
    sampler.recording = False
    step_ms = sum(a.elapsed_time(c) for a, _, c in ev)
    kern_ms = sum(a.elapsed_time(b) for a, b, _ in ev) / args.steps
    kern_ms_each = [round(a.elapsed_time(b), 3) for a, b, _ in ev]
    ms_per_step = max_over_ranks(step_ms) / args.steps
    value = world * B * K_STEPS / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:
        # what a caller of the timed path receives from its last step: x_T [B, 50] and rnd [B, 1] in float32 (13.4 MB),
        # the 8 merged estimator partials in float64
        dump_outputs(args.dump_outputs, {"x_T": x, "rnd": rnd, "estimator_partials": last})

    # ---- reduced-precision fast mode, reported separately ------------------------------------------------------
    fast = None
    if args.fast_mode:
        from sde_sampler_lrds_b200.estimators import estimator_partials
        built_fast = Built(case, dev, "bf16")
        for w in range(3):
            built_fast.simulate(x0, None, seed=4000 + w, particle_offset=offset)
        barrier()
        fev = [(torch.cuda.Event(True), torch.cuda.Event(True)) for _ in range(3)]
        for i, (fa, fb) in enumerate(fev):
            flush.fill_(i & 0xFF)
            fa.record()
            _, rnd_f, _ = built_fast.simulate(x0, None, seed=2000 + i, particle_offset=offset)
            fb.record()
        barrier()
        fms = max_over_ranks(sum(fa.elapsed_time(fb) for fa, fb in fev) / len(fev))
        mf = metrics_from_partials(estimator_partials(rnd_f))
        fast = {"precision": "bf16", "value": world * B * K_STEPS / (fms * 1e-3), "unit": UNIT,
                "kernel_ms": fms, "tolerance": FAST_MODE_TOLERANCE,
                "check": {"log_norm_const_is": mf["log_norm_const_is"], "elbo": mf["elbo"]}}

    # ---- end to end through the public host-buffer API (sde_sampler_lrds_b200.streaming.HostRolloutStream) -------
    # Every step: H2D of the step's x0 from pinned host memory, the rollout + estimator (+ all_gather / merge on the
    # device), D2H of x_T, rnd and the 8 merged doubles into pinned host memory.  The copies of neighbouring steps overlap
    # the kernel (three streams, two slots); the host blocks only on the results of the step it reads.
    pipe = HostRolloutStream(lambda xd, seed, off: built.simulate(xd, None, seed=seed, particle_offset=off)[:2],
                             B, DIM, dev, group=group, depth=2)

    def e2e_run(n, seed0):
        res = None
        for i in range(n):
            t = pipe.submit(x0_host, seed0 + i, offset)
            if i >= 1:
                res = pipe.wait(t - 1)
        return pipe.wait(n - 1) if n else res

    e2e_run(3, 2900)  # untimed: first touch of the pinned buffers, allocator entries of the staging tensors
    barrier()
    t0 = time.perf_counter()
    _, _, part_host = e2e_run(args.steps, 3000)
    barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_value = world * B * K_STEPS * args.steps / e2e_s
    e2e_check = metrics_from_partials(part_host.clone())
    # the phases of one step measured alone (CUDA events, nothing overlapped): what the pipeline has to hide
    pe = [torch.cuda.Event(True) for _ in range(4)]
    xd = torch.empty(B, DIM, device=dev)
    xh, rh = torch.empty(B, DIM).pin_memory(), torch.empty(B, 1).pin_memory()
    barrier()
    pe[0].record()
    xd.copy_(x0_host, non_blocking=True)
    pe[1].record()
    xo, ro, _ = step(3900)
    pe[2].record()
    xh.copy_(xo, non_blocking=True)
    rh.copy_(ro, non_blocking=True)
    pe[3].record()
    barrier()
    phases = {"h2d_ms": pe[0].elapsed_time(pe[1]), "rollout_estimator_collective_ms": pe[1].elapsed_time(pe[2]),
              "d2h_ms": pe[2].elapsed_time(pe[3]), "pipelined_ms_per_step": e2e_s * 1e3 / args.steps}

    # ---- the other BASELINE shapes on the device (rank 0 of a single-GPU run only) ------------------------------
    workloads = None
    if world == 1 and not args.no_workloads:
        workloads = other_workloads(dev, args.precision, flush)
    clocks = sampler.stop()

    if rank != 0:
        if group is not None:
            dist.destroy_process_group()
        return

    peaks, how = measured_peaks()
    achieved = FLOPS_PER_PARTICLE_STEP * B * K_STEPS / (kern_ms * 1e-3) / 1e12
    peak = float(peaks["bf16_tflops"])
    m = metrics_from_partials(last.cpu())
    threads = os.cpu_count() or 1
    cpu_value = cpu_dt = None
    if world == 1 and not args.no_cpu_baseline:
        cpu_value, cpu_dt = cpu_port_throughput(CPU_SAMPLE_B, threads, steps=2, warmup=1)
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    mhz = clocks.get("sm_mhz") or clocks.get("sm_max_mhz") or 1965
    per_gpu = B * K_STEPS / (kern_ms * 1e-3)
    simt = {}
    for name, ops in SIMT_LANE_OPS.items():
        roof = FFMA_LANE_INSTR_PER_CLK_SM * sms * mhz * 1e6 / ops
        simt[name] = {"lane_ops_per_particle_step": ops, "peak": roof, "achieved": per_gpu, "unit": UNIT, "frac": per_gpu / roof}
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": bench_config(world, args.precision),
        "clocks": clocks,
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": pipe.h2d_bytes, "d2h_bytes_per_step": pipe.d2h_bytes,
                "api": "sde_sampler_lrds_b200.streaming.HostRolloutStream (pinned host buffers in and out, two slots)",
                "phases": phases,
                "check": {"log_norm_const_is": e2e_check["log_norm_const_is"], "elbo": e2e_check["elbo"]}},
        "gpu_launches": int(launches),
        "roofline": {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                     "traffic": DRAM_BYTES_PER_LAUNCH.get(args.precision), "kernel_ms": kern_ms, "kernel_ms_each": kern_ms_each,
                     "peak_source": how + ", dense bf16 burst", "flops_per_particle_step": FLOPS_PER_PARTICLE_STEP,
                     "passes": "f16x3 issues 3 MMAs per algorithmic FLOP (fp32-grade products): tensor-pipe time = 3 x frac",
                     # the work that is not a GEMM at fp32 parity, against the measured FFMA rate: an ALGORITHMIC budget
                     "simt": {"ffma_lane_instr_per_clk_sm": FFMA_LANE_INSTR_PER_CLK_SM, "sm_mhz": mhz, "sms": sms,
                              "applies": "shared_variance_mixtures", **simt}},
        "check": {"log_norm_const_is": m["log_norm_const_is"], "elbo": m["elbo"], "ess": m["effective_sample_size"]},
    }
    if workloads is not None:
        line["workloads"] = workloads
    if fast is not None:
        line["fast_mode"] = fast
    if cpu_value is not None:
        line["cpu_baseline"] = {"value": cpu_value, "unit": UNIT, "cores": threads, "kind": "port",
                                "sample": f"B={CPU_SAMPLE_B} of {B} particles, all K={K_STEPS} steps, d={DIM}; "
                                          f"{cpu_dt:.1f} s per rollout, torch {torch.__version__} CPU threads={threads}"}
    sys.stdout.flush()
    os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if group is not None:
        dist.destroy_process_group()


def dump_outputs(out_dir, arrays):
    """Writes each tensor as <out_dir>/<name>.npy in the dtype it was computed in, so that two builds of the project run
    with the same arguments (hence the same seeded inputs) can be compared output for output."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), t.detach().cpu().numpy())


def other_workloads(dev, precision, flush):
    """Device-resident kernel time of the other BASELINE.json shapes (production mode, in-kernel noise): 2 warm-ups,
    3 timed launches each with the L2 flushed in between; tensor-roof fraction from BASELINE.md's FLOP counts."""
    import torch
    from tests.product_builders import Built
    from tools.shape_bench import SHAPES
    peaks, _ = measured_peaks()
    out = {}
    for key, (needle, flops) in WORKLOADS.items():
        name = next(n for n in SHAPES if n.startswith(needle) and ("DDS" in n) == ("dds" in key))
        try:
            case = SHAPES[name]()
            p = case["problem"]
            Bw = case["B"]
            d = p["target"]["loc"].shape[1] if p["target"]["kind"] == "gmm" else p["target"]["dim"]
            K = len(p["ts"]) - 1
            gen = torch.Generator().manual_seed(1)
            x0 = (torch.zeros(Bw, d) if case["prior"][0] == "delta" else torch.randn(Bw, d, generator=gen)).to(dev)
            if case.get("eubo") and p["target"]["kind"] == "gmm":  # compute_eubo starts at TARGET samples (hacking.py:14-19)
                t = p["target"]
                idx = torch.multinomial(t["weights"] / t["weights"].sum(), Bw, replacement=True, generator=gen)
                x0 = (t["loc"][idx] + t["scale"][idx] * torch.randn(Bw, d, generator=gen)).to(dev)
            built = Built(case, dev, precision)
            run = (lambda seed: built.compute_eubo(x0.clone(), None, seed=seed)) if case.get("eubo") else \
                (lambda seed: built.simulate(x0, None, seed=seed))
            for w in range(2):
                run(w)
            torch.cuda.synchronize(dev)
            evs = [(torch.cuda.Event(True), torch.cuda.Event(True)) for _ in range(3)]
            for i, (a, b) in enumerate(evs):
                flush.fill_(i)
                a.record()
                run(10 + i)
                b.record()
            torch.cuda.synchronize(dev)
            ms = sum(a.elapsed_time(b) for a, b in evs) / len(evs)
            ps = Bw * K / (ms * 1e-3)
            out[key] = {"B": Bw, "K": K, "d": d, "ms": ms, "particle_steps_per_s": ps,
                        "tensor_frac": flops * ps / 1e12 / float(peaks["bf16_tflops"]), "flops_per_particle_step": flops}
            del built, x0
        except Exception as e:  # a shape that fails must not take the headline down with it
            out[key] = {"error": f"{type(e).__name__}: {e}"[:200]}
    try:  # one LV training objective + gradient of the benchmark problem (rollout + lrds_mlp_grad + lrds_score_cot_sums)
        from tests import cases as T
        Bt, Kt = 65536, 200
        built = Built(T.case_ei_many_modes(K=Kt, B=Bt), dev, precision)
        x0 = torch.randn(Bt, 50, generator=torch.Generator().manual_seed(1)).to(dev)
        params = list(built.ctrl.parameters())

        def train_step(seed):
            for q in params:
                q.grad = None
            loss, _ = built.train_loss(x0, None, seed=seed)
            loss.backward()
        for w in range(2):
            train_step(w)
        torch.cuda.synchronize(dev)
        evs = [(torch.cuda.Event(True), torch.cuda.Event(True)) for _ in range(3)]
        for i, (a, b) in enumerate(evs):
            flush.fill_(i)
            a.record()
            train_step(10 + i)
            b.record()
        torch.cuda.synchronize(dev)
        ms = sum(a.elapsed_time(b) for a, b in evs) / len(evs)
        out["cfg2_lv_training_step"] = {"B": Bt, "K": Kt, "d": 50, "ms": ms, "particle_steps_per_s": Bt * Kt / (ms * 1e-3),
                                        "what": "loss(ts, x, ...) + loss.backward(): rollout, lrds_mlp_grad, lrds_score_cot_sums"}
        del built, x0
    except Exception as e:
        out["cfg2_lv_training_step"] = {"error": f"{type(e).__name__}: {e}"[:200]}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default="f16x3", choices=["fp32", "tf32x3", "f16x3", "tf32", "bf16"])
    ap.add_argument("--fast-mode", action="store_true", help="also time the reduced-precision bf16 kernel")
    ap.add_argument("--no-fast-mode", action="store_true", help=argparse.SUPPRESS)  # accepted for older command lines
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-workloads", action="store_true", help="skip the other BASELINE shapes (single-GPU runs time them too)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's x_T, rnd and estimator partials (rank 0) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the outputs of --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
