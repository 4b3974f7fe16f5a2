#!/usr/bin/env python
"""bench.py -- the headline benchmark of the hot path (BASELINE.json):

    waveform windows/sec, MyCNN5 architecture at [4096, 3, 75000] bf16 per GPU
    (configs[1]; weak scaling: every rank scores its own 4096-window shard), independent
    windows (the semantics of bin/predictStream.py's per-row loop), synthetic N(0,1) data,
    seeded random-init weights (no trained weights exist for this shape).

    python bench.py --gpus N --steps K --warmup W          # our arm (one rank per GPU)
    python bench.py --impl reference ...                   # the reference's CPU path, same JSON
    python bench.py ... --dump-outputs DIR                 # also save the last timed step's logits as DIR/logits.npy

A "step" = one pass of the hot path over one batch.  `value` is measured with the inputs
resident in HBM; `e2e` goes through the reference-facing predict() call with HOST (pinned)
tensors, host<->device copies inside the timed region.  One JSON line on stdout (rank 0).

Blocks of the line beyond the base contract:
  roofline      dominant kernel: algorithmic bytes / its CUDA-event duration vs the measured HBM peak
  parity        in-run check of the benchmarked tensor: >= 256 of its windows through the CPU oracle,
                per-element relative error of the logits the timed steps produced (tolerance 1e-4)
  sustained     >= 3 s of back-to-back steps with NVML clock / power samples and its own windows/s
  e2e.pcie      a plain pinned cudaMemcpyAsync H2D peak measured in the same run + the fraction achieved
  cpu_baseline  the reference's CPU path on this box's host cores (persistent single-thread workers,
                pool sized from sched_getaffinity and the cgroup quota, calibrated worker count)
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

KIND, C, W, B_PER_GPU = "mycnn5", 3, 75000, 4096
METRIC = "waveform windows/sec (MyCNN5, W=75000)"
UNIT = "windows/s"
PARITY_TOL = 1e-4            # north_star: 1e-4 relative on the logits


def workload(B, dtype="bf16"):
    """Identical for both arms (the driver compares the two `config` objects)."""
    return {"workload": f"MyCNN5-arch forward, [{B},{C},{W}] {dtype} per GPU, mode=independent",
            "arch": KIND, "batch_per_gpu": B, "channels": C, "window": W, "mode": "independent",
            "values": "N(0,1) seed 1234+rank", "weights": "default init, seed 0",
            "l2": "inputs (1.84 GB per GPU) are larger than the 126 MB L2; no flush needed"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------
class ClockSampler:
    """SM clock + throttle reasons sampled DURING the timed region (B200_PROFILING.md's clocks
    line), through NVML in a background thread: the timed region is only tens of milliseconds,
    too short for an `nvidia-smi -lms` child process to produce a sample."""

    def __init__(self, index):
        self.index, self.rows, self.run, self.thread, self.h = index, [], False, None, None
        try:
            import pynvml
            self.nv = pynvml
            pynvml.nvmlInit()
            self.h = pynvml.nvmlDeviceGetHandleByIndex(self._physical_index(index))
            self.max_sm = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.h = None

    @staticmethod
    def _physical_index(i):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            try:
                return int(vis.split(",")[i])
            except Exception:
                return i
        return i

    def _loop(self):
        nv = self.nv
        while self.run:
            try:
                self.rows.append((time.perf_counter(), nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM),
                                  nv.nvmlDeviceGetCurrentClocksEventReasons(self.h),
                                  nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0))
            except Exception:
                pass
            time.sleep(0.001)

    def start(self):
        if self.h is None:
            return
        self.run = True
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def stop(self):
        if self.h is None:
            return
        self.run = False
        self.thread.join(timeout=2)

    def summary(self, t_begin, t_end, fallback_all=True):
        if self.h is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml unavailable"]}
        nv = self.nv
        rows = [r for r in self.rows if t_begin <= r[0] <= t_end]
        where = "timed region"
        if len(rows) < 3 and fallback_all:   # region shorter than a few NVML polls: include the warm-up just before it
            rows, where = [r for r in self.rows if r[0] <= t_end], "warm-up + timed region"
        names = {nv.nvmlClocksEventReasonHwSlowdown: "hw_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksEventReasonSwThermalSlowdown: "sw_thermal_slowdown", nv.nvmlClocksEventReasonSwPowerCap: "sw_power_cap",
                 nv.nvmlClocksEventReasonHwPowerBrakeSlowdown: "hw_power_brake"}
        reasons = sorted({n for r in rows for bit, n in names.items() if r[2] & bit})
        sm = [r[1] for r in rows]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_min_mhz": min(sm) if sm else None,
                "sm_max_mhz": self.max_sm, "samples": len(sm),
                "power_w_max": max((r[3] for r in rows), default=None),
                "power_w_median": statistics.median([r[3] for r in rows]) if rows else None,
                "window": where, "reasons": reasons}


# ------------------------------------------------------------------------------------------
# The reference's path on the host cores
# ------------------------------------------------------------------------------------------
def usable_cpus():
    """Logical CPUs this process may actually use: sched_getaffinity capped by the cgroup CPU quota
    (os.cpu_count() reports the machine, not the container)."""
    try:
        n_aff = len(os.sched_getaffinity(0))
    except Exception:
        n_aff = os.cpu_count() or 1
    quota = None
    try:
        parts = open("/sys/fs/cgroup/cpu.max").read().split()          # cgroup v2
        if parts and parts[0] != "max":
            quota = float(parts[0]) / float(parts[1])
    except Exception:
        try:                                                            # cgroup v1
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0 and p > 0:
                quota = q / p
        except Exception:
            pass
    cap = n_aff if quota is None else max(1, min(n_aff, int(math.floor(quota + 1e-9))))
    return cap, n_aff, quota


def build_cpu_model():
    """The reference's own class (oracle/_ref/models.py, a build-time copy of bin/models.py) re-instantiated for the
    benchmark shape as tests/golden/make_golden.py does; the restatement when the copy is absent."""
    from oracle import ref_models
    cls = ref_models.reference_class()
    if cls is not None:
        return ref_models.stretched(cls, KIND, C, W, seed=0), "reference"
    from oracle import mycnn_torch as O
    return O.make_ref(O.stretched(O.ARCH_MYCNN5, C, W), seed=0), "port"


def _cpu_worker(idx, conn, counter):
    """One single-threaded scorer: per-window model(x[i:i+1], age[i:i+1]) under no_grad
    (bin/predictStream.py:154-157), PyTorch-CPU fp32.  Stays alive across steps.  Within a step the workers
    pull windows from ONE shared counter until the step's total is scored, so a worker the container's CPU
    quota throttles does not decide the step time by itself."""
    try:
        torch.set_num_threads(1)
        import tskd_b200
        model, kind = build_cpu_model()
        n = 8
        x = tskd_b200.synth.make_windows(n, C, W, "normal", seed=1234 + idx, dtype=torch.bfloat16).float()
        ages = tskd_b200.synth.make_ages(n, seed=1234 + idx)
        with torch.no_grad():
            for i in range(2):
                model(x[i:i + 1], ages[i:i + 1])
        conn.send(("ready", kind))
        while True:
            cmd = conn.recv()
            if cmd[0] == "stop":
                break
            _, t_at = cmd
            while time.perf_counter() < t_at:        # CLOCK_MONOTONIC: one time base for all processes
                time.sleep(0.0005)
            t0 = time.perf_counter()
            done = 0
            with torch.no_grad():
                while True:
                    with counter.get_lock():
                        if counter.value <= 0:
                            break
                        counter.value -= 1
                    i = done % n
                    model(x[i:i + 1], ages[i:i + 1])
                    done += 1
            conn.send((t0, time.perf_counter(), done))
    except Exception as e:                            # never leave the parent waiting
        try:
            conn.send(("error", repr(e)))
        except Exception:
            pass


class CpuPool:
    """All host cores on the reference's path.  One torch process with N intra-op threads is SLOWER than one
    thread on this per-window call (137 vs 461 windows/s measured on a 64-core box: the ops are too small to
    split), so the cores are used the way the path shards: one single-threaded scorer process per usable CPU, each
    looping predictStream-style over windows.  The workers are spawned once and stay alive; the number of ACTIVE
    workers is calibrated (hyper-threads / memory bandwidth / a cgroup quota can make fewer workers faster)."""

    def __init__(self, max_workers=None):
        import torch.multiprocessing as mp
        self.cap, self.n_aff, self.quota = usable_cpus()
        n = min(self.cap, max_workers or 128)
        ctx = mp.get_context("spawn")
        self.counter = ctx.Value("q", 0)
        self.procs, self.conns = [], []
        for i in range(n):
            a, b = ctx.Pipe()
            p = ctx.Process(target=_cpu_worker, args=(i, b, self.counter), daemon=True)
            p.start()
            self.procs.append(p); self.conns.append(a)
        self.kind = None
        for c in self.conns:
            if not c.poll(600):
                raise RuntimeError("CPU worker did not start")
            msg = c.recv()
            if msg[0] != "ready":
                raise RuntimeError(f"CPU worker failed: {msg}")
            self.kind = msg[1]
        self.active = n

    def step(self, active, total):
        """`active` workers score `total` windows between them, started together; returns (windows, wall_s, per-worker counts)."""
        with self.counter.get_lock():
            self.counter.value = int(total)
        t_at = time.perf_counter() + 0.02
        for c in self.conns[:active]:
            c.send(("run", t_at))
        res = []
        for c in self.conns[:active]:
            if not c.poll(1800):
                raise RuntimeError("CPU worker timed out")
            r = c.recv()
            if r[0] == "error":
                raise RuntimeError(f"CPU worker failed: {r[1]}")
            res.append(r)
        wall = max(r[1] for r in res) - t_at
        done = sum(r[2] for r in res)
        assert done == int(total), (done, total)
        return done, wall, [r[2] for r in res]

    def calibrate(self, seconds=1.5):
        """Pick the active-worker count with the best whole-pool throughput (candidates: all usable CPUs, 1/2, 1/4)."""
        n = len(self.procs)
        cands = sorted({n, max(1, n // 2), max(1, n // 4)}, reverse=True)
        table = []
        for a in cands:
            wins, w0, _ = self.step(a, 4 * a)                              # short probe -> windows for ~`seconds`
            total = max(2 * a, int(seconds * wins / w0))
            wins, wall, _ = self.step(a, total)
            table.append({"workers": a, "windows_per_s": wins / wall})
        best = max(table, key=lambda t: t["windows_per_s"])
        self.active = best["workers"]
        self.rate = best["windows_per_s"]
        return table

    def close(self):
        for c in self.conns:
            try:
                c.send(("stop",))
            except Exception:
                pass
        for p in self.procs:
            p.join(timeout=5)
            if p.is_alive():
                p.terminate()


def cpu_reference_run(steps, warmup, seconds_total):
    """K timed steps (after W warm-up steps) of the reference path on the calibrated pool; every step the active
    workers score the same fixed number of windows between them, sized so that the timed region lasts
    ~`seconds_total` (>= 5 s).  Returns the numbers both bench legs report."""
    pool = CpuPool()
    try:
        table = pool.calibrate()
        per_step_s = max(0.25, seconds_total / max(1, steps))
        total = max(2 * pool.active, int(round(per_step_s * pool.rate)))
        for _ in range(max(1, warmup)):
            pool.step(pool.active, total)
        wins = 0; wall = 0.0; counts = []; step_rates = []
        for _ in range(steps):
            n, dt, c = pool.step(pool.active, total)
            wins += n; wall += dt; counts.append(c); step_rates.append(n / dt)
        per_worker = [sum(col) / wall for col in zip(*counts)]
        return {"value": wins / wall, "windows": wins, "seconds": wall, "workers": pool.active, "kind": pool.kind,
                "windows_per_step": total, "calibration": table,
                "usable_cpus": pool.cap, "affinity_cpus": pool.n_aff, "cgroup_quota": pool.quota,
                "per_worker_windows_per_s": {"min": min(per_worker), "median": statistics.median(per_worker), "max": max(per_worker)},
                "step_windows_per_s": {"min": min(step_rates), "median": statistics.median(step_rates), "max": max(step_rates)}}
    finally:
        pool.close()


def cpu_baseline_block(r, steps):
    what = ("the UNMODIFIED reference class bin/models.py:MyCNN (build-time copy in oracle/_ref/), re-instantiated for [3,75000] as "
            "tests/golden/make_golden.py does" if r["kind"] == "reference" else "oracle/mycnn_torch.py (restatement of bin/models.py)")
    return {"value": r["value"], "unit": UNIT, "cores": r["workers"], "kind": r["kind"],
            "sample": (f"{r['windows']} windows in {r['seconds']:.1f} s: {steps} steps x {r['workers']} persistent single-thread worker "
                       f"processes sharing {r['windows_per_step']} windows per step (pulled from one counter), per-window model(x[i:i+1], age[i:i+1]) loop under no_grad "
                       f"(bin/predictStream.py:154-157) on {what}, torch {torch.__version__} CPU fp32"),
            "usable_cpus": r["usable_cpus"], "affinity_cpus": r["affinity_cpus"], "cgroup_quota": r["cgroup_quota"],
            "os_cpu_count": os.cpu_count(), "calibration": r["calibration"],
            "per_worker_windows_per_s": r["per_worker_windows_per_s"], "step_windows_per_s": r["step_windows_per_s"]}


def run_reference(args, rank):
    if rank != 0:
        return
    r = cpu_reference_run(args.steps, args.warmup, max(6.0, args.ref_seconds))
    v = r["value"]
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 * r["seconds"] / max(1, args.steps), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload(B_PER_GPU),
        "cpu_baseline": cpu_baseline_block(r, args.steps),
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}))


# ------------------------------------------------------------------------------------------
def oracle_parity(model, x, ages, y, n_check):
    """The benchmarked tensors against the CPU oracle: `n_check` windows spread over the batch, the logits the
    timed steps produced vs oracle/mycnn_torch.py with the model's own weights, per-element relative error."""
    from oracle import mycnn_torch as O
    B = x.shape[0]
    idx = torch.linspace(0, B - 1, min(n_check, B)).round().long().unique()
    ref = O.make_ref(O.stretched(O.ARCH_MYCNN5, C, W), seed=0)
    ref.load_state_dict({k: v.detach().cpu() for k, v in model.state_dict().items() if k in ref.state_dict()})
    xs = x[idx.to(x.device)].float().cpu()
    ags = ages[idx.to(ages.device)].cpu()
    t0 = time.perf_counter()
    # ONE thread: torch's multi-threaded GEMV over the 18745 LSTM inputs splits the reduction by thread, and how many threads
    # the OpenMP runtime actually hands out varies from run to run on a busy box -- seen once as a parity figure of 8.4e-6
    # instead of 1.6e-6 for bit-identical GPU results (scripts/cross_process_check.sh); single-threaded the oracle is reproducible
    nt = torch.get_num_threads()
    torch.set_num_threads(1)
    want = O.ref_independent(ref, xs, ags).double()
    torch.set_num_threads(nt)
    got = y[idx.to(y.device)].cpu().double()
    err = (got - want).abs()
    rel = err / want.abs().clamp_min(1e-30)
    # a logit within 1e-4 * max|logit| of zero has no meaningful relative error: judged on the absolute one
    floor = 1e-4 * float(want.abs().max())
    small = want.abs() < 1e-2 * float(want.abs().max())
    max_rel = float(rel[~small].max()) if (~small).any() else 0.0
    ok = bool((rel[~small] <= PARITY_TOL).all()) and bool((err[small] <= floor).all())
    return {"n": int(idx.numel()), "max_rel": max_rel, "max_abs": float(err.max()), "max_abs_logit": float(want.abs().max()),
            "small_logits_judged_abs": int(small.sum()), "tol_rel": PARITY_TOL, "ok": ok,
            "oracle": "oracle/mycnn_torch.py per-window loop, torch CPU fp32", "seconds": time.perf_counter() - t0}


def production_shape_block(dev, with_cpu):
    """NOT the headline: the reference's production call shape (bin/predictStream.py:105,157, config.cfg:23) -- one
    [1,10,120] window per patient row -- through the same public API: latency of the single call with device and with host
    tensors, and all patients of a trigger as ONE predict() over [P,10,120]; each with an in-run check against the oracle
    and, beside it, the reference class itself timed single-threaded on this host (BASELINE.md section 2: 462 us/call)."""
    import tskd_b200
    from oracle import mycnn_torch as O
    from oracle import ref_models
    m = tskd_b200.B200MyCNN(tskd_b200.ARCH_PRESETS["mycnn5"]).to(dev)
    ref = O.make_ref(O.ARCH_MYCNN5, seed=0)
    m.load_state_dict(ref.state_dict())
    blk = {"shape": "[P,10,120] fp32, MyCNN5 (the checkpoint's own geometry)", "weights": "default init, seed 0"}

    def host_us(fn, n):
        for _ in range(max(20, n // 20)):
            fn()
        torch.cuda.synchronize(dev)
        t0 = time.perf_counter()
        for _ in range(n):
            fn()
        torch.cuda.synchronize(dev)
        return (time.perf_counter() - t0) / n * 1e6

    g = torch.Generator().manual_seed(7)
    x1h = torch.randn(1, 10, 120, generator=g) * 20 + 80
    a1h = torch.tensor([65.0])
    x1, a1 = x1h.to(dev), a1h.to(dev)
    with torch.no_grad():
        want1 = float(ref(x1h, a1h))
    got1 = float(m(x1, a1)[0])
    blk["single_call"] = {"device_tensors_us": host_us(lambda: m(x1, a1), 3000),
                          "call_plan_us": host_us(m.call_plan(x1, a1), 3000),
                          "host_tensors_us": host_us(lambda: m(x1h, a1h), 1000),
                          "launches_per_call": int(m.gpu_launches), "path": m.last_path,
                          "rel_err_vs_oracle": abs(got1 - want1) / max(abs(want1), 1e-30),
                          "note": "back-to-back calls, wall clock / n; host_tensors = H2D + kernel + D2H per call as predictStream.py:155-160 does it"}
    trig = {}
    for P in (256, 4096, 32768):
        xp = (torch.randn(P, 10, 120, generator=g) * 20 + 80).to(dev)
        ap_ = (torch.rand(P, generator=g) * 70 + 18).to(dev)
        for _ in range(5):
            yp = m.predict(xp, ap_)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(dev)
        e0.record()
        for _ in range(50):
            yp = m.predict(xp, ap_)
        e1.record()
        torch.cuda.synchronize(dev)
        us = e0.elapsed_time(e1) / 50 * 1e3
        n_chk = min(P, 128)
        want = O.ref_independent(ref, xp[:n_chk].cpu(), ap_[:n_chk].cpu()).double()
        got = yp[:n_chk].cpu().double()
        rel = float((got - want).abs().max() / want.abs().max().clamp_min(1e-6))     # as tests/conftest.py rel_err
        trig[str(P)] = {"us_per_call": us, "windows_per_s": P / (us / 1e6), "launches_per_call": int(m.gpu_launches),
                        "max_rel_vs_oracle": rel, "n_checked": n_chk}
    blk["trigger_batch"] = trig
    blk["parity_ok"] = bool(blk["single_call"]["rel_err_vs_oracle"] <= PARITY_TOL and all(t["max_rel_vs_oracle"] <= PARITY_TOL for t in trig.values()))
    if with_cpu:
        cls = ref_models.reference_class()
        cpu_m = ref if cls is None else cls().eval()
        if cls is not None:
            cpu_m.load_state_dict(ref.state_dict(), strict=False)
        nt = torch.get_num_threads()
        torch.set_num_threads(1)
        with torch.no_grad():
            for _ in range(50):
                cpu_m(x1h, a1h)
            t0 = time.perf_counter()
            for _ in range(1000):
                cpu_m(x1h, a1h)
            us_cpu = (time.perf_counter() - t0) / 1000 * 1e6
        torch.set_num_threads(nt)
        blk["reference_cpu"] = {"us_per_call": us_cpu, "threads": 1, "kind": "reference" if cls is not None else "port",
                                "note": "output = model(x_arr, a_arr) with [1,10,120] under no_grad, torch CPU fp32 (bin/predictStream.py:157)"}
    return blk


def dump_outputs(out_dir, arrays):
    """One float32 .npy per output tensor.  Inputs and weights are seeded, so two builds run with the same arguments can be
    compared array for array."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, f"{name}.npy"), t.detach().float().cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=B_PER_GPU, help="windows per GPU (default: the BASELINE config)")
    ap.add_argument("--path", default="auto", choices=["auto", "generic", "tensorcore"])
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--sustained-seconds", type=float, default=3.0)
    ap.add_argument("--parity-windows", type=int, default=256)
    ap.add_argument("--cpu-seconds", type=float, default=10.0, help="timed CPU work of the cpu_baseline leg (N=1 only)")
    ap.add_argument("--ref-seconds", type=float, default=10.0, help="timed CPU work of the whole --impl reference run")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--extra-steps", type=int, default=10, help="steps of the `extra` block (tc_splits=2 option line); 0 = skip")
    ap.add_argument("--dtype", default="bf16", choices=["bf16", "f32"],
                    help="window dtype: bf16 is the BASELINE workload; f32 (the reference's native dtype) is an extra line")
    ap.add_argument("--tc-splits", type=int, default=3, help="bf16 pieces per fp32 conv1 weight on the tensor cores (3 = fp32-equivalent)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the logits predict() returned in the last timed step to DIR/logits.npy (float32; "
                         "DIR/logits_rank<r>.npy per rank when N > 1) to compare two builds output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to the b200 arm")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.warmup < 3:
        args.warmup = 3

    import torch.distributed as dist
    import tskd_b200
    from tskd_b200.dist import broadcast_weights

    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    B = args.batch
    arch = tskd_b200.ARCH_PRESETS[KIND].with_shape(C, W)
    torch.manual_seed(0 if rank == 0 else 1000 + rank)     # only rank 0's weights survive
    model = tskd_b200.B200MyCNN(arch, path=args.path, tc_splits=args.tc_splits).to(dev)
    if world > 1:
        broadcast_weights(model, src=0)                    # the one init-time NCCL collective
    esz = 2 if args.dtype == "bf16" else 4
    x = tskd_b200.synth.make_windows(B, C, W, "normal", seed=1234 + rank, dtype=torch.bfloat16, device=dev)
    if args.dtype == "f32":
        x = x.float()                                      # same bf16-representable values, fp32 storage
    ages = tskd_b200.synth.make_ages(B, seed=1234 + rank, device=dev)
    model.set_profile(True)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()
    for _ in range(args.warmup):
        y = model.predict(x, ages)
    barrier()
    launches_per_step = model.gpu_launches
    path = model.last_path

    t_begin = time.perf_counter()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    barrier()
    ev[0].record()
    for s in range(args.steps):
        y = model.predict(x, ages)
        ev[s + 1].record()
    barrier()
    t_end = time.perf_counter()
    total_ms = ev[0].elapsed_time(ev[args.steps])
    # the dominant kernel's own duration: events the library recorded around it on the same
    # stream inside the timed region (last step's value; steps are identical)
    k_ms = model.last_stage_ms(0)
    head_ms = model.last_stage_ms(1)
    clocks = sampler.summary(t_begin, t_end) if sampler else None
    t = torch.tensor([total_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms = float(t.item())
    value = world * B * args.steps / (total_ms / 1e3)
    assert torch.isfinite(y).all()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"logits" if world == 1 else f"logits_rank{rank}": y})

    # ---- sustained: >= 3 s of back-to-back steps (the 12 ms headline region is a burst; an issue-bound
    #      kernel scales with the SM clock, which sags under sustained load) -----------------------------
    model.set_profile(False)
    sustained = None
    if args.sustained_seconds > 0:
        n_sus = max(args.steps, int(math.ceil(args.sustained_seconds / (total_ms / args.steps / 1e3) * 1.05)))
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        ts0 = time.perf_counter()
        e0.record()
        for _ in range(n_sus):
            ys = model.predict(x, ages)
        e1.record()
        barrier()
        ts1 = time.perf_counter()
        sus_ms = e0.elapsed_time(e1)
        tt = torch.tensor([sus_ms], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        sus_ms = float(tt.item())
        assert torch.equal(ys, y), "sustained steps must reproduce the timed steps bit-for-bit"
        sustained = {"steps": n_sus, "seconds": sus_ms / 1e3, "ms_per_step": sus_ms / n_sus,
                     "value": world * B * n_sus / (sus_ms / 1e3), "unit": UNIT,
                     "clocks": sampler.summary(ts0 + 0.25 * (ts1 - ts0), ts1, fallback_all=False) if sampler else None}
    model.set_profile(True)

    # ---- e2e: the public predict() call with pinned HOST tensors, H2D + D2H timed ---------
    Be = min(B, 4096)                                       # e2e sample (pinned host copy); == B for the BASELINE batch
    xh = x[:Be].cpu().pin_memory()
    ah = ages[:Be].cpu().pin_memory()
    model.predict(xh[:256], ah[:256])                       # staging buffers allocated untimed
    model.predict(xh, ah)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.e2e_steps):
        yh = model.predict(xh, ah)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    te = torch.tensor([e2e_s], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
    e2e_value = world * Be * args.e2e_steps / float(te.item())
    assert torch.allclose(yh, y[:Be].cpu(), rtol=1e-5, atol=1e-6)
    # the PCIe roofline of that number: a plain pinned cudaMemcpyAsync of the same bytes, same run
    e2e_bytes = Be * (C * W * esz + 4)
    xd = torch.empty_like(x[:Be])
    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    xd.copy_(xh, non_blocking=True)
    torch.cuda.synchronize()
    reps = 3
    c0.record()
    for _ in range(reps):
        xd.copy_(xh, non_blocking=True)
    c1.record()
    torch.cuda.synchronize()
    h2d_gbs = reps * xh.numel() * esz / (c0.elapsed_time(c1) / 1e3) / 1e9
    del xd
    e2e_gbs = (e2e_bytes + Be * 4) * args.e2e_steps / float(te.item()) / 1e9

    if rank == 0:
        hbm_peak, peak_src = peaks()
        # algorithmic bytes per launch of the dominant kernel (SURVEY 8d): every window's input
        # once (C*W*esz B) + its logit (4 B) + the weights once per launch
        n_w = sum(v.numel() for k, v in model.state_dict().items() if k in tskd_b200.arch.BLOB_KEYS)
        alg_bytes = B * (C * W * esz + 4) + n_w * 4
        achieved = alg_bytes / (k_ms / 1e3) / 1e9 if k_ms and k_ms > 0 else None
        step_gbs = alg_bytes / (total_ms / args.steps / 1e3) / 1e9
        roof = {"bound": "hbm", "kernel": {"generic": "front end (conv1+pool+conv2+pool)", "stream": "fp32 streaming front end (CUDA-core conv1 + tcgen05 projection)"}.get(path, "tcgen05 fused front end"),
                "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                "frac": (achieved / hbm_peak) if achieved else None, "peak_source": peak_src,
                "kernel_ms": k_ms, "head_ms": head_ms, "algorithmic_bytes_per_launch": alg_bytes,
                "traffic": TRAFFIC.get(path),
                "whole_step_frac": step_gbs / hbm_peak,
                "sustained_step_frac": (alg_bytes / (sustained["ms_per_step"] / 1e3) / 1e9 / hbm_peak) if sustained else None,
                "compute_note": "co-bound by FP32/MUFU: 21.9 MFLOP + 169k tanh per window (DESIGN.md)"}
        parity = oracle_parity(model, x, ages, y, args.parity_windows) if args.parity_windows > 0 else None
        out = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
               "scaling": "weak", "vs_baseline": None, "dtype": "bf16 in / f32 math" if args.dtype == "bf16" else "f32", "data": "synthetic",
               "config": workload(B) if args.dtype == "bf16" else workload(B, "fp32 (extra line, not the BASELINE dtype)"),
               "path": path, "parallelism": f"dp{world} (window shards, no data-path collective)",
               "roofline": roof, "parity": parity, "clocks": clocks, "sustained": sustained,
               "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": e2e_bytes,
                       "d2h_bytes_per_step": Be * 4, "steps": args.e2e_steps, "note": "per GPU; pinned host tensors through predict()",
                       "pcie": {"h2d_peak_gbs": h2d_gbs, "achieved_gbs": e2e_gbs, "frac": e2e_gbs / h2d_gbs,      # per GPU: every rank moves its own shard over its own link
                                "peak_source": "pinned cudaMemcpyAsync H2D of the same buffer, same run (CUDA events)"}},
               "gpu_launches": launches_per_step * args.steps}
        if world == 1 and args.dtype == "bf16" and args.tc_splits == 3 and args.extra_steps > 0:
            # NOT the headline: the library option tc_splits=2 (conv1 weights as two bf16 pieces = 16 mantissa bits, 6 instead
            # of 9 MMAs per block; samples exact, fp32 accumulation).  The kernel sits on the board's power cap and the tensor
            # cores draw most of it, so a third fewer MMAs is a large step; reported with its own in-run parity figure.
            m2 = tskd_b200.B200MyCNN(arch, path=args.path, tc_splits=2).to(dev)
            m2.load_state_dict(model.state_dict())
            for _ in range(3):
                y2 = m2.predict(x, ages)
            torch.cuda.synchronize()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record()
            for _ in range(args.extra_steps):
                y2 = m2.predict(x, ages)
            f1.record()
            torch.cuda.synchronize()
            ms2 = f0.elapsed_time(f1) / args.extra_steps
            p2 = oracle_parity(m2, x, ages, y2, min(64, args.parity_windows)) if args.parity_windows > 0 else None
            out["extra"] = {"tc_splits_2": {"ms_per_step": ms2, "value": B / (ms2 / 1e3), "unit": UNIT, "steps": args.extra_steps,
                                            "whole_step_frac": alg_bytes / (ms2 / 1e3) / 1e9 / hbm_peak, "parity": p2,
                                            "max_abs_diff_vs_headline_logits": float((y2 - y).abs().max()),
                                            "note": "option, not the default: conv1 weights rounded to 16 mantissa bits (two bf16 pieces)"}}
            del m2
        if world == 1 and args.dtype == "bf16" and args.extra_steps > 0:
            try:                                        # an extra block never costs the headline line
                ps = production_shape_block(dev, not args.no_cpu_baseline)
            except Exception as e:                      # noqa: BLE001
                ps = {"error": f"{type(e).__name__}: {e}"}
            out.setdefault("extra", {})["production_shape"] = ps
            if not ps.get("parity_ok", False):
                print(f"bench.py: production-shape extra block: {ps}", file=sys.stderr)
        if world == 1 and not args.no_cpu_baseline:
            steps_cpu = 10
            r = cpu_reference_run(steps_cpu, 1, max(5.0, args.cpu_seconds))
            out["cpu_baseline"] = cpu_baseline_block(r, steps_cpu)
        print(json.dumps(out))
        if parity is not None and not parity["ok"]:
            print(f"bench.py: PARITY FAILED {parity}", file=sys.stderr)
            sys.exit(3)
    if sampler:
        sampler.stop()
    if world > 1:
        dist.destroy_process_group()


# dram__bytes_read.sum + dram__bytes_write.sum per launch of the dominant kernel, from the
# committed ncu captures under profiles/ (None until a capture exists for that path).
TRAFFIC = {"generic": 1.846642e9 + 0.297926e9,      # profiles/r01_generic_frontend_ncu_full.txt (features written to HBM)
           "tensorcore": 1.974513e9 + 0.032842e9,   # profiles/r02_final2_fused_ncu_full.txt (halo re-reads + gate partials)
           "stream": 3.801502e9 + 0.034493e9}       # profiles/r01_final_stream_ncu_full.txt (fp32 windows)

if __name__ == "__main__":
    main()
