#!/usr/bin/env python
"""bench.py — entity-steps/s of the B200 six_dof() RK4 path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl b200|reference] [--worlds M] [--dump-outputs DIR]

One "step" = one RK4 tick of the hot path over the whole batch of synthetic worlds
(one body kernel launch, the state streaming HBM -> registers -> HBM).  Workload at
every N: BASELINE.json configs[1] — the cube-sat single 6DOF body, RK4, dt = 1e-3 —
batched over the Monte-Carlo world axis (SURVEY §8d C2 "also run M = 2^20.. copies for
throughput"): 1 body x M worlds per GPU, M = 2^22 (read set 671 MB > 126 MB L2), weak
scaling (per-GPU work fixed, worlds shard with no data-path collective).  The literal
configs[1] latency chain (1 body, dependent steps) is reported beside it as
`single_body`.

value     whole-job entity-steps/s, inputs resident in HBM, CUDA-event timed on the
          launching stream, max over ranks.
e2e       the same metric through the reference-shaped C-ABI call
          b200_sixdof_invoke_batch with pinned HOST buffers (NUMA-local to the GPU): every call
          uploads every live input column (pos, vel, inertia), integrates `ticks_per_call` ticks and
          downloads the state (pos, vel); `e2e.curve` repeats it at 1 / 10 / 100 / 1000 ticks per call,
          `e2e.all_outputs` with every output column (the round-1 contract), `e2e.pcie` is the
          concurrent host<->device copy bandwidth of all ranks — the ceiling e2e sits under.
verified  the timed executor's final state (256 strided worlds) against the CPU oracle advanced the
          same number of ticks: the timed launches did the work.
roofline  algorithmic 264 B/entity-step (SURVEY §8d) / mean kernel time vs the measured
          HBM copy peak (MEASURED_PEAKS.json, else the 6.65 TB/s fallback).
multi_gpu BASELINE configs[3] (n-body 1024, sharded worlds; one world: replicas vs row shards) and
          configs[4] (falcon9-style Monte-Carlo, 100 000 rollouts over the N GPUs, wall time including
          the end-of-run NCCL gather done inside libb200_sixdof.so).
cpu_baseline / --impl reference
          the CPU oracle port of the reference arithmetic (oracle/, the reference's
          Rust+JAX+Cranelift stack cannot be built here) on every CPU this process may use,
          one driver call for the whole run (threads created once), >= 1 s timed.
"""

from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the benchmark only reads the tree build() left (it may be read-only)

import numpy as np

B_ALG = 264  # algorithmic bytes per entity-step, f64: read pos 56 + vel 48 + inertia 56, write pos 56 + vel 48
B_TOUCHED = 240  # what the free-body kernel moves: the 3 momentum planes of Inertia (24 B) are never read
DT = 1.0e-3
METRIC = "entity-steps/sec (6DOF RK4)"
UNIT = "entity-steps/s"


def synth_world(M: int, seed: int):
    """cube-sat-like bodies (examples/cube-sat/main.py:14-16: omega = normalize([1,1,1]) * 80 deg/s,
    m = 2.8252 kg) perturbed per world so that no two worlds are identical (SURVEY §8d synthetic inputs)."""
    rng = np.random.default_rng(seed)
    q = rng.normal(size=(M, 1, 4))
    q /= np.linalg.norm(q, axis=-1, keepdims=True)
    pos = np.concatenate([q, rng.uniform(-1e3, 1e3, (M, 1, 3))], -1)
    w0 = np.array([1.0, 1.0, 1.0]) / np.sqrt(3.0) * np.radians(80.0)
    vel = np.concatenate([w0 + rng.normal(0, 0.05, (M, 1, 3)), rng.normal(0, 10, (M, 1, 3))], -1)
    ine = np.concatenate([rng.uniform(0.01, 0.05, (M, 1, 3)), np.zeros((M, 1, 3)), np.full((M, 1, 1), 2.8252)], -1)
    return np.ascontiguousarray(pos), np.ascontiguousarray(vel), np.ascontiguousarray(ine)


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_traffic(workload_key: str):
    """dram bytes per launch of the dominant kernel from the committed ncu --set full capture."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            return json.load(f).get(workload_key)
    except Exception:
        return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.perf_counter(), [c.strip() for c in line.split(",")]))

    def wait_first(self, timeout=5.0):
        t0 = time.perf_counter()
        while self.proc and not self.rows and time.perf_counter() - t0 < timeout:
            time.sleep(0.02)

    def stop(self, t_begin=None, t_end=None):
        """Summarise the samples taken while the timed region [t_begin, t_end] ran (under load)."""
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        rows = [r for (t, r) in self.rows if (t_begin is None or t >= t_begin) and (t_end is None or t <= t_end + 0.06)]
        sm = [float(r[1]) for r in rows if len(r) > 2 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows_all() if len(r) > 2 and r[2].replace(".", "").isdigit()]
        reasons = set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in rows:
            for name, v in zip(names, r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples_under_load": len(sm), "samples_total": len(self.rows)}

    def rows_all(self):
        return [r for (_, r) in self.rows]


def effective_cores() -> int:
    """CPUs this process may run on: scheduler affinity clipped by the cgroup quota (not os.cpu_count())."""
    n = len(os.sched_getaffinity(0))
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, -(-int(quota) // int(period))))
    except Exception:
        pass
    return max(n, 1)


def cpu_oracle_run(worlds: int, ticks: int, threads: int, warm_ticks: int = 1, seed: int = 1):
    """One driver call of the CPU oracle port (checker code, timed as the CPU baseline only): every thread is
    created once and integrates its share of the worlds for all `ticks` (the reference's Monte-Carlo workers run a
    world to completion each, libs/monte-carlo/src/lib.rs:2530-2538).  Returns (entity-steps/s, seconds)."""
    from oracle import oracle as O

    pos, vel, ine = synth_world(worlds, seed)
    w = O.World(pos, vel, ine)
    if warm_ticks:
        w.rk4(DT, warm_ticks, threads=threads)
    t0 = time.perf_counter()
    w.rk4(DT, ticks, threads=threads)
    dt = time.perf_counter() - t0
    return worlds * ticks / dt, dt


def cpu_arm(steps: int, warmup: int, target_s: float):
    """The CPU arm both `--impl reference` and the GPU arm's `cpu_baseline` report: the same function, the same
    sample rule, so the two agree on one box.  A step = one tick over `worlds` worlds; `worlds` is the largest power
    of two (2^12..2^22 = the GPU arm's batch) that keeps `steps` ticks near `target_s` seconds on this host."""
    from oracle import oracle as O

    threads = min(O.max_threads(), effective_cores())
    r1, _ = cpu_oracle_run(1 << 12, 100, 1)                      # one thread, 0.2 s
    rN, _ = cpu_oracle_run(1 << 16, 40, threads)                 # calibration, all threads
    worlds = 1 << 12
    while worlds < (1 << 22) and 2 * worlds * steps <= rN * target_s:
        worlds *= 2
    ticks = steps
    if worlds * ticks < rN * 1.0:                                # keep the timed region >= ~1 s: more ticks per world
        ticks = int(rN * 1.2 / worlds) + 1
    rate, secs = cpu_oracle_run(worlds, ticks, threads, warm_ticks=max(warmup, 1))
    return {"value": rate, "unit": UNIT, "cores": threads, "kind": "port",
            "one_thread_value": r1, "all_threads_over_one": rate / r1,
            "sample": f"{worlds} worlds x {ticks} ticks in {secs:.2f} s, oracle/sixdof_oracle.c, {threads} threads created once "
                      f"(one orc_rk4_ticks call); 1 thread: {r1:.3e} entity-steps/s",
            "worlds": worlds, "ticks": ticks, "seconds": secs}


def run_reference(args):
    """--impl reference: the reference's CPU path.  Its Rust/JAX/Cranelift stack cannot be
    built in this image, so this arm times the oracle port (oracle/sixdof_oracle.c, validated
    bit-for-bit against the reference's golden telemetry) on every CPU the process may use."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cpu = cpu_arm(args.steps, args.warmup, target_s=20.0)
    value = cpu["value"]
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": cpu["seconds"] / cpu["ticks"] * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": "cube-sat 6DOF RK4 dt=1e-3, 1 body x M worlds (BASELINE configs[1] batched over the Monte-Carlo world axis); "
                               f"CPU sample of {cpu['worlds']} worlds per step",
                   "worlds_per_step": cpu["worlds"], "ticks_timed": cpu["ticks"], "dt": DT, "integrator": "rk4"},
        "cpu_baseline": {k: cpu[k] for k in ("value", "unit", "cores", "kind", "sample", "one_thread_value", "all_threads_over_one")},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def bind_to_gpu_numa(index: int):
    """Pin this rank's host threads (and therefore its first-touch pinned buffers) to the CPUs
    NVML reports as local to GPU `index`.  With 8 ranks pushing PCIe traffic at once, leaving
    every rank on NUMA node 0 makes the host memory system the e2e bottleneck."""
    try:
        import pynvml

        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(index)
        n_cpu = os.cpu_count() or 1
        words = pynvml.nvmlDeviceGetCpuAffinity(h, (n_cpu + 63) // 64)
        cpus = {w * 64 + b for w, mask in enumerate(words) for b in range(64) if (mask >> b) & 1}
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def run_baseline_configs(args, torch, el, stream, local, rank, world_size):
    """The other BASELINE.json configs (parity-test cases, reported for context; not the headline)."""
    out = {}
    ev = lambda: torch.cuda.Event(enable_timing=True)

    def timed(ex, ticks, warm):
        ex.set_stream(stream.cuda_stream)
        with torch.cuda.stream(stream):
            ex.step(warm)
            torch.cuda.synchronize()
            a, b = ev(), ev()
            a.record(stream)
            ex.step(ticks)
            b.record(stream)
            torch.cuda.synchronize()
        return a.elapsed_time(b)

    rng = np.random.default_rng(42)
    # configs[2]: rocket 6DOF + gravity + thrust + drag, 10k Monte-Carlo worlds, 5000 steps @120 Hz (SURVEY §8d C3)
    M = 10000
    q = el.Quaternion.from_euler([0.0, np.radians(70.0), 0.0]).arr
    pos = np.tile(np.concatenate([q, [0, 0, 1.0]]), (M, 1, 1))
    vel = np.zeros((M, 1, 6))
    ine = np.tile(np.array([0.1, 1.0, 1.0, 0, 0, 0, 3.0]), (M, 1, 1))
    effs = [el.GravityConst((0, 0, -9.81)), el.ThrustBody((-1.0, 0, 0), "thrust"),
            el.DragQuadratic(column="wind", per_body_params=True)]
    # per-world drag: wind ~ N(0,1), Cd*rho ~ U(0.3, 0.9), A ~ U(1e-3, 1e-2)  (SURVEY §8d C3: per-world Cd*rho*A)
    drag_col = np.concatenate([rng.normal(0, 1, (M, 1, 3)), rng.uniform(0.3, 0.9, (M, 1, 1)), rng.uniform(1e-3, 1e-2, (M, 1, 1))], -1)
    for math in ("fast", "exact"):
        ex = el.B200Exec(1, M, 0.008333333, None, effs, "rk4", math, device=local, max_fused_ticks=100)
        ex.set_state(pos, vel, ine, thrust=np.full((M, 1, 1), 88.426), wind=drag_col)
        ms = timed(ex, 5000, 100)
        out[f"rocket_10k_worlds_{math}"] = {"worlds": M, "steps": 5000, "seconds": ms * 1e-3, "value": M * 5000 / (ms * 1e-3), "unit": UNIT}
        ex.close()
    # configs[3]: n-body, 1024 bodies pairwise softened gravity + 6DOF (SURVEY §8d C4), M = 1 and M = 8
    N = 1024
    for Mw in (1, 8):
        p = np.zeros((Mw, N, 7)); p[..., 3] = 1.0; p[..., 4:] = rng.uniform(-30, 30, (Mw, N, 3))
        v = np.zeros((Mw, N, 6)); v[..., 3:] = rng.normal(0, 1e-7, (Mw, N, 3))
        m = 10 ** rng.uniform(-10, -3, (Mw, N)); m[:, 0] = 1.0
        I = np.zeros((Mw, N, 7)); I[..., :3] = m[..., None]; I[..., 6] = m
        g = el.GravityEdges("softened", k_squared=2.9591220828e-4 / 86400.0 ** 2, softening=1e-10, edges=el.all_pairs_edges(N))
        for math in ("fast", "exact"):
            ex = el.B200Exec(N, Mw, 3600.0, None, [g], "rk4", math, device=local)
            ex.set_state(p, v, I)
            ticks = 200 if math == "fast" else 50
            ms = timed(ex, ticks, 5)
            out[f"nbody_1024_M{Mw}_{math}"] = {"bodies": N, "worlds": Mw, "steps": ticks, "us_per_tick": ms * 1e3 / ticks,
                                               "value": N * Mw * ticks / (ms * 1e-3), "unit": UNIT,
                                               "pair_evals_per_s": 3.0 * N * (N - 1) * Mw * ticks / (ms * 1e-3)}
            ex.close()
    # configs[4]: falcon9-style Monte-Carlo, 100k rollouts over 8 GPUs = 12.5k worlds per GPU, dt = 1e-3
    M = 12500
    pos = np.tile(np.array([0, 0, 0, 1.0, 6.4e6, 0, 0]), (M, 1, 1)) + np.concatenate([np.zeros((M, 1, 4)), rng.normal(0, 10, (M, 1, 3))], -1)
    vel = np.concatenate([rng.normal(0, 0.01, (M, 1, 3)), rng.normal(0, 50, (M, 1, 3))], -1)
    ine = np.tile(np.array([4e6, 4e6, 1e5, 0, 0, 0, 3e4]), (M, 1, 1))
    effs = [el.GravityFrame(), el.WrenchBody("body_wrench", "linear_first")]
    ex = el.B200Exec(1, M, 1e-3, None, effs, "rk4", "fast", device=local, max_fused_ticks=100)
    ex.set_state(pos, vel, ine, body_wrench=rng.normal(0, 1e4, (M, 1, 6)))
    ms = timed(ex, 10000, 100)
    out["falcon9_mc_12500_worlds_per_gpu_fast"] = {"worlds": M, "steps": 10000, "seconds": ms * 1e-3, "value": M * 10000 / (ms * 1e-3), "unit": UNIT}
    ex.close()
    # configs[0]: three-body, 1000 steps (plumbing; EXACT == oracle bit for bit is asserted in tests/ and smoke())
    G = 6.6743e-11
    p3 = np.array([[[0, 0, 0, 1, 0.8920281421, 0, 0], [0, 0, 0, 1, -0.6628498947, 0, 0], [0, 0, 0, 1, -0.2291782474, 0, 0]]], dtype=np.float64)
    v3 = np.array([[[0, 0, 0, 0, 0.9957939373, 0], [0, 0, 0, 0, -1.6191613336, 0], [0, 0, 0, 0, 0.6233673964, 0]]], dtype=np.float64)
    i3 = np.tile(np.array([1 / G, 1 / G, 1 / G, 0, 0, 0, 1 / G]), (1, 3, 1))
    edges3 = np.array([[0, 1], [1, 0], [0, 2], [1, 2], [2, 0], [2, 1]])
    for math in ("exact", "fast"):
        ex = el.B200Exec(3, 1, 0.008333333, None, [el.GravityEdges("newton", G=G, edges=edges3)], "rk4", math, device=local,
                         max_fused_ticks=32)
        ex.set_state(p3, v3, i3)
        ms = timed(ex, 1000, 32)
        out[f"three_body_1000_steps_{math}"] = {"steps": 1000, "us_per_tick": ms, "value": 3 * 1000 / (ms * 1e-3), "unit": UNIT,
                                               "note": "one world in one warp (small_world_kernel), 32 ticks per launch: a dependent "
                                                       "latency chain, no roofline"}
        ex.close()
    # the same system as a Monte-Carlo batch: 2^18 perturbed three-body worlds
    Mw = 1 << 18
    pM = np.tile(p3, (Mw, 1, 1)); pM[..., 4:] += rng.normal(0, 1e-3, (Mw, 3, 3))
    for math in ("exact", "fast"):
        ex = el.B200Exec(3, Mw, 0.008333333, None, [el.GravityEdges("newton", G=G, edges=edges3)], "rk4", math, device=local,
                         max_fused_ticks=32)
        ex.set_state(pM, np.tile(v3, (Mw, 1, 1)), np.tile(i3, (Mw, 1, 1)))
        ms = timed(ex, 64, 32)
        out[f"three_body_{Mw}_worlds_{math}"] = {"worlds": Mw, "steps": 64, "us_per_tick": ms * 1e3 / 64,
                                                 "value": 3 * Mw * 64 / (ms * 1e-3), "unit": UNIT}
        ex.close()
    return out


DUMP_WORLDS = 1 << 16  # worlds sampled by --dump-outputs: 4 f64 columns x 2^16 worlds = 13 MB


def dump_outputs(ex, out_dir: str):
    """Write the columns a caller of the timed executor downloads (WorldPos, WorldVel, WorldAccel, Force) as
    <out_dir>/<column>.npy, float64 [worlds, 1, width], for a fixed, seeded sample of DUMP_WORLDS worlds in
    ascending order (every world when the batch is smaller)."""
    from elodin_b200.executor import FORCE, WORLD_ACCEL, WORLD_POS, WORLD_VEL

    M = ex.n_worlds
    idx = np.sort(np.random.default_rng(0).choice(M, size=min(M, DUMP_WORLDS), replace=False))
    os.makedirs(out_dir, exist_ok=True)
    for name, cid in (("world_pos", WORLD_POS), ("world_vel", WORLD_VEL), ("world_accel", WORLD_ACCEL), ("force", FORCE)):
        np.save(os.path.join(out_dir, name + ".npy"), ex.download(cid)[idx])


def run_b200(args):
    import torch
    import torch.distributed as dist

    import elodin_b200 as el
    from elodin_b200.executor import FORCE, INERTIA, WORLD_ACCEL, WORLD_POS, WORLD_VEL

    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    world_size = int(os.environ.get("WORLD_SIZE", "1"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: elodin_b200 has no CPU fallback")
    torch.cuda.set_device(local)
    numa_cpus = bind_to_gpu_numa(local) if world_size > 1 else None
    distributed = world_size > 1
    if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"  # keep stdout to the one JSON line (NCCL prints its version banner there)
    if distributed:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    M = args.worlds
    K, W = args.steps, max(args.warmup, 3)
    pos, vel, ine = synth_world(M, 1000 + rank)
    stream = torch.cuda.Stream()
    from elodin_b200 import _lib

    fp64_peak = float(_lib.lib().b200_probe_fp64_gflops(local, 20000))   # DFMA issue rate of this GPU, GFLOP/s
    copy_probe = float(_lib.lib().b200_probe_copy_gbs(local, 1 << 30, 5))  # D2D copy, read + write GB/s

    def barrier():
        if distributed:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms: float) -> float:
        if not distributed:
            return ms
        t = torch.tensor([ms], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ------------------------------------------------------------------ device-resident throughput
    ex = el.B200Exec(1, M, DT, None, [], "rk4", "fast", device=local, max_fused_ticks=1)
    ex.set_stream(stream.cuda_stream)
    ex.set_state(pos, vel, ine)
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
        sampler.wait_first()
    with torch.cuda.stream(stream):
        ex.step(W)
        barrier()
        launches0 = ex.timings()["kernel_launches"]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        t_begin = time.perf_counter()
        e0.record(stream)
        ex.step(K)
        e1.record(stream)
        barrier()
        t_end = time.perf_counter()
        ms = max_over_ranks(e0.elapsed_time(e1))
        launches = ex.timings()["kernel_launches"] - launches0
        if args.dump_outputs and rank == 0:  # the state of the last timed step, before the clock replay below moves it on
            dump_outputs(ex, args.dump_outputs)
        window = "timed region"
        if ms * 1e-3 < 0.3:  # `ms` is the max over ranks, so every rank takes the same branch
            # too short for nvidia-smi's 50 ms period: replay the identical loop for ~0.5 s and sample that
            reps = max(1, int(0.5 / max(ms * 1e-3 / K, 1e-6)))
            barrier()
            t_begin = time.perf_counter()
            ex.step(reps)
            barrier()
            t_end = time.perf_counter()
            window = f"replay of the timed loop ({reps} steps; the timed region itself was {ms:.1f} ms)"
        clocks = sampler.stop(t_begin, t_end) if rank == 0 else None
        if clocks is not None:
            clocks["window"] = window
    # integrity sample: the state the TIMED executor ended in, for a strided set of worlds (checked against
    # the CPU oracle below, rank 0 / N = 1 only) — shows the timed launches really integrated every tick
    ticks_total = ex.tick
    vidx = np.arange(0, M, max(M // 256, 1))[:256]
    final_pos = ex.download(WORLD_POS)[vidx]
    final_vel = ex.download(WORLD_VEL)[vidx]
    value = world_size * M * K / (ms * 1e-3)
    kernel_ms = ms / K
    peak, peak_src = measured_peak()
    achieved = B_ALG * M / (kernel_ms * 1e-3) / 1e9

    if args.kernel_only:
        if rank == 0:
            print(json.dumps({"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world_size, "steps": K, "warmup": W,
                              "ms_per_step": kernel_ms, "roofline_frac": achieved / peak, "kernel_only": True}))
        ex.close()
        if distributed:
            dist.destroy_process_group()
        return 0

    # ------------------------------------------------------------------ secondary device numbers (rank 0, N=1 extras)
    extras = {}
    with torch.cuda.stream(stream):
        # fused ticks: state stays in registers across `fuse` ticks (invoke_batch with ticks_per_telemetry > 1)
        fx = el.B200Exec(1, M, DT, None, [], "rk4", "fast", device=local, max_fused_ticks=args.fuse)
        fx.set_stream(stream.cuda_stream)
        fx.set_state(pos, vel, ine)
        fx.step(args.fuse)
        barrier()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record(stream)
        fx.step(args.fuse * 4)
        f1.record(stream)
        barrier()
        fms = max_over_ranks(f0.elapsed_time(f1))
        extras["fused"] = {"ticks_per_launch": args.fuse, "value": world_size * M * args.fuse * 4 / (fms * 1e-3),
                           "unit": UNIT, "note": "FP64-pipe bound: HBM traffic amortised over the fused ticks"}
        fx.close()
        if rank == 0:
            # EXACT arithmetic (bit-identical to the reference-validated oracle)
            xM = min(M, 1 << 20)
            xx = el.B200Exec(1, xM, DT, None, [], "rk4", "exact", device=local)
            xx.set_stream(stream.cuda_stream)
            xx.set_state(pos[:xM], vel[:xM], ine[:xM])
            xx.step(3)
            torch.cuda.synchronize()
            x0, x1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            x0.record(stream)
            xx.step(10)
            x1.record(stream)
            torch.cuda.synchronize()
            extras["exact_math"] = {"value": xM * 10 / (x0.elapsed_time(x1) * 1e-3), "unit": UNIT, "worlds": xM}
            xx.close()
            # the same kernel with effector sets loaded (every stage rotates body-frame forces / torques):
            # rocket = const-g + body thrust + quadratic drag; falcon9 = rotating-frame gravity + body wrench
            rng = np.random.default_rng(5)
            sets = {
                "rocket": ([el.GravityConst(), el.ThrustBody((-1.0, 0.0, 0.0), "thrust"), el.DragQuadratic(0.6, 0.01, "wind")],
                           {"thrust": rng.uniform(50, 100, (M, 1, 1)), "wind": rng.normal(0, 1, (M, 1, 3))}, 264 + 8 * 4),
                "falcon9": ([el.GravityFrame(), el.WrenchBody("body_wrench", "linear_first")],
                            {"body_wrench": rng.normal(0, 1e3, (M, 1, 6))}, 264 + 8 * 6),
                # the cube-sat example's own effector shape (examples/cube-sat/main.py:492-527): reaction-wheel fold +
                # orbital gravity (J2 here: the example's EGM08 tables are a download), satellites on a 400 km orbit
                "cube_sat": ([el.TorqueBodyFold("wheel_torques", 3), el.GravityJ2()],
                             {"wheel_torques": rng.normal(0, 2e-3, (M, 1, 9))}, 264 + 8 * 9),
            }
            eff_out = {}
            for name, (effs, cols, bytes_per) in sets.items():
                p2 = pos.copy()
                if name in ("falcon9", "cube_sat"):
                    p2[..., 4:] += np.array([6.778e6 if name == "cube_sat" else 6.4e6, 0.0, 0.0])
                sx = el.B200Exec(1, M, DT, None, effs, "rk4", "fast", device=local)
                sx.set_stream(stream.cuda_stream)
                sx.set_state(p2, vel, ine, **cols)
                sx.step(5)
                torch.cuda.synchronize()
                q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                q0.record(stream)
                sx.step(100)
                q1.record(stream)
                torch.cuda.synchronize()
                t_ms = q0.elapsed_time(q1) / 100
                tr = ncu_traffic("body_fast_rk4_%s_bytes_per_launch_M%d" % (name, M))
                eff_out[name] = {"value": M / (t_ms * 1e-3), "unit": UNIT, "bytes_per_entity_step": bytes_per, "us_per_tick": t_ms * 1e3,
                                 "achieved_GBps": bytes_per * M / (t_ms * 1e-3) / 1e9, "frac": bytes_per * M / (t_ms * 1e-3) / 1e9 / peak,
                                 "traffic": tr, "dram_frac": (tr / (t_ms * 1e-3) / 1e9 / peak) if tr else None,
                                 "touched_bytes_per_entity_step": bytes_per - (B_ALG - B_TOUCHED),
                                 "kernel": "body_fast_spec_kernel<RK4, sig %s, 128 x 3, 2 bodies/thread>" % {"rocket": "THRUST|DRAG", "falcon9": "FRAME|WRENCH", "cube_sat": "WHEELS|J2"}[name]}
                sx.close()
                del p2, cols
            extras["effector_sets"] = eff_out
            # the cube-sat example's integrator (Integrator.SemiImplicit, examples/cube-sat/main.py:710) on the same set
            sx = el.B200Exec(1, M, DT, None, [el.TorqueBodyFold("wheel_torques", 3), el.GravityJ2()], "semi_implicit", "fast", device=local)
            sx.set_stream(stream.cuda_stream)
            p2 = pos.copy(); p2[..., 4:] += np.array([6.778e6, 0.0, 0.0])
            sx.set_state(p2, vel, ine, wheel_torques=rng.normal(0, 2e-3, (M, 1, 9)))
            sx.step(5)
            torch.cuda.synchronize()
            q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            q0.record(stream); sx.step(100); q1.record(stream)
            torch.cuda.synchronize()
            t_ms = q0.elapsed_time(q1) / 100
            eff_out["cube_sat_semi_implicit"] = {"value": M / (t_ms * 1e-3), "unit": UNIT, "bytes_per_entity_step": 336, "us_per_tick": t_ms * 1e3,
                                                 "achieved_GBps": 336 * M / (t_ms * 1e-3) / 1e9, "frac": 336 * M / (t_ms * 1e-3) / 1e9 / peak,
                                                 "note": "entity-steps of the semi-implicit integrator (one stage per tick), not RK4 ticks"}
            sx.close()
            del p2
            # spherical-harmonic gravity (GRAVITY_EGM08, degree 64 like the cube-sat example) on 2^16 satellites: its own
            # launch per tick, FP64-issue bound (synthetic Kaula-rule coefficients: the reference's tables are a download)
            gM, gL = 1 << 18, 64
            grng = np.random.default_rng(8)
            cb, sb = np.zeros((gL + 1, gL + 1)), np.zeros((gL + 1, gL + 1))
            for l_ in range(2, gL + 1):
                cb[l_, : l_ + 1] = grng.normal(0, 1e-5 / l_**2, l_ + 1)
                sb[l_, 1: l_ + 1] = grng.normal(0, 1e-5 / l_**2, l_)
            cb[0, 0], cb[2, 0] = 1.0, -1.08262668e-3 / np.sqrt(5.0)
            gx = el.B200Exec(1, gM, DT, None, [el.TorqueBodyFold("wheel_torques", 3), el.GravityEGM08(cb, sb, gL)], "rk4", "fast", device=local)
            gx.set_stream(stream.cuda_stream)
            gp = pos[:gM].copy(); gp[..., 4:] += np.array([6.778e6, 0.0, 0.0])
            gx.set_state(gp, vel[:gM], ine[:gM], wheel_torques=rng.normal(0, 2e-3, (gM, 1, 9)))
            gx.step(2)
            torch.cuda.synchronize()
            q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            q0.record(stream); gx.step(10); q1.record(stream)
            torch.cuda.synchronize()
            t_ms = q0.elapsed_time(q1) / 10
            extras["egm08_degree_64"] = {"worlds": gM, "us_per_tick": t_ms * 1e3, "value": gM / (t_ms * 1e-3), "unit": UNIT,
                                         "field_evaluations_per_s": 3 * gM / (t_ms * 1e-3),
                                         "terms_per_s": 3 * gM * ((gL + 1) * (gL + 2) // 2) / (t_ms * 1e-3),
                                         "fp64_pipe_frac": (3 * gM * ((gL + 1) * (gL + 2) // 2) / (t_ms * 1e-3) * 33.0 / (fp64_peak * 1e9 / 2.0)) if fp64_peak else None,
                                         "note": "cube-sat effector shape with the degree-64 series instead of J2: egm08_force_kernel (3 stage "
                                                 "positions per body and tick, 2145 terms each, the oracle's IEEE operations: 33 FP64 "
                                                 "instructions per term, none fused) + the wheel-fold body kernel; fp64_pipe_frac = those "
                                                 "instructions / the DFMA issue rate of the probe"}
            gx.close()
            del gp
            # telemetry on every tick: the trajectory ring adds 104 B per body and tick (13 more planes written)
            tcap = 16
            tx = el.B200Exec(1, M, DT, None, [], "rk4", "fast", device=local, trajectory_every=1, trajectory_capacity=tcap)
            tx.set_stream(stream.cuda_stream)
            tx.set_state(pos, vel, ine)
            tx.step(4)
            tx.sync()
            tx.trajectory_reset()
            torch.cuda.synchronize()
            q0, q1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            q0.record(stream); tx.step(tcap); q1.record(stream)
            torch.cuda.synchronize()
            t_ms = q0.elapsed_time(q1) / tcap
            extras["telemetry_every_tick"] = {"value": M / (t_ms * 1e-3), "unit": UNIT, "bytes_per_entity_step": 264 + 104, "us_per_tick": t_ms * 1e3,
                                              "achieved_GBps": 368 * M / (t_ms * 1e-3) / 1e9, "frac": 368 * M / (t_ms * 1e-3) / 1e9 / peak,
                                              "note": "free body, one (WorldPos, WorldVel) sample per tick into the device trajectory ring"}
            tx.close()
            # BASELINE configs[1] literally: ONE body, dependent steps (latency chain, one persistent launch per 10^4 ticks)
            sb = el.B200Exec(1, 1, DT, None, [], "rk4", "fast", device=local, max_fused_ticks=10000)
            sb.set_stream(stream.cuda_stream)
            sb.set_state(pos[:1], vel[:1], ine[:1])
            sb.step(10000)
            torch.cuda.synchronize()
            s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            n_single = 200000
            s0.record(stream)
            sb.step(n_single)
            s1.record(stream)
            torch.cuda.synchronize()
            sms = s0.elapsed_time(s1)
            extras["single_body"] = {"steps": n_single, "ns_per_step": sms * 1e6 / n_single,
                                     "value": n_single / (sms * 1e-3), "unit": UNIT,
                                     "note": "configs[1] as written: 1 body, 1e6 dependent steps = %.2f s" % (sms * 1e-3 * 1e6 / n_single)}
            sb.close()

    # ------------------------------------------------------------------ e2e through the C ABI with host buffers
    e2e = run_e2e(args, el, local, rank, world_size, barrier, max_over_ranks, numa_cpus)

    # ------------------------------------------------------------------ BASELINE configs[3] / configs[4] at N GPUs
    try:
        multi = run_multi_gpu(args, torch, dist, el, stream, local, rank, world_size, barrier, max_over_ranks, fp64_peak)
    except Exception as e:  # secondary section: never lose the headline line over it (a failure here is the same on every rank)
        import traceback

        multi = {"error": repr(e)[:300], "traceback_tail": traceback.format_exc()[-600:]}
    ex.close()

    if rank == 0:
        cpu = None
        verified = None
        traffic = ncu_traffic("body_fast_rk4_bytes_per_launch_M%d" % M)
        steady = ncu_traffic("body_fast_rk4_steady_bytes_per_launch_M%d" % M)
        if world_size == 1:
            from oracle import oracle as O

            cpu_full = cpu_arm(args.steps, args.warmup, target_s=args.cpu_seconds)
            cpu = {k: cpu_full[k] for k in ("value", "unit", "cores", "kind", "sample", "one_thread_value", "all_threads_over_one")}
            chk = O.World(pos[vidx], vel[vidx], ine[vidx]).rk4(DT, ticks_total, threads=min(cpu_full["cores"], 64))
            scale = lambda a: max(float(np.max(np.abs(a))), 1e-300)
            verified = {"worlds_checked": int(len(vidx)), "ticks": int(ticks_total), "against": "CPU oracle (exact arithmetic)",
                        "max_rel_err_q": float(np.max(np.abs(final_pos[..., :4] - chk.pos[..., :4])) / scale(chk.pos[..., :4])),
                        "max_rel_err_x": float(np.max(np.abs(final_pos[..., 4:] - chk.pos[..., 4:])) / scale(chk.pos[..., 4:])),
                        "max_rel_err_vel": float(np.max(np.abs(final_vel - chk.vel)) / scale(chk.vel))}
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world_size, "steps": K, "warmup": W,
            "ms_per_step": kernel_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": "cube-sat 6DOF RK4 dt=1e-3, 1 body x M worlds (BASELINE configs[1] batched over the Monte-Carlo world axis)",
                       "worlds_per_gpu": M, "bodies_per_world": 1, "dt": DT, "integrator": "rk4", "math": "fast (<=1e-12/tick vs exact)",
                       "ticks_per_launch": 1, "parallelism": f"worlds sharded x{world_size}, no data-path collective",
                       "l2_policy": "inputs larger than L2 (read set %.0f MB per tick > 126 MB)" % (160 * M / 1e6),
                       "e2e_ticks_per_call": e2e["ticks_per_call"], "e2e_worlds_per_gpu": args.e2e_worlds},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_entity_step": B_ALG, "kernel": "body_fast_spec_kernel<RK4, sig 0, 128 x 3, 2 bodies/thread>",
                         "kernel_ms": kernel_ms,
                         "dram_frac": (traffic / (kernel_ms * 1e-3) / 1e9 / peak) if traffic else None,
                         "touched_bytes_per_entity_step": B_TOUCHED,
                         "touched_frac": B_TOUCHED * M / (kernel_ms * 1e-3) / 1e9 / peak,
                         "traffic_steady": steady, "steady_dram_frac": (steady / (kernel_ms * 1e-3) / 1e9 / peak) if steady else None,
                         "copy_probe_GBps_this_run": copy_probe, "fp64_probe_GFLOPs_this_run": fp64_peak,
                         "note": "frac counts the algorithmic 264 B/entity-step against the measured copy peak and reads above 1.0 for "
                                 "two reasons: the kernel touches 240 B of them (the free tick never needs the three Inertia momentum "
                                 "planes), and consecutive launches walk the planes in opposite directions, so the tail of the "
                                 "previous launch's state is served from the 126 MB L2 (event-timed 152 -> 142 us per tick, "
                                 "profiles/r02_tune_snake.txt).  traffic = DRAM bytes of one cold-cache launch (ncu --set full); "
                                 "traffic_steady = DRAM bytes per launch with ncu --cache-control none (profiles/r02_steady_traffic.txt): "
                                 "the touched 240 B/body and nothing twice — ncu serialises launches, so the L2 saving of the "
                                 "alternating traversal is not visible to it and steady_dram_frac (traffic_steady / kernel time / "
                                 "peak) is an upper bound on what DRAM moves in the timed loop"},
            "e2e": e2e,
            "gpu_launches": int(launches),
            "verified": verified,
            "clocks": clocks,
            "cpu_baseline": cpu,
            "multi_gpu": multi,
            **extras,
        }
        if args.configs:
            line["baseline_configs"] = run_baseline_configs(args, torch, el, stream, local, rank, world_size)
        print(json.dumps(line))
    if distributed:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def run_e2e(args, el, local, rank, world_size, barrier, max_over_ranks, numa_cpus):
    """entity-steps/s through b200_sixdof_invoke_batch with pinned host columns: every call uploads the live input
    columns and downloads the outputs the caller reads.  Headline point: `--e2e-ticks` ticks per call, state outputs."""
    import ctypes as C

    from elodin_b200 import _lib
    from elodin_b200.executor import FORCE, INERTIA, WORLD_ACCEL, WORLD_POS, WORLD_VEL

    L = _lib.lib()
    eM = args.e2e_worlds
    epos, evel, eine = synth_world(eM, 2000 + rank)
    ee = el.B200Exec(1, eM, DT, None, [], "rk4", "fast", device=local, max_fused_ticks=args.fuse)
    tick_id, dt_id = el.component_id("tick"), el.component_id("simulation_time_step")
    host = {WORLD_POS: epos, WORLD_VEL: evel, INERTIA: eine, WORLD_ACCEL: np.zeros((eM, 1, 6)), FORCE: np.zeros((eM, 1, 6)),
            tick_id: np.zeros(1, dtype=np.uint64), dt_id: np.array([DT])}
    pin_in, pin_out = {}, {}
    for cid in ee.input_ids:
        a = el.pinned_empty(host[cid].shape, host[cid].dtype, device=local)  # on the NUMA node of this GPU's PCIe root
        a[...] = host[cid]
        pin_in[cid] = a
    for cid in ee.output_ids:
        pin_out[cid] = el.pinned_empty(host[cid].shape, host[cid].dtype, device=local)
    nodes = {"gpu_numa_node": int(L.b200_device_numa_node(local)), "host_buffer_node": int(L.b200_host_node_of(C.c_void_p(pin_in[WORLD_POS].ctypes.data)))}
    in_ptrs = [pin_in[c].ctypes.data for c in ee.input_ids]
    # the library does not upload dead inputs (Force is cleared before any effector runs; WorldAccel only enters as
    # 0*a_prev, which FAST math does not evaluate): these are the bytes that cross PCIe
    h2d = sum(pin_in[c].nbytes for c in ee.input_ids if c not in (FORCE, WORLD_ACCEL))

    def measure(T, calls, outputs, dirty=None):
        want = (WORLD_POS, WORLD_VEL, tick_id) if outputs == "state" else tuple(ee.output_ids)
        out_ptrs = [pin_out[c].ctypes.data if c in want else None for c in ee.output_ids]
        d2h = sum(pin_out[c].nbytes for c in ee.output_ids if c in want and c not in (INERTIA,))  # Inertia: host-to-host fill
        ins = in_ptrs if dirty is None else [pin_in[c].ctypes.data if c in dirty else None for c in ee.input_ids]
        up = h2d if dirty is None else sum(pin_in[c].nbytes for c in ee.input_ids if c in dirty and c not in (FORCE, WORLD_ACCEL))
        ee.invoke_batch_ptrs(in_ptrs, out_ptrs, T)  # warm (every column uploaded once)
        barrier()
        t0 = time.perf_counter()
        for _ in range(calls):
            ee.invoke_batch_ptrs(ins, out_ptrs, T)  # synchronous: returns with the outputs on the host
        el_s = time.perf_counter() - t0
        ms = max_over_ranks(el_s * 1e3)
        return {"ticks_per_call": T, "outputs": outputs, "value": world_size * eM * T * calls / (ms * 1e-3), "unit": UNIT,
                "ms_per_call": ms / calls, "calls": calls, "h2d_bytes_per_call": up, "d2h_bytes_per_call": d2h,
                "h2d_bytes_per_step": up / T, "d2h_bytes_per_step": d2h / T}

    head = measure(args.e2e_ticks, args.e2e_calls, "state")
    tm = ee.timings()
    checksum = float(np.sum(pin_out[WORLD_POS][:1024]))  # the host really has the result
    curve = [measure(T, max(3, min(args.e2e_calls, 5)), "state") for T in (1, 10, 100, 1000)]
    full = measure(args.e2e_ticks, args.e2e_calls, "all")
    # a host with the reference's dirty-component tracking (world.rs:43,249-252) re-uploads only what it modified: here
    # the state (as a per-cycle host system would), not the constant Inertia
    dirty = measure(args.e2e_ticks, args.e2e_calls, "state", dirty=(WORLD_POS, WORLD_VEL, tick_id, dt_id))
    ee.close()
    # the ceiling: every rank's H2D and D2H engines busy at once with the same byte counts, no kernels
    probe_h2d, probe_d2h = head["h2d_bytes_per_call"], head["d2h_bytes_per_call"]
    scratch = el.pinned_empty((probe_h2d + probe_d2h) // 8 + 1, np.float64, device=local)
    out2 = (C.c_double * 2)()
    barrier()
    L.b200_probe_pcie_gbs(local, C.c_void_p(scratch.ctypes.data), probe_h2d, probe_d2h, 5, out2)
    barrier()
    t_copy_ms = max(probe_h2d / max(out2[0], 1e-9), probe_d2h / max(out2[1], 1e-9)) / 1e6  # the slower direction bounds a call
    t_copy_ms = max_over_ranks(t_copy_ms)
    pcie = {"h2d_GBps_rank0": out2[0], "d2h_GBps_rank0": out2[1], "concurrent_ranks": world_size,
            "copy_bound_ms_per_call": t_copy_ms,
            "copy_bound_value": world_size * eM * head["ticks_per_call"] / (t_copy_ms * 1e-3),
            "e2e_frac_of_copy_bound": head["value"] / (world_size * eM * head["ticks_per_call"] / (t_copy_ms * 1e-3)),
            "note": "both copy engines of every rank moving one call's bytes at the same time, no kernels: what PCIe Gen5 x16 and "
                    "the host memory system allow; at 4-8 ranks the sockets' memory bandwidth, not the links, sets it"}
    el.pinned_free(scratch)
    for a in list(pin_in.values()) + list(pin_out.values()):
        el.pinned_free(a)
    return {**head, "curve": curve, "all_outputs": full, "dirty_inputs_only": dirty,
            "engine_busy_ms_last_call": {k: tm[k] for k in ("h2d_upload_ms", "kernel_invoke_ms", "d2h_download_ms", "invoke_wall_ms")},
            "api": "b200_sixdof_invoke_batch (pinned host columns in; WorldPos/WorldVel/tick out, other outputs NULL = not read)",
            "checksum": checksum, "host_cpus_bound": numa_cpus, "pcie": pcie, **nodes}


def run_multi_gpu(args, torch, dist, el, stream, local, rank, world_size, barrier, max_over_ranks, fp64_peak):
    """BASELINE configs[3] and configs[4] on the N GPUs of this run (also at N = 1, so the scaling run has a base)."""
    from elodin_b200.executor import WORLD_POS
    from elodin_b200.sharding import Comm, shard_sizes, shard_worlds

    out = {}
    ev = lambda: torch.cuda.Event(enable_timing=True)
    distributed = world_size > 1

    def timed(step, ticks, warm):
        with torch.cuda.stream(stream):
            step(warm)
            barrier()
            a, b = ev(), ev()
            a.record(stream)
            step(ticks)
            b.record(stream)
            barrier()
        return max_over_ranks(a.elapsed_time(b))

    # ---- configs[3]: n-body, 1024 bodies, softened all-pairs gravity + 6DOF (SURVEY §8d C4)
    N = 1024
    rng = np.random.default_rng(7)  # the same world(s) on every rank where a single world is replicated

    def nbody_world(Mw, gen, n=N):
        p = np.zeros((Mw, n, 7)); p[..., 3] = 1.0; p[..., 4:] = gen.uniform(-30, 30, (Mw, n, 3))
        v = np.zeros((Mw, n, 6)); v[..., 3:] = gen.normal(0, 1e-7, (Mw, n, 3))
        m = 10 ** gen.uniform(-10, -3, (Mw, n)); m[:, 0] = 1.0
        I = np.zeros((Mw, n, 7)); I[..., :3] = m[..., None]; I[..., 6] = m
        return p, v, I

    grav = lambda n=N: el.GravityEdges("softened", k_squared=2.9591220828e-4 / 86400.0 ** 2, softening=1e-10, edges=el.all_pairs_edges(n))
    FLOP_PAIR, SLOT_PAIR = 27.0, 18.0  # per pair evaluation: flops (FMA = 2) / FP64-pipe instruction slots (DESIGN.md §5)
    # (a) worlds sharded: M = 8 worlds per GPU (weak scaling), no collective; and a batch that fills every SM with whole
    # worlds (2 per SM), where the fixed per-tick costs no longer matter
    def nbody_batch(Mw, ticks, warm):
        p, v, I = nbody_world(Mw, np.random.default_rng(100 + rank))
        ex = el.B200Exec(N, Mw, 3600.0, None, [grav()], "rk4", "fast", device=local)
        ex.set_stream(stream.cuda_stream)
        ex.set_state(p, v, I)
        ms = timed(ex.step, ticks, warm)
        ex.close()
        pair_rate = 3.0 * N * (N - 1) * Mw * world_size * ticks / (ms * 1e-3)
        return {"worlds_per_gpu": Mw, "ticks": ticks, "us_per_tick": ms * 1e3 / ticks, "value": N * Mw * world_size * ticks / (ms * 1e-3),
                "unit": UNIT, "pair_evals_per_s": pair_rate,
                "roofline": {"bound": "fp64", "achieved": pair_rate * FLOP_PAIR / 1e9 / world_size, "peak": fp64_peak, "unit": "GFLOP/s",
                             "frac": pair_rate * FLOP_PAIR / 1e9 / world_size / fp64_peak if fp64_peak else None,
                             "pipe_frac": pair_rate * SLOT_PAIR / world_size / (fp64_peak * 1e9 / 2.0) if fp64_peak else None}}

    small = nbody_batch(8, 200, 10)
    small["roofline"].update({
        "peak_source": "b200_probe_fp64_gflops (dependent-free DFMA chains), this run, per GPU",
        "flops_per_pair_eval": FLOP_PAIR, "fp64_slots_per_pair_eval": SLOT_PAIR, "kernel": "graph_dense_world_kernel<RK4, 1024, 512 x 1, 2 sources x 2 targets>",
        "note": "3 N (N-1) pair evaluations per world-tick (three distinct stage positions); pipe_frac = FP64-pipe instruction slots "
                "of the pair arithmetic / the DFMA issue rate (a non-fused op takes a whole slot); the tick also holds the body "
                "launch and, at 8 worlds, 5.3 rounds of work items quantised to 6"})
    out["nbody_1024_sharded_worlds"] = {
        "config": "BASELINE configs[3]: 1024 bodies, softened all-pairs gravity + 6DOF RK4, dt = 3600 s, 8 worlds per GPU", "scaling": "weak",
        **small, "saturated_batch": nbody_batch(296, 30, 3)}
    # (b) ONE world on N GPUs: replicas (every GPU integrates the whole world, zero communication) ...
    p1, v1, I1 = nbody_world(1, rng)
    ex = el.B200Exec(N, 1, 3600.0, None, [grav()], "rk4", "fast", device=local)
    ex.set_stream(stream.cuda_stream)
    ex.set_state(p1, v1, I1)
    ms_rep = timed(ex.step, 400, 20)
    ref_pos = ex.download(WORLD_POS)
    ex.close()
    single = {"config": "BASELINE configs[3], M = 1: one 1024-body world on N GPUs",
              "replicas": {"us_per_tick": ms_rep * 1e3 / 400, "value": N * 400 / (ms_rep * 1e-3), "unit": UNIT,
                           "note": "every GPU integrates the whole world; no communication; value counts the world once"}}
    # ... vs row shards (each GPU folds N / n_gpus sources, stage positions exchanged through NVLink peer memory)
    single["row_shards"] = run_row_shards(args, torch, dist, el, stream, local, rank, world_size, barrier, max_over_ranks,
                                          (p1, v1, I1), grav, ref_pos)
    out["nbody_1024_single_world"] = single
    # the same comparison for a world large enough that the pair folds, not the per-tick latency, dominate
    NL = 8192
    pl, vl, Il = nbody_world(1, np.random.default_rng(11), NL)
    ex = el.B200Exec(NL, 1, 3600.0, None, [grav(NL)], "rk4", "fast", device=local)
    ex.set_stream(stream.cuda_stream)
    ex.set_state(pl, vl, Il)
    ms_big = timed(ex.step, 40, 5)
    ref_big = ex.download(WORLD_POS)
    ex.close()
    big = {"config": "one 8192-body world on N GPUs (beyond BASELINE: where row shards start to pay)",
           "replicas": {"us_per_tick": ms_big * 1e3 / 40, "value": NL * 40 / (ms_big * 1e-3), "unit": UNIT}}
    if world_size > 1:
        try:
            from elodin_b200.sharding import RowShardedWorld

            big["row_shards"] = RowShardedWorld.bench_large(torch, dist, el, stream, local, rank, world_size, barrier, max_over_ranks,
                                                            (pl, vl, Il), grav, ref_big, 5, 40)
        except Exception as e:  # the comparison is secondary: never lose the line over it
            big["row_shards"] = {"error": repr(e)[:200]}
    else:
        big["row_shards"] = {"skipped": "needs more than one GPU"}
    out["nbody_8192_single_world"] = big

    # ---- configs[4]: falcon9-style Monte-Carlo, 100 000 rollouts over the N GPUs (strong scaling: total work fixed)
    TOTAL = args.mc_rollouts
    w0, w1 = shard_worlds(TOTAL, rank, world_size)
    Ml = w1 - w0
    gen = np.random.default_rng(20170814 + rank)
    pos = np.tile(np.array([0, 0, 0, 1.0, 6.4e6, 0, 0]), (Ml, 1, 1)) + np.concatenate([np.zeros((Ml, 1, 4)), gen.normal(0, 10, (Ml, 1, 3))], -1)
    vel = np.concatenate([gen.normal(0, 0.01, (Ml, 1, 3)), gen.normal(0, 50, (Ml, 1, 3))], -1)
    ine = np.tile(np.array([4e6, 4e6, 1e5, 0, 0, 0, 3e4]), (Ml, 1, 1))
    steps, every = args.mc_steps, max(args.mc_steps // 50, 1)
    ex = el.B200Exec(1, Ml, 1e-3, None, [el.GravityFrame(), el.WrenchBody("body_wrench", "linear_first")], "rk4", "fast", device=local,
                     max_fused_ticks=100, trajectory_every=every, trajectory_capacity=steps // every)
    ex.set_stream(stream.cuda_stream)
    ex.set_state(pos, vel, ine, body_wrench=gen.normal(0, 1e4, (Ml, 1, 6)))
    ex.step(100)  # warm (kernel image, clocks); the ring restarts below
    ex.sync()
    ex.trajectory_reset()
    with torch.cuda.stream(stream):
        barrier()
        a, b = ev(), ev()
        a.record(stream)
        ex.step(steps)
        b.record(stream)
        barrier()
    ms_steps = max_over_ranks(a.elapsed_time(b))
    # end-of-run gather of the trajectory ring inside the library (NCCL over NVLink), every rank gets every world
    uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
    if rank == 0:
        uid = torch.tensor(list(Comm.unique_id()), dtype=torch.uint8, device="cuda")
    if distributed:
        dist.broadcast(uid, 0)
    comm = Comm(bytes(uid.cpu().tolist()), world_size, rank, local)
    sizes = shard_sizes(TOTAL, world_size)
    n_s, Wt = ex.trajectory_len(), ex.trajectory_width()
    full = torch.empty((TOTAL, n_s, 1, Wt), device="cuda", dtype=torch.float64)
    gms = []
    for i in range(7):  # 2 warm-ups at full size (NCCL builds its channels on first use), 5 timed
        barrier()
        comm.trajectory_allgather(ex, sizes, out_ptr=full.data_ptr())
        if i >= 2:
            gms.append(max_over_ranks(comm.last_ms))
    g_ms = float(np.median(gms))
    recv_bytes = full.numel() * 8 * (world_size - 1) / world_size  # what one GPU receives over NVLink
    # integrity of the gathered array: rank r's first world sits at offset sum(sizes[:r]) with its own sample 0
    own = ex.trajectory()[:, 0, 0, :]
    got = full[w0, :, 0, :].cpu().numpy() if Ml else own
    gather_ok = bool(np.array_equal(own, got))
    ex.close()
    comm.close()
    out["falcon9_mc_rollouts"] = {
        "config": f"BASELINE configs[4]: falcon9-style worlds (rotating-frame gravity + body wrench), {TOTAL} rollouts sharded over "
                  f"{world_size} GPU(s), dt = 1e-3, {steps} steps, trajectory sample every {every} ticks",
        "rollouts_total": TOTAL, "rollouts_per_gpu": sizes, "steps": steps, "scaling": "strong",
        "seconds_steps": ms_steps * 1e-3, "seconds_gather": g_ms * 1e-3, "seconds_total": (ms_steps + g_ms) * 1e-3,
        "value": TOTAL * steps / ((ms_steps + g_ms) * 1e-3), "value_steps_only": TOTAL * steps / (ms_steps * 1e-3), "unit": UNIT,
        "gather": {"collective": "b200_sixdof_trajectory_allgather: layout kernel + ncclAllGather (ragged: grouped ncclBroadcast) "
                                 "inside libb200_sixdof.so, device-timed on the handle's stream",
                   "nccl_version": int(__import__("elodin_b200")._lib.lib().b200_comm_version()),
                   "bytes_result_per_gpu": int(full.numel() * 8), "bytes_received_per_gpu": int(recv_bytes),
                   "ms_median_of_5": g_ms, "ms_all": gms, "recv_GBps_per_gpu": recv_bytes / (g_ms * 1e-3) / 1e9 if world_size > 1 else None,
                   "nvlink5_peak_GBps_per_direction": 900.0,
                   "frac_of_nvlink_peak": recv_bytes / (g_ms * 1e-3) / 1e9 / 900.0 if world_size > 1 else None,
                   "result_checked": gather_ok}}
    return out


def run_row_shards(args, torch, dist, el, stream, local, rank, world_size, barrier, max_over_ranks, world, grav, ref_pos):
    """One 1024-body world split by source rows over the GPUs of the node (SURVEY §8e: "report both")."""
    if world_size == 1:
        return {"skipped": "needs more than one GPU"}
    try:
        from elodin_b200.sharding import RowShardedWorld
    except ImportError:
        return {"skipped": "row sharding is not built in this version"}
    return RowShardedWorld.bench(args, torch, dist, el, stream, local, rank, world_size, barrier, max_over_ranks, world, grav, ref_pos)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--worlds", type=int, default=1 << 22, help="worlds per GPU (1 body each)")
    ap.add_argument("--fuse", type=int, default=25, help="ticks per launch of the fused / e2e runs")
    ap.add_argument("--e2e-ticks", type=int, default=100, help="ticks per invoke_batch call (ticks_per_telemetry)")
    ap.add_argument("--e2e-worlds", type=int, default=1 << 20)
    ap.add_argument("--e2e-calls", type=int, default=5)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--mc-rollouts", type=int, default=100000, help="configs[4]: Monte-Carlo rollouts over all GPUs")
    ap.add_argument("--mc-steps", type=int, default=1000, help="configs[4]: ticks per rollout (dt = 1e-3)")
    ap.add_argument("--configs", action="store_true", help="also time the other BASELINE.json configs (adds ~1 min)")
    ap.add_argument("--kernel-only", action="store_true", help="profiling aid: only the main timed loop (no e2e / cpu / extras)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the timed executor's final state columns (a fixed sample of "
                                                            f"{DUMP_WORLDS} worlds) to DIR/<column>.npy")
    args = ap.parse_args()
    if args.impl == "reference":
        if args.dump_outputs:
            ap.error("--dump-outputs writes the state of the B200 executor: it needs --impl b200")
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
