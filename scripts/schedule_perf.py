"""Input schedules against plain columns and host systems, on one GPU.

    python scripts/schedule_perf.py [--out profiles/r04_input_schedules.txt] [--rounds 3] [--baseline-tree DIR]

Arms (each pair / triple alternated `--rounds` times in this one process; the card's name and power limit are
read in the same call and written at the top of the report):
  A  rocket set (gravity + thrust + per-body drag), 2^22 worlds, FAST, one tick per launch: thrust scheduled per
     world against a plain thrust column (same instantiation, same bytes per tick);
  B  configs[2] shape (10^4 worlds, 100 fused ticks per launch, 5000 ticks), FAST and EXACT: a scheduled thrust curve
     against the plain column and against the same curve forced to one tick per launch;
  C  the one-body rocket ECS sim, 1200 ticks at 120 Hz: wall time per tick, host_system against input_schedule;
  D  the rocket golden telemetry replayed in one EXACT step(100) with the recorded thrust / aero_force as schedules:
     the largest deviation from the recorded rows (the reference gates them at 1e-4);
  E  with --baseline-tree: the headline bench.py line of that tree and of this one, alternated.
"""

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import elodin_b200 as el  # noqa: E402

LINES = []


def log(s=""):
    print(s, flush=True)
    LINES.append(s)


def timed_step(ex, ticks, warm):
    ex.step(warm, sync=True)
    t0 = time.perf_counter()
    ex.step(ticks, sync=True)
    return (time.perf_counter() - t0) * 1e6 / ticks  # us per tick


def rocket_exec(M, math, fused, rng):
    q = el.Quaternion.from_euler([0.0, np.radians(70.0), 0.0]).arr
    pos = np.tile(np.concatenate([q, [0, 0, 1.0]]), (M, 1, 1))
    vel = np.zeros((M, 1, 6))
    ine = np.tile(np.array([0.1, 1.0, 1.0, 0, 0, 0, 3.0]), (M, 1, 1))
    effs = [el.GravityConst((0, 0, -9.81)), el.ThrustBody((-1.0, 0, 0), "thrust"), el.DragQuadratic(column="wind", per_body_params=True)]
    drag = np.concatenate([rng.normal(0, 1, (M, 1, 3)), rng.uniform(0.3, 0.9, (M, 1, 1)), rng.uniform(1e-3, 1e-2, (M, 1, 1))], -1)
    ex = el.B200Exec(1, M, 0.008333333, None, effs, "rk4", math, max_fused_ticks=fused)
    ex.set_state(pos, vel, ine, thrust=np.full((M, 1, 1), 88.426), wind=drag)
    return ex


def arm_a(rounds):
    M, ticks, T = 1 << 22, 200, 8
    rng = np.random.default_rng(1)
    log(f"A  rocket set (gravity + thrust + per-body drag), {M} worlds, FAST RK4, one tick per launch, {ticks} ticks timed")
    plain = rocket_exec(M, "fast", 1, rng)
    sched = rocket_exec(M, "fast", 1, rng)
    sched.set_schedule("thrust", rng.uniform(50, 120, (T, M, 1, 1)), 0)
    res = {"plain": [], "scheduled": []}
    for r in range(rounds):
        for name, ex in (("plain", plain), ("scheduled", sched)):
            res[name].append(timed_step(ex, ticks, 10))
    for name, v in res.items():
        log(f"   {name:10s} us/tick: " + "  ".join(f"{x:8.2f}" for x in v) + f"   median {np.median(v):8.2f}")
    plain.close(); sched.close()
    return res


def arm_b(rounds):
    M, ticks = 10000, 5000
    rng = np.random.default_rng(2)
    curve = 88.426 * np.exp(-np.arange(ticks) / 2000.0)
    rows = np.broadcast_to(curve[:, None, None, None], (ticks, M, 1, 1))
    out = {}
    for math in ("fast", "exact"):
        log(f"B  configs[2] shape: {M} worlds, {math.upper()} RK4, {ticks} ticks, thrust curve of {ticks} rows")
        arms = {"plain_fused100": rocket_exec(M, math, 100, rng), "scheduled_fused100": rocket_exec(M, math, 100, rng),
                "scheduled_1_per_launch": rocket_exec(M, math, 1, rng)}
        for k in ("scheduled_fused100", "scheduled_1_per_launch"):
            arms[k].set_schedule("thrust", rows, 0)
        for ex in arms.values():  # module loads and first launches stay out of the timed rounds
            ex.step(100, sync=True)
        res = {k: [] for k in arms}
        for r in range(rounds):
            for k, ex in arms.items():
                ex.trajectory_reset()
                ex.upload("tick", np.array([0], dtype=np.uint64))
                res[k].append(timed_step(ex, ticks, 0) * ticks * 1e-3)  # ms per 5000 ticks
        for k, v in res.items():
            log(f"   {k:24s} ms/{ticks} ticks: " + "  ".join(f"{x:8.2f}" for x in v) + f"   median {np.median(v):8.2f}")
        for ex in arms.values():
            ex.close()
        out[math] = res
    return out


def rocket_world():
    Thrust = el.Annotated[np.ndarray, el.Component("thrust", el.ComponentType.F64)]

    @el.dataclass
    class Motor(el.Archetype):
        thrust: Thrust

    w = el.World()
    q = el.Quaternion.from_euler([0.0, np.radians(70.0), 0.0])
    w.spawn([el.Body(world_pos=el.SpatialTransform(angular=q, linear=np.array([0.0, 0.0, 1.0])),
                     inertia=el.SpatialInertia(3.0, np.array([0.1, 1.0, 1.0]))), Motor(np.array([0.0]))], name="rocket")
    return w


def arm_c(rounds):
    ticks = 1200
    curve = lambda k: 300.0 * np.exp(-0.05 * k)

    @el.host_system
    def thrust(ctx):
        ctx.column("thrust")[...] = curve(ctx.tick)

    effs = el.GravityConst((0.0, 0.0, -9.81)) | el.ThrustBody((-1.0, 0.0, 0.0), "thrust")
    table = np.array([[curve(k)] for k in range(ticks)])
    log(f"C  one-body rocket ECS sim, {ticks} ticks at 120 Hz, EXACT: wall time per tick (build excluded)")
    res = {"host_system": [], "input_schedule": []}
    same = True
    for r in range(rounds):
        hist = {}
        for name in res:
            system = (thrust if name == "host_system" else el.input_schedule("thrust", table)) | el.six_dof(sys=effs)
            ex = rocket_world().build(system, simulation_rate=120.0)
            t0 = time.perf_counter()
            ex.run(ticks)
            res[name].append((time.perf_counter() - t0) * 1e6 / ticks)
            hist[name] = ex.history(["rocket.world_pos", "rocket.world_vel"])
        same &= all(np.array_equal(np.asarray(hist["host_system"][k]), np.asarray(hist["input_schedule"][k])) for k in hist["host_system"])
    for name, v in res.items():
        log(f"   {name:15s} us/tick: " + "  ".join(f"{x:8.2f}" for x in v) + f"   median {np.median(v):8.2f}")
    log(f"   history rows identical between the two: {same}")
    return res


def arm_d():
    g = np.load(os.path.join(ROOT, "tests", "golden", "elodin_ci_baseline.npz"))
    dt = float(g["rocket.simulation_time_step"][0, 0])
    effs = [el.GravityConst((0.0, 0.0, -9.81)), el.ThrustBody((-1.0, 0.0, 0.0), "thrust"), el.WrenchBody("aero_force")]
    with el.B200Exec(1, 1, dt, None, effs, "rk4", "exact", max_fused_ticks=100, trajectory_every=1, trajectory_capacity=100,
                     trajectory_full=True) as ex:
        ex.set_state(*(g[f"rocket.{c}"][0][None, None] for c in ("world_pos", "world_vel", "inertia")),
                     accel=g["rocket.world_accel"][0][None, None])
        ex.set_schedule("thrust", g["rocket.thrust"][1:101].reshape(100, 1, 1, 1))
        ex.set_schedule("aero_force", g["rocket.aero_force"][1:101].reshape(100, 1, 1, 6))
        ex.step(100, sync=True)
        traj = ex.trajectory()[:, 0, 0]
    log("D  rocket golden telemetry, 100 ticks in one EXACT step, recorded thrust / aero_force rows 1..100 as schedules")
    for name, lo, hi in (("world_pos", 0, 7), ("world_vel", 7, 13), ("world_accel", 13, 19), ("force", 19, 25)):
        ref = g[f"rocket.{name}"][1:101]
        dev = np.abs(traj[:, lo:hi] - ref)
        rel = dev / np.maximum(np.abs(ref), 1e-300)
        log(f"   {name:12s} max |dev| {dev.max():.3e}   max rel dev (nonzero refs) {rel[np.abs(ref) > 0].max():.3e}")


def arm_e(rounds, base):
    cmd = ["--gpus", "1", "--steps", "2000", "--warmup", "5"]
    log(f"E  headline bench.py {' '.join(cmd)}: parent tree ({base}) vs this tree, alternated")
    res = {"parent": [], "this": []}
    for r in range(rounds):
        for name, tree in (("parent", base), ("this", ROOT)):
            p = subprocess.run([sys.executable, os.path.join(tree, "bench.py"), *cmd], capture_output=True, text=True, cwd=tree)
            line = [ln for ln in p.stdout.splitlines() if ln.startswith("{")]
            if p.returncode or not line:
                log(f"   {name}: bench.py failed (rc {p.returncode}): {p.stderr[-400:]}")
                continue
            j = json.loads(line[-1])
            res[name].append(j.get("value"))
            log(f"   {name:7s} round {r}: value {j.get('value'):.4e} {j.get('unit', '')}")
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r04_input_schedules.txt"))
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--baseline-tree", default=None)
    ap.add_argument("--arms", default="ABCDE")
    args = ap.parse_args()
    if el.device_count() < 1:
        raise SystemExit("schedule_perf.py measures on a CUDA device; none is visible")
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    log(f"GPU: {smi[0] if smi else 'unknown'} (name, power limit, max SM clock)")
    log(f"rounds: {args.rounds}, arms alternated within each round")
    log()
    if "A" in args.arms:
        arm_a(args.rounds); log()
    if "B" in args.arms:
        arm_b(args.rounds); log()
    if "C" in args.arms:
        arm_c(args.rounds); log()
    if "D" in args.arms:
        arm_d(); log()
    if "E" in args.arms and args.baseline_tree:
        arm_e(args.rounds, os.path.abspath(args.baseline_tree)); log()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        f.write("\n".join(LINES) + "\n")


if __name__ == "__main__":
    main()
