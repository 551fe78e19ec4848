"""Developer: step time of the multi-robot DWA controller (DWAFleet) against the batched sweep
(kc_planner_batch_cloud) on matched inputs and against one DWA handle per robot.

    python tools/fleet_dev.py [--robots 1024] [--warmup 50] [--steps 500] [--out profiles/fleet_b200.json]

Robots are C2-shaped (tests/workloads.py cfg_c2, ~10k velocity slots, P = 50), each with its own cloud
(the sweep's distribution, seed 5000 + robot id, 100k points, page-locked) and its own velocity. Three
fleets of the same robots and clouds:
  own paths  every robot on its own path through its position: lines at varied headings and offsets,
             and circles of radius 0.5 - 3 m (`distinct_P` lists the horizons the step ran with)
  one path   every robot on the same straight path, as kc_planner_batch_cloud needs
  sweep      kc_planner_batch_cloud on that path and tracked segment, same clouds, poses, velocities
The one-path fleet and the sweep alternate step by step in the same loop. Then one
DWA.compute_velocity_commands per robot on independent handles, one after the other."""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import __graft_entry__ as ge  # noqa: E402
import workloads as wl  # noqa: E402

DISTRIBUTION = "dense_cluster_on_path"  # bench.py's sweep headline
N_POINTS = 100_000


def pct(a, q):
    return float(np.percentile(np.asarray(a) * 1e3, q))


def stats(t):
    return {"p50_ms": pct(t, 50), "p90_ms": pct(t, 90), "p99_ms": pct(t, 99), "mean_ms": float(np.mean(t) * 1e3)}


def own_path(r, rng):
    """A path through the origin: a 20 m line (heading, start offset) or a circle of radius 0.5 - 3 m."""
    if r % 3 == 2:
        rad, phi = float(rng.uniform(0.5, 3.0)), float(rng.uniform(-math.pi, math.pi))
        cx, cy = rad * math.cos(phi), rad * math.sin(phi)
        a0 = phi + math.pi  # the origin's angle on the circle, then counter-clockwise
        pts = [(cx + rad * math.cos(a0 + t), cy + rad * math.sin(a0 + t)) for t in np.linspace(0, 1.8 * math.pi, 60)]
        pts[0] = (0.0, 0.0)
        return pts, a0 + math.pi / 2
    h, back = float(rng.uniform(-math.pi, math.pi)), float(rng.uniform(0.0, 5.0))
    return [(-back * math.cos(h), -back * math.sin(h)), ((20 - back) * math.cos(h), (20 - back) * math.sin(h))], h


def batch_split(fn, n):
    """planner-side host split of n fleet / sweep calls (KC_BATCH_TIMING lines on stderr)"""
    os.environ["KC_BATCH_TIMING"] = "1"
    fd = os.dup(2)
    with tempfile.TemporaryFile(mode="w+") as f:
        os.dup2(f.fileno(), 2)
        try:
            wall = []
            for _ in range(n):
                t0 = time.perf_counter()
                fn()
                wall.append(time.perf_counter() - t0)
        finally:
            os.dup2(fd, 2)
            os.close(fd)
            del os.environ["KC_BATCH_TIMING"]
        f.seek(0)
        rows = [line for line in f.read().splitlines() if line.startswith("[kc batch]")]
    prep = [float(x.split("host prep ")[1].split(" ms")[0]) for x in rows]
    enq = [float(x.split("enqueue ")[1].split(" ms")[0]) for x in rows]
    wait = [float(x.split("wait+fetch ")[1].split(" ms")[0]) for x in rows]
    call = 1e3 * float(np.median(wall))
    inner = float(np.median(prep) + np.median(enq) + np.median(wait))
    return {"call_p50_ms": call, "ctx_prep_ms": float(np.median(prep)), "enqueue_ms": float(np.median(enq)),
            "wait_and_gather_ms": float(np.median(wait)),
            "outside_planner_ms": call - inner}  # follower steps, result fill, Python


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--robots", type=int, default=1024)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--steps", type=int, default=500)
    ap.add_argument("--sequential", type=int, default=-1, help="robots of the sequential-handle leg (-1: all)")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "fleet_b200.json"))
    a = ap.parse_args()
    pkg = ge.load_package()
    smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    R = a.robots
    gen, w = wl.CLOUD_FAMILY[DISTRIBUTION]
    kw = wl.cfg_c2() if w is None else wl.cfg_c2(weights=w)
    cfg = pkg.planner_config(**kw)
    host = pkg.PinnedArray((R * N_POINTS, 3), np.float32)
    vels, paths, yaws = [], [], []
    prng = np.random.default_rng(wl.SEED + 4242)
    for r in range(R):
        rng = np.random.default_rng(wl.SEED + 7 * r)  # bench.py's sweep velocities
        vels.append((float(rng.uniform(0.0, 2.0)), 0.0, float(rng.uniform(-2.0, 2.0))))
        host.array[r * N_POINTS:(r + 1) * N_POINTS] = gen(5000 + r, n=N_POINTS)
        p, yaw = own_path(r, prng)
        paths.append(p)
        yaws.append(yaw)
    offsets = np.arange(R, dtype=np.int64) * N_POINTS
    counts = np.full(R, N_POINTS, np.int32)
    clouds = (host.array, offsets, counts)
    vels = np.asarray(vels)

    own = pkg.DWAFleet(cfg, n_robots=R)
    for r in range(R):
        own.set_current_path(r, paths[r])
    own.set_current_states([(0.0, 0.0, yaws[r], 0.0) for r in range(R)])
    one = pkg.DWAFleet(cfg, n_robots=R)
    line = wl.straight_points(20.0)
    for r in range(R):
        one.set_current_path(r, line)
    poses = np.zeros((R, 3))
    poses[:, 2] = np.random.default_rng(wl.SEED + 4343).uniform(-0.5, 0.5, R)
    one.set_current_states(np.concatenate([poses, np.zeros((R, 1))], axis=1))
    info0 = one.compute_velocity_commands(vels, clouds=clouds)["info"]
    seg = (int(info0.seg_start[0]), int(info0.seg_count[0]))
    assert (info0.seg_start == seg[0]).all() and (info0.seg_count == seg[1]).all()
    path = pkg.path_prepare(line)
    pl = pkg.Planner(cfg)
    pl.set_path(path["X"], path["Y"], path["acc"], path["total_length"])

    for _ in range(a.warmup):
        own.compute_velocity_commands(vels, clouds=clouds)
        one.compute_velocity_commands(vels, clouds=clouds)
        pl.batch_cloud(vels, poses, host.array, seg[0], seg[1], offsets=offsets, counts=counts)
    t_own, t_one, t_sweep = [], [], []
    for _ in range(a.steps):
        t0 = time.perf_counter()
        out_own = own.compute_velocity_commands(vels, clouds=clouds)
        t_own.append(time.perf_counter() - t0)
    for _ in range(a.steps):
        t0 = time.perf_counter()
        out_one = one.compute_velocity_commands(vels, clouds=clouds)
        t_one.append(time.perf_counter() - t0)
        t0 = time.perf_counter()
        sweep = pl.batch_cloud(vels, poses, host.array, seg[0], seg[1], offsets=offsets, counts=counts)
        t_sweep.append(time.perf_counter() - t0)
    same_as_sweep = [s[2] for s in sweep] == out_one["slot"].tolist()  # matched inputs: the same winners
    split_n = min(50, a.steps)
    splits = {"own_paths": batch_split(lambda: own.compute_velocity_commands(vels, clouds=clouds), split_n),
              "one_path": batch_split(lambda: one.compute_velocity_commands(vels, clouds=clouds), split_n),
              "sweep": batch_split(lambda: pl.batch_cloud(vels, poses, host.array, seg[0], seg[1], offsets=offsets,
                                                          counts=counts), split_n)}
    n_points = out_own["n_points"]
    own.close()
    one.close()
    pl.close()

    # one DWA handle per robot, one step each (after one untimed step), one after the other
    S = R if a.sequential < 0 else min(a.sequential, R)
    dwas = []
    for r in range(S):
        d = pkg.DWA(cfg)
        d.set_current_path(paths[r])
        d.set_current_state(0.0, 0.0, yaws[r])
        dwas.append(d)
    views = [host.array[r * N_POINTS:(r + 1) * N_POINTS] for r in range(S)]
    for r in range(S):
        dwas[r].compute_velocity_commands(vels[r], cloud=views[r])
    t0 = time.perf_counter()
    seq = [dwas[r].compute_velocity_commands(vels[r], cloud=views[r]) for r in range(S)]
    t_seq = time.perf_counter() - t0
    same_as_fleet = [s.slot for s in seq] == out_own["slot"][:S].tolist()
    for d in dwas:
        d.close()
    host.free()

    rec = {
        "device": smi, "robots": R, "points_per_cloud": N_POINTS, "distribution": DISTRIBUTION,
        "config": "tests/workloads.py cfg_c2 (%d velocity slots, P = %d)" % (int(np.median(out_one["n_slots"])),
                                                                              int(out_one["n_points"][0])),
        "warmup_steps": a.warmup, "timed_steps": a.steps, "input": "page-locked clouds (PinnedArray), flat layout",
        "fleet_own_paths": dict(stats(t_own), distinct_P=sorted(set(n_points.tolist())),
                                robots_with_a_trajectory=int(out_own["found"].sum())),
        "fleet_one_path": dict(stats(t_one), robots_with_a_trajectory=int(out_one["found"].sum())),
        "batch_cloud_one_path": stats(t_sweep),
        "fleet_one_path_over_batch_cloud_p50": pct(t_one, 50) / pct(t_sweep, 50),
        "fleet_one_path_winners_equal_batch_cloud": same_as_sweep,
        "host_split_ms": splits,
        "sequential_dwa_handles": {"robots": S, "total_ms": t_seq * 1e3, "per_robot_ms": t_seq * 1e3 / S,
                                   "winners_equal_fleet_own_paths": same_as_fleet},
        "fleet_own_paths_speedup_over_sequential_handles": (t_seq * R / S) / (pct(t_own, 50) * 1e-3),
    }
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec))


if __name__ == "__main__":
    main()
