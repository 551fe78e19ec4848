#!/usr/bin/env python
"""bench.py — driver contract for the B200-native DWA hot path.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload cycle|sweep]
                    [--dump-outputs DIR]

A "step" is one DWA control cycle of one robot on BASELINE.json configs[1]: differential drive,
9 900 velocity slots x 50 points (dt 0.02 s, 1 s horizon) against a 100 000-point synthetic cloud,
all five cost weights = 1. Unit of work: trajectory-steps = slots x points per cycle.

The pruned pipeline is data dependent (the reference's brute force is not), so the cycle is measured
over a FAMILY of cloud distributions (tests/workloads.py CLOUD_FAMILY: SURVEY 8d's own C2 cloud,
clutter inside reach, pillars, a dense cluster on the path, the all-ties case, an empty cloud, and
round 1's friendly ring); the headline (`value`, `e2e`, `ms_per_step`) is the distribution named in
config.distribution = the worst one, and e2e.by_distribution carries p50/p90/p99 of every member.

  value  device-resident throughput: K cycles enqueued back to back on the planner's stream, cycle i
         reading cloud (i mod 128) of a bank of 128 cloud slots (154 MB > the 126 MB L2, so every
         cycle reads its cloud cold from HBM); CUDA events on that stream; max over ranks.
  e2e    the same metric through the public call kc_planner_cycle_cloud with HOST buffers (page-locked):
         per step the 1.2 MB cloud travels host->device and the winner record comes back; wall clock
         over max(K, 1000) calls, with p50/p90/p99 of the per-call latency.
  N > 1  weak scaling: each rank (one process per GPU, torchrun) plans for its own robot / clouds;
         no data-path collective (robots are independent, north_star); barrier + max over ranks.
         roofline.sweep carries the STRONG-scaled 1024-robot sweep (north_star config 5) of the same
         run; `--workload sweep` makes that sweep the headline (value, "scaling": "strong").
  --impl reference   the CPU restatement of the reference path (oracle/, or oracle/_ref when the
         reference's own sources were compiled) with all host threads on the same config.
  --dump-outputs DIR   after the timed steps, rank 0 writes what the headline's timed path returned in
         its last step. Cycle: the winner record of the LAST timed cycle as the public call returns it,
         DIR/winner.npy (float64: found, cost, slot, n_admissible, n_slots, n_points) and
         DIR/trajectory_{vx,vy,omega,x,y}.npy (float32 rows of the winning trajectory). Sweep
         (--workload sweep): DIR/sweep_winners.npy, float64 [robots, 4] = found, cost, slot,
         n_admissible of every robot in the last timed replay, gathered in robot order. The clouds are
         seeded, so two builds run with the same arguments can be compared output for output.
"""
import argparse
import json
import math
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "dwa_trajectory_steps_per_s"
UNIT = "trajectory-steps/s"
N_POINTS_CLOUD = 100_000
BANK = 128       # 128 x 1.2 MB = 154 MB > 126 MB L2
DISTINCT = 8     # distinct clouds per distribution (the bank cycles them over its 128 slots)
N_LAT = 1000     # latency samples per distribution, regardless of --steps
# The member of the cloud family the headline is quoted on: the worst p99 of the family as measured on
# B200 (profiles/r2_family.json); e2e.by_distribution shows every member of the same run.
HEADLINE = os.environ.get("KC_BENCH_DISTRIBUTION", "dense_cluster_on_path")
SWEEP_ROBOTS = 1024

_REAL_STDOUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout. Libraries (NCCL prints its version banner to stdout)
    must not add lines: keep a private handle of the real stdout and point fd 1 at stderr."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line):
    out = _REAL_STDOUT if _REAL_STDOUT is not None else sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def config_dict(workload="cycle"):
    """The workload both arms run — identical dict from `--impl ours` and `--impl reference`."""
    import workloads as wl

    kw = wl.cfg_c2()
    n_slots, P = 9900, 50
    cfg = {
        "workload": "configs[1]: DWA differential-drive, 9900 velocity slots (101 x 101 grid minus the "
                    "|vx| < 0.01 row) x 50 points vs 100000-point cloud, all five cost weights = 1, "
                    "cylinder r=0.2 h=0.4 robot, octree 0.1 m, current velocity (1, 0, 0), pose origin, "
                    "20 m straight reference path interpolated at 0.01 m",
        "slots": n_slots, "points_per_trajectory": P, "cloud_points": N_POINTS_CLOUD,
        "distribution": HEADLINE,
        "cloud_family": list(wl.CLOUD_FAMILY),
        "cloud_seed": "numpy default_rng(20261018 + offset + 1000 * rank + i), i = cloud index",
        "l2_policy": "inputs larger than L2: bank of %d cloud slots (%.0f MB) cycled" %
                     (BANK, BANK * N_POINTS_CLOUD * 12 / 1e6),
        "robots_per_gpu": 1,
        "sweep": "%d independent robots (own cloud seed, own current velocity), sharded by robot" % SWEEP_ROBOTS,
    }
    if workload == "sweep":
        cfg["workload"] = ("configs[4]: batched sweep of %d independent robots, each = " % SWEEP_ROBOTS) + cfg["workload"]
        cfg["robots_per_gpu"] = "%d / n_gpus" % SWEEP_ROBOTS
    del kw
    return cfg


class ProductPath:
    """Interpolated reference path from the product's own kc_path_prepare (Path::interpolate +
    Path::segment on the host) — the repo arm does not touch oracle/ for its inputs."""

    def __init__(self, pkg, pts, interp=0.01, seg_len=1.0):
        d = pkg.path_prepare(pts, True, interp, seg_len)
        self.X, self.Y, self.acc = d["X"], d["Y"], d["acc"]
        self.total_length = d["total_length"]
        self.n = len(self.X)


def make_planner(pkg, kw, path=None):
    p = pkg.Planner(pkg.planner_config(**kw))
    if path is not None:
        p.set_path(path.X, path.Y, path.acc, path.total_length)
    return p


def dist_setup(n_gpus):
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist = None
    if world > 1:
        import torch
        import torch.distributed as dist_mod

        torch.cuda.set_device(local)
        dist_mod.init_process_group(backend="nccl", device_id=torch.device("cuda", local))
        dist = dist_mod
    return world, rank, local, dist


def _is_nccl(dist):
    return dist is not None and dist.get_backend() == "nccl"


def barrier(dist, local):
    if dist is not None:
        if _is_nccl(dist):
            import torch

            dist.barrier(device_ids=[local])
            torch.cuda.synchronize()
        else:
            dist.barrier()


def _reduce(dist, value, local, op):
    if dist is None:
        return value
    import torch

    dev = f"cuda:{local}" if _is_nccl(dist) else "cpu"
    t = torch.tensor([value], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=op)
    return float(t.item())


def max_over_ranks(dist, value, local):
    """MAX over ranks of a per-rank scalar (device time). Works on nccl (GPU box) and gloo (CPU tests)."""
    return _reduce(dist, value, local, dist.ReduceOp.MAX) if dist is not None else value


def sum_over_ranks(dist, value, local):
    return _reduce(dist, value, local, dist.ReduceOp.SUM) if dist is not None else value


def shard_robots(n_robots, world, rank):
    """Contiguous shard of independent robots for this rank: [lo, hi). north_star: the sweep is
    partitioned by robot, no data-path collective."""
    lo = (n_robots * rank) // world
    hi = (n_robots * (rank + 1)) // world
    return lo, hi


def gather_results(dist, local_results, world, rank):
    """Final result gather: rank 0 receives every rank's [(found, cost, slot, n_admissible), ...]
    in robot order (8-16 bytes per robot; the only exchange of the sweep)."""
    if dist is None:
        return list(local_results)
    out = [None] * world if rank == 0 else None
    dist.gather_object(list(local_results), out, dst=0)
    if rank != 0:
        return None
    flat = []
    for part in out:
        flat.extend(part)
    return flat


def pin_to_gpu_numa(local):
    """Bind this rank's threads and future page-locked allocations to the CPU cores / NUMA node of its
    GPU (nvidia-smi topo), so that eight ranks do not share one socket's memory controllers for their
    host->device streams. Best effort: returns a description, never raises."""
    try:
        out = subprocess.run(["nvidia-smi", "topo", "-m"], capture_output=True, text=True, timeout=20).stdout
        hdr = None
        for line in out.splitlines():
            cells = [c.strip() for c in line.split("\t") if c.strip() != ""]
            if not cells:
                continue
            if hdr is None and "CPU Affinity" in line:
                hdr = cells
                continue
            if hdr is not None and cells[0] == f"GPU{local}":
                # columns: GPUn, <links...>, CPU Affinity, NUMA Affinity, ...
                aff_i = hdr.index("CPU Affinity") + 1
                aff = cells[aff_i] if aff_i < len(cells) else ""
                cpus = set()
                for part in aff.split(","):
                    if "-" in part:
                        a, b = part.split("-")
                        cpus.update(range(int(a), int(b) + 1))
                    elif part.strip().isdigit():
                        cpus.add(int(part))
                avail = os.sched_getaffinity(0)
                cpus &= avail
                if cpus:
                    os.sched_setaffinity(0, cpus)
                    return "cpus %s" % aff
                return "topology names no usable cpus (%r)" % aff
        return "no topology row for GPU%d" % local
    except Exception as e:  # noqa: BLE001
        return "unavailable: %r" % (e,)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                       "-lms", "100", "-i", str(gpu_index)], stdout=self.f,
                                      stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        time.sleep(0.12)
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            c = [x.strip() for x in line.split(",")]
            if len(c) < 9:
                continue
            try:
                sm.append(float(c[1]))
                mx.append(float(c[2]))
            except ValueError:
                continue
            for nm, v in zip(names, c[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        os.unlink(self.f.name)
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(np.max(mx)), reasons=sorted(reasons),
                       samples=len(sm))
        return out


def algorithmic_flops(n_adm, n_slots, P, M, S):
    """SURVEY §8(d): brute-force-equivalent FLOPs of one cycle (FMA = 2): what the reference's
    loops execute. Obstacle term N*P*M*6, path N*P*S*8, goal N*S*6, smooth+jerk N*(P-1)*3*7,
    rollout slots*(P-1)*40."""
    return (n_adm * P * M * 6.0 + n_adm * P * S * 8.0 + n_adm * S * 6.0 + n_adm * (P - 1) * 21.0 +
            n_slots * (P - 1) * 40.0)


def pct(a, q):
    return float(np.percentile(a, q) * 1e3)


def dump_cycle_outputs(out_dir, r):
    """--dump-outputs: the winner record `r` (TrajSearchResult) of one cycle, as a caller receives it."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {
        "winner": np.array([r.is_found, r.cost, r.slot, r.n_admissible, r.n_slots, r.n_points], np.float64),
        "trajectory_vx": np.asarray(r.vx, np.float32), "trajectory_vy": np.asarray(r.vy, np.float32),
        "trajectory_omega": np.asarray(r.omega, np.float32),
        "trajectory_x": np.asarray(r.x, np.float32), "trajectory_y": np.asarray(r.y, np.float32),
    }
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def dump_sweep_outputs(out_dir, rows):
    """--dump-outputs, --workload sweep: one (found, cost, slot, n_admissible) row per robot."""
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "sweep_winners.npy"), np.array(rows, np.float64).reshape(-1, 4))


# =================================================================================================
# CPU legs (the only places that touch oracle/): --impl reference and the cpu_baseline subprocess
# =================================================================================================
def oracle_cycle_inputs():
    import orc
    import workloads as wl

    orc.build()
    kw = wl.cfg_c2()
    gen, w = wl.CLOUD_FAMILY[HEADLINE]
    if w is not None:
        kw = wl.cfg_c2(weights=w)
    path = orc.Path(wl.straight_points(20.0), 0.01, 1.0)
    seg = wl.tracked_segment(path, 0, 2.0)
    return orc, wl, kw, path, seg, (1.0, 0.0, 0.0), (0.0, 0.0, 0.0)


def oracle_cycle(orc, kw, path, seg, vel, pose, cloud, threads, max_traj=None):
    """One DWA cycle through the oracle; returns (seconds, n_slots, P, n_admissible, m_evaluated,
    winner). max_traj bounds the cost stage to the first m admissible trajectories (sample)."""
    from parity_util import _split

    common, ccfg = _split(kw)
    scfg = orc.sampler_cfg(max_num_threads=threads, **common)
    D = float(np.float32(kw["max_local_range"]) / np.float32(3.0))
    t0 = time.perf_counter()
    samples = orc.sampler_generate(scfg, vel, pose, cloud=cloud)
    t_s = time.perf_counter() - t0
    n_adm = len(samples["slots"])
    n_slots = len(orc.velocity_samples(scfg, vel)[0])
    P = samples["P"]
    t0 = time.perf_counter()
    obs = orc.cost_points(ccfg, pose, cloud=cloud) if len(cloud) else None
    m = n_adm if max_traj is None else min(n_adm, max_traj)
    sub = samples if m == n_adm else {k: (v[:m] if isinstance(v, np.ndarray) else v) for k, v in samples.items()}
    win = None
    if m > 0:
        found, idx, cost, _ = orc.cost_evaluate(ccfg, sub, path, seg, obs, D, n_threads=threads)
        if found and m == n_adm:
            win = {"slot": int(samples["slots"][idx]), "cost": float(np.float32(cost))}
    t_c = time.perf_counter() - t0
    return t_s, t_c, n_slots, P, n_adm, m, win


def ref_cycle(orc, wl, kw, seg, vel, pose, cloud, threads, max_traj):
    """One cycle through the REFERENCE'S OWN classes (oracle/_ref): sampler with its ThreadPool, cost
    evaluation single-threaded as the reference's CPU CostEvaluator is (cost_evaluator.cpp:49-109)."""
    from parity_util import _split

    common, ccfg = _split(kw)
    return orc.ref_cycle_cloud(orc.sampler_cfg(max_num_threads=threads, **common), ccfg, wl.straight_points(20.0), 0.01,
                               seg, vel, pose, cloud if len(cloud) else np.zeros((0, 3), np.float32),
                               kw["max_local_range"], max_traj=max_traj)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    orc, wl, kw, path, seg, vel, pose = oracle_cycle_inputs()
    gen, _ = wl.CLOUD_FAMILY[HEADLINE]
    threads = os.cpu_count() or 1
    steps, warmup = args.steps, args.warmup
    total_s = float(os.environ.get("KC_BENCH_REF_SECONDS", "150"))  # CPU work of the whole run, roughly
    clouds = [gen(i, n=N_POINTS_CLOUD) if HEADLINE != "empty_cloud" else wl.cloud_empty() for i in range(DISTINCT)]
    budget = total_s / max(steps + warmup, 1)
    use_ref = orc.ref_available() and not os.environ.get("KC_BENCH_REF_PORT")
    # cross-check record (winner of cloud 0) and the all-threads figure of the PORT, which
    # tests/test_oracle_vs_ref.py holds bit-identical to the reference sources
    t_s, t_c, n_slots, P, n_adm0, m, win0 = oracle_cycle(orc, kw, path, seg, vel, pose, clouds[0], threads)
    port_full = t_s + t_c
    vals, tcyc, desc = [], [], ""
    if use_ref:
        kind = "reference"
        cal = ref_cycle(orc, wl, kw, seg, vel, pose, clouds[0], threads, 64)
        per_traj = cal["t_cost"] / max(cal["evaluated"], 1)
        for i in range(warmup + steps):
            c = clouds[i % len(clouds)]
            m = int(max(32, (budget - cal["t_sampler"]) / max(per_traj, 1e-9)))
            r = ref_cycle(orc, wl, kw, seg, vel, pose, c, threads, m)
            t_cycle = r["t_sampler"] + r["t_points"] + r["t_cost"] * (r["n_admissible"] / max(r["evaluated"], 1))
            if i >= warmup:
                vals.append(n_slots * r["P"] / t_cycle)
                tcyc.append(t_cycle)
                desc = ("per step one cycle of the reference's OWN classes (oracle/_ref: its sources compiled against "
                        "stand-in Eigen/FCL/octomap headers): TrajectorySampler::generateTrajectories over all %d slots "
                        "with its ThreadPool (%d threads, %.3f s) + CostEvaluator::setPointScan + getMinTrajectoryCost, "
                        "single-threaded as the reference's CPU evaluator is, over %s admissible trajectories vs the "
                        "full %d-point cloud (%.2f s)%s" %
                        (n_slots, threads, r["t_sampler"],
                         ("all %d" % r["n_admissible"]) if r["evaluated"] == r["n_admissible"]
                         else ("the first %d of %d" % (r["evaluated"], r["n_admissible"])), len(c), r["t_cost"],
                         "" if r["evaluated"] == r["n_admissible"] else ", cost part extrapolated to all admissible"))
    else:
        kind = "port"
        max_traj = None
        if port_full > budget and n_adm0 > 0:  # bounded sample: cost terms over the first m admissible, >= 16 per thread
            max_traj = min(n_adm0, int(max(16 * threads, n_adm0 * max(budget - t_s, 0.02) / max(t_c, 1e-9))))
        for i in range(warmup + steps):
            c = clouds[i % len(clouds)]
            t_s, t_c, n_slots, P, n_adm, m, _ = oracle_cycle(orc, kw, path, seg, vel, pose, c, threads, max_traj)
            t_cycle = t_s + t_c * (n_adm / max(m, 1))
            if i >= warmup:
                vals.append(n_slots * P / t_cycle)
                tcyc.append(t_cycle)
                desc = ("per step one whole cycle of the oracle port: sampler + collision over all %d slots, the five "
                        "cost terms over %s admissible trajectories vs the full %d-point cloud%s; %d thread(s)" %
                        (n_slots, ("all %d" % n_adm) if m == n_adm else ("the first %d of %d" % (m, n_adm)), len(c),
                         "" if m == n_adm else " (cost part extrapolated to all admissible)", threads))
    value = float(np.mean(vals))
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": steps, "warmup": warmup, "ms_per_step": float(np.mean(tcyc) * 1e3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32+f64",
        "data": "synthetic", "config": config_dict("cycle"),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": kind, "sample": desc,
                         "port_all_threads": {"value": n_slots * P / port_full, "unit": UNIT, "cores": threads,
                                              "ms_per_cycle": port_full * 1e3,
                                              "note": "the oracle PORT with every stage (cost terms included) fanned "
                                                      "out over all host threads, one whole cycle, no extrapolation: "
                                                      "faster than the reference can run, bit-identical results"}},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                "winner_cloud0": win0, "admissible_cloud0": n_adm0},
        "gpu_launches": 0,
        "note": "collision queries go through the analytic occupied-voxel model that stands in for FCL/octomap "
                "(absent here), cheaper than FCL -> this baseline flatters the CPU",
    }
    emit(line)
    return 0


def run_cpu_baseline_only(args):
    """Subprocess of the repo arm (rank 0, N = 1): the oracle port, ONE thread, bounded sample. Kept out
    of the repo arm's own process so that process never loads anything from oracle/."""
    orc, wl, kw, path, seg, vel, pose = oracle_cycle_inputs()
    gen, _ = wl.CLOUD_FAMILY[HEADLINE]
    cloud = gen(0, n=N_POINTS_CLOUD) if HEADLINE != "empty_cloud" else wl.cloud_empty()
    t_s, t_c, n_slots, P, n_adm, m, _ = oracle_cycle(orc, kw, path, seg, vel, pose, cloud, 1, 8)
    kind = "port"
    if orc.ref_available():  # the reference's own classes, 1 thread (its default max_num_threads)
        kind = "reference"
        cal = ref_cycle(orc, wl, kw, seg, vel, pose, cloud, 1, 16)
        m = int(max(16, args.cpu_budget / max(cal["t_cost"] / max(cal["evaluated"], 1), 1e-9)))
        r = ref_cycle(orc, wl, kw, seg, vel, pose, cloud, 1, m)
        t_s, t_c, n_adm, m = r["t_sampler"] + r["t_points"], r["t_cost"], r["n_admissible"], r["evaluated"]
    else:
        per_traj = t_c / max(m, 1)
        m = int(max(8, min(n_adm, args.cpu_budget / max(per_traj, 1e-9))))
        t_s, t_c, n_slots, P, n_adm, m, _ = oracle_cycle(orc, kw, path, seg, vel, pose, cloud, 1, m)
    t_cycle = t_s + t_c * (n_adm / max(m, 1))
    out = {"cycle": {"value": n_slots * P / t_cycle, "unit": UNIT, "cores": 1, "kind": kind,
                     "sample": "%s: sampler + collision over all %d slots (%.2f s) + five cost terms over the "
                               "first %d of %d admissible trajectories vs the full %d-point cloud (%.2f s), cost part "
                               "extrapolated; 1 thread; distribution %s" %
                               ("the reference's own classes (oracle/_ref)" if kind == "reference" else "oracle port",
                                n_slots, t_s, m, n_adm, len(cloud), t_c, HEADLINE),
                     "full_cycle_ms_extrapolated": t_cycle * 1e3}}
    out["entry_points"] = cpu_entry_points(orc, wl)
    emit(out)
    return 0


def cpu_entry_points(orc, wl):
    """Oracle (port) timings of the other entry points on the reference's published shapes, 1 thread."""
    res = {}
    kind = "port"
    if orc.ref_available():  # the reference's own sources (oracle/_ref)
        orc.set_backend("ref")
        kind = "reference"

    def timed(fn, reps):
        fn()
        t = []
        for _ in range(reps):
            t0 = time.perf_counter()
            fn()
            t.append(time.perf_counter() - t0)
        return float(np.median(t) * 1e3)

    for beams in (3600, 1080):
        angles, ranges = wl.mapping_scan(beams)
        res["mapper_scan_%d" % beams] = {
            "value": timed(lambda: orc.mapper_scan_to_grid(400, 400, 0.05, (0.0, 0.0, 0.0), 0.0, angles, ranges), 20),
            "unit": "ms", "cores": 1, "kind": kind, "sample": "median of 20 calls"}
    pts = wl.cloud_lattice(0)
    data = wl.cloud_bytes_xyz16(pts)
    ang = np.array([2 * math.pi * i / 360 for i in range(360)], np.float64)
    czc = orc.cz_cfg()
    res["critical_zone_cloud_100k"] = {
        "value": timed(lambda: orc.cz_check_cloud(czc, ang, data, 16, 16 * len(pts), 1, len(pts), 0, 4, 8, True), 20),
        "unit": "ms", "cores": 1, "kind": kind, "sample": "median of 20 calls"}
    a36, r36 = wl.dense_slowdown_scan(3600)
    res["critical_zone_scan_3600"] = {
        "value": timed(lambda: orc.cz_check_scan(czc, a36, r36, True), 50),
        "unit": "ms", "cores": 1, "kind": kind, "sample": "median of 50 calls"}
    # CostEvaluator_5k_Trajs on a bounded sample of rows (the port needs ~30 s for all 5001)
    s = wl.heavy_trajectory_samples()
    way = [(0.0, 0.0), (5.0, 0.0), (10.0, 0.0)]
    path = orc.Path(way, 0.01, 1000.0, 1000)
    seg = path.segment(0)
    ccfg = orc.cost_cfg(w_path=1.0, w_goal=1.0, w_obstacles=0.0, w_smooth=1.0, w_jerk=1.0, acc_limits=(3.0, 3.0, 3.0))
    m = 256
    sub = {k: np.ascontiguousarray(v[:m]) for k, v in s.items()}
    t0 = time.perf_counter()
    if kind == "reference":
        orc.ref_cost_evaluate(ccfg, sub, way, 0.01, seg, (0.0, 0.0, 0.0), 10.0, want_costs=False)
    else:
        orc.cost_evaluate(ccfg, sub, path, seg, None, 0.0, n_threads=1)
    dt = time.perf_counter() - t0
    res["cost_evaluator_5k"] = {"value": dt * (len(s["x"]) / m) * 1e3, "unit": "ms", "cores": 1, "kind": kind,
                                "sample": "first %d of %d rows, extrapolated" % (m, len(s["x"]))}
    orc.set_backend("port")
    return res


# =================================================================================================
# the repo arm
# =================================================================================================
def measure_distribution(pkg, planner, wl, name, rank, seg, vel, pose, n_lat, resident_cycles):
    """p50/p90/p99 of the public host-buffer call and the device-resident cycle time on one member of
    the cloud family. Returns (record, pinned clouds, last result)."""
    gen, w = wl.CLOUD_FAMILY[name]
    if w is not None:
        planner.set_weights(*w)
    else:
        planner.set_weights(1.0, 1.0, 1.0, 1.0, 1.0)
    clouds = []
    for s in range(DISTINCT):
        c = gen(1000 * rank + s, n=N_POINTS_CLOUD) if name != "empty_cloud" else wl.cloud_empty()
        pa = pkg.PinnedArray((max(len(c), 1), 3), np.float32)
        pa.array[:len(c)] = c
        clouds.append((pa, len(c)))
    for s in range(BANK):
        pa, n = clouds[s % DISTINCT]
        planner.bank_upload(s, pa.array[:n])
    for i in range(30):
        pa, n = clouds[i % DISTINCT]
        r0 = planner.cycle_cloud(vel, pose, pa.array[:n], seg[0], seg[1])
    lat = np.zeros(n_lat)
    t_begin = time.perf_counter()
    for i in range(n_lat):
        pa, n = clouds[i % DISTINCT]
        t0 = time.perf_counter()
        r = planner.cycle_cloud(vel, pose, pa.array[:n], seg[0], seg[1])
        lat[i] = time.perf_counter() - t0
    wall = time.perf_counter() - t_begin
    pa, n = clouds[0]
    r0 = planner.cycle_cloud(vel, pose, pa.array[:n], seg[0], seg[1])
    planner.replay(0, BANK, vel, pose, seg[0], seg[1])  # every bank slot's launch graph captured / warm
    ms, _, last = planner.replay(0, resident_cycles, vel, pose, seg[0], seg[1])
    rec = {"p50_ms": pct(lat, 50), "p90_ms": pct(lat, 90), "p99_ms": pct(lat, 99), "max_ms": float(lat.max() * 1e3),
           "mean_ms": wall / n_lat * 1e3, "resident_ms": ms / resident_cycles, "samples": n_lat,
           "admissible_cloud0": r0.n_admissible,
           "winner_cloud0": {"slot": r0.slot, "cost": float(np.float32(r0.cost))} if r0.is_found else None}
    return rec, clouds, lat, wall


def run_sweep(pkg, wl, kw, path, seg, world, rank, local, dist, robots_total, iters, dump_dir=None):
    """north_star config 5: `robots_total` independent robots (own cloud seed, own current velocity),
    sharded contiguously by robot id across the ranks; no data-path collective, the final gather
    carries 20 bytes per robot. Returns a dict for the JSON line (rank 0) or None."""
    lo, hi = shard_robots(robots_total, world, rank)
    R = hi - lo
    gen, w = wl.CLOUD_FAMILY[HEADLINE]
    n_pts = N_POINTS_CLOUD if HEADLINE != "empty_cloud" else 1
    host = pkg.PinnedArray((R * n_pts, 3), np.float32)
    vels, poses = [], []
    for i, r in enumerate(range(lo, hi)):
        rng = np.random.default_rng(wl.SEED + 7 * r)
        vels.append((float(rng.uniform(0.0, 2.0)), 0.0, float(rng.uniform(-2.0, 2.0))))
        poses.append((0.0, 0.0, 0.0))
        if HEADLINE != "empty_cloud":
            host.array[i * n_pts:(i + 1) * n_pts] = gen(5000 + r, n=n_pts)  # one cloud seed per robot (SURVEY 8d C5)
    planner = make_planner(pkg, kw if w is None else dict(kw, weights=w), path)
    offsets = np.arange(R, dtype=np.int64) * n_pts
    counts = np.full(R, n_pts if HEADLINE != "empty_cloud" else 0, np.int32)
    # one untimed warm-up sweep (device buffers are grown on first use, like the W warm-up steps)
    planner.batch_cloud(vels, poses, host.array, seg[0], seg[1], offsets=offsets, counts=counts)
    e2e_runs = []
    for _ in range(max(1, iters)):
        barrier(dist, local)
        t0 = time.perf_counter()
        res = planner.batch_cloud(vels, poses, host.array, seg[0], seg[1], offsets=offsets, counts=counts)
        e2e_runs.append(max_over_ranks(dist, time.perf_counter() - t0, local))
    e2e_s = float(np.median(e2e_runs))
    host.free()
    slots = list(planner.batch_slots)
    # device resident: the same launch set replayed on the resident batch
    planner.batch_replay(1, R)
    barrier(dist, local)
    ms, res2 = planner.batch_replay(iters, R)
    barrier(dist, local)
    ms = max_over_ranks(dist, ms, local)
    assert [x[2] for x in res] == [x[2] for x in res2], "replayed sweep changed its winners"
    if dump_dir:
        last = gather_results(dist, res2, world, rank)
        if rank == 0:
            dump_sweep_outputs(dump_dir, last)
    P = planner.num_points
    units = sum_over_ranks(dist, float(sum(slots)) * P, local)
    gathered = gather_results(dist, res, world, rank)
    planner.close()
    if rank != 0:
        return None
    found = sum(1 for g in gathered if g[0])
    h2d = R * n_pts * 12
    return {
        "workload": "configs[4]: %d independent robots (cloud seed 5000 + robot id, distribution %s) x ~10k slots x "
                    "%d points vs their own %d-point cloud, sharded by robot over %d GPU(s)" %
                    (robots_total, HEADLINE, P, n_pts, world),
        "robots": robots_total, "robots_per_gpu": R, "iters": iters, "scaling": "strong",
        "ms_per_sweep": ms / iters, "us_per_robot_per_gpu": ms / iters * 1e3 / max(R, 1),
        "value": units / (ms / iters * 1e-3), "unit": UNIT,
        "robots_per_s": robots_total / (ms / iters * 1e-3),
        "e2e_ms_per_sweep": e2e_s * 1e3, "e2e_value": units / e2e_s,
        "h2d_bytes_per_sweep_per_gpu": h2d, "d2h_bytes_per_sweep_per_gpu": R * 20,
        "h2d_effective_gbs_per_gpu": h2d / e2e_s / 1e9,
        "robots_with_a_trajectory": found,
    }


def run_entry_points(pkg, wl, peaks, cpu):
    """The other entry points of the path on the reference's PUBLISHED shapes (benchmark_runner.cpp:
    152-377; protocol benchmark_common.h:256-319: host wall clock around the whole call, host buffers in,
    result in host memory), each with its own roofline and cpu_baseline. published_best_ms = best GPU
    bar of BASELINE.md (AMD Strix iGPU)."""
    out = {}
    hbm = peaks.get("hbm_gbs") or 6550.0

    def lat_loop(fn, n=400, warm=40):
        for _ in range(warm):
            fn()
        lat = np.zeros(n)
        for i in range(n):
            t0 = time.perf_counter()
            fn()
            lat[i] = time.perf_counter() - t0
        return lat

    def entry(name, lat, published, algo_bytes, resident_ms, what, extra=None):
        p50 = pct(lat, 50)
        rec = {"what": what, "p50_ms": p50, "p99_ms": pct(lat, 99), "samples": len(lat),
               "published_best_ms": published, "vs_published": (published / p50) if published else None,
               "roofline": {"bound": "hbm", "unit": "GB/s", "algorithmic_bytes": algo_bytes,
                            "kernel_ms_resident": resident_ms,
                            "achieved": (algo_bytes / (resident_ms * 1e-3) / 1e9) if resident_ms else None,
                            "peak": hbm, "frac": (algo_bytes / (resident_ms * 1e-3) / 1e9 / hbm) if resident_ms else None,
                            "pcie_floor_ms": algo_bytes / 50e9 * 1e3,
                            "note": "these calls move <= 1.6 MB and are bound by launch latency and the PCIe "
                                    "transfer of their host buffers, not by HBM"},
               "cpu_baseline": (cpu or {}).get(name)}
        if extra:
            rec.update(extra)
        out[name] = rec

    for beams, published in ((3600, 0.07), (1080, None)):
        angles, ranges = wl.mapping_scan(beams)
        mp = pkg.LocalMapperGPU(400, 400, 0.05, (0.0, 0.0, 0.0), 0.0, False, beams, 2 * math.pi / beams, 2.0, 0.0, 20.0)
        box = {}

        def call():
            box["g"] = mp.scan_to_grid(angles, ranges, copy=False)  # view of the mapper's buffer, as the reference binding returns
        lat = lat_loop(call)
        g = box["g"]
        res_ms = mp.replay(200) / 200
        entry("mapper_scan_%d" % beams, lat, published, 8 * 400 * 400 + 12 * beams, res_ms,
              "LocalMapperGPU.scanToGrid: %d-ray scan -> 400x400 grid @ 0.05 m (Mapper_Dense_400x400 shape%s); "
              "occupied %d empty %d" % (beams, "" if beams == 3600 else ", BASELINE configs[3] beam count",
                                        int((g == 100).sum()), int((g == 0).sum())))
        mp.close()
    pts = wl.cloud_lattice(0)
    data = wl.cloud_bytes_xyz16(pts)
    ang = np.array([2 * math.pi * i / 360 for i in range(360)], np.float64)
    cz = pkg.CriticalZoneCheckerGPU(pkg.SensorInputType.POINTCLOUD, pkg.RobotGeometry.CYLINDER, (0.51, 2.0),
                                    (0.22, 0.0, 0.4), (0.0, 0.0, 0.99, 0.0), 160.0, 0.3, 0.6, ang, 0.1, 2.0, 20.0)
    box = {}

    def call_cz():
        box["f"] = cz.check(data, 16, 16 * len(pts), 1, len(pts), 0, 4, 8, True)
    lat = lat_loop(call_cz)
    res_ms = cz.replay(200) / 200
    pinned = pkg.PinnedArray(data.shape, np.int8)
    pinned.array[...] = data

    def call_cz_pinned():
        box["f2"] = cz.check(pinned.array, 16, 16 * len(pts), 1, len(pts), 0, 4, 8, True)
    lat_p = lat_loop(call_cz_pinned)
    assert box["f"] == box["f2"]
    entry("critical_zone_cloud_100k", lat, 0.06, 16 * len(pts), res_ms,
          "CriticalZoneCheckerGPU.check: 100000 points x 16 B from a PAGEABLE host buffer, 360 bins "
          "(CriticalZone_100k_Cloud shape); factor %.4f" % box["f"],
          {"p50_ms_page_locked_input": pct(lat_p, 50)})
    cz.close()
    pinned.free()
    a36, r36 = wl.dense_slowdown_scan(3600)
    cz = pkg.CriticalZoneCheckerGPU(pkg.SensorInputType.LASERSCAN, pkg.RobotGeometry.CYLINDER, (0.51, 2.0),
                                    (0.22, 0.0, 0.4), (0.0, 0.0, 0.99, 0.0), 160.0, 0.3, 0.6, a36, 0.1, 2.0, 20.0)

    def call_cz_scan():
        box["fs"] = cz.check(r36, True)
    lat = lat_loop(call_cz_scan)
    res_ms = cz.replay(200) / 200
    entry("critical_zone_scan_3600", lat, 0.02, 8 * 3600, res_ms,
          "CriticalZoneCheckerGPU.check: 3600-ray scan, every ray in the slowdown band (CriticalZone_Dense_Scan "
          "shape); factor %.4f" % box["fs"])
    cz.close()
    # CostEvaluator_5k_Trajs: getMinTrajectoryCost on 5001 rows x 1000 points vs a 1000-point segment,
    # path + goal + smoothness + jerk, no obstacles; the 100 MB of rows travel host -> device inside the clock
    s = wl.heavy_trajectory_samples()
    pth = ProductPath(pkg, [(0.0, 0.0), (5.0, 0.0), (10.0, 0.0)], 0.01, 1000.0)
    kw = wl.cfg_c1(weights=(1.0, 1.0, 0.0, 1.0, 1.0))
    kw.update(vx=(1.0, 3.0, 5.0), vy=(1.0, 3.0, 5.0), omega=(3.14, 3.0, 5.0))
    pl = make_planner(pkg, kw, pth)
    seg_n = min(1000, pth.n)

    def call_ce():
        box["ce"] = pl.get_min_trajectory_cost(s, 0, seg_n)
    lat = lat_loop(call_ce, n=30, warm=3)
    res, costs = box["ce"]
    nbytes = sum(v.nbytes for v in s.values())
    entry("cost_evaluator_5k", lat, 8.23, nbytes, None,
          "CostEvaluator.getMinTrajectoryCost: 5001 trajectories x 1000 points vs a %d-point tracked segment, path + "
          "goal + smoothness + jerk (CostEvaluator_5k_Trajs shape), %.0f MB of pageable rows uploaded inside the "
          "clock; winner row %d cost %.6f" % (seg_n, nbytes / 1e6, res.slot, res.cost),
          {"h2d_gbs": nbytes / (pct(lat, 50) * 1e-3) / 1e9})
    pl.close()
    return out


def run_ours(args):
    world, rank, local, dist = dist_setup(args.gpus)
    numa = pin_to_gpu_numa(local) if world > 1 and not args.no_pin else "not pinned (single rank)"
    import __graft_entry__ as ge
    import workloads as wl

    pkg = ge.load_package()
    kw = wl.cfg_c2()
    path = ProductPath(pkg, wl.straight_points(20.0), 0.01, 1.0)
    seg = wl.tracked_segment(path, 0, 2.0)
    vel, pose = (1.0, 0.0, 0.0), (0.0, 0.0, 0.0)
    planner = make_planner(pkg, kw, path)
    planner.bank_alloc(BANK, N_POINTS_CLOUD)
    steps, warmup = args.steps, max(args.warmup, 3)

    # ---- the cloud family (untimed with respect to the K-step contract; every member measured the
    # same way: N_LAT public calls from page-locked host buffers + a resident replay) ---------------
    family = {}
    names = [HEADLINE] if args.headline_only else [n for n in wl.CLOUD_FAMILY if n != HEADLINE] + [HEADLINE]
    keep = None
    for name in names:
        rec, clouds, lat, wall = measure_distribution(pkg, planner, wl, name, rank, seg, vel, pose,
                                                      max(N_LAT, steps) if name == HEADLINE else N_LAT, 256)
        family[name] = rec
        if name == HEADLINE:
            keep = (clouds, lat, wall)
        else:
            for pa, _ in clouds:
                pa.free()
    clouds, lat, e2e_wall = keep  # the planner's bank and weights are now the headline distribution's

    # ---- warm-up + device-resident timed region: EXACTLY K cycles --------------------------------
    planner.replay(0, max(warmup, BANK), vel, pose, seg[0], seg[1])
    barrier(dist, local)
    sampler = ClockSampler(local) if rank == 0 else None
    l0 = planner.launch_count
    total_ms, _, last = planner.replay(warmup, steps, vel, pose, seg[0], seg[1])
    launches = planner.launch_count - l0
    barrier(dist, local)
    total_ms = max_over_ranks(dist, total_ms, local)
    n_slots, P = last.n_slots, last.n_points
    units_per_step = n_slots * P
    value = world * steps * units_per_step / (total_ms * 1e-3)
    if args.dump_outputs and rank == 0 and args.workload == "cycle":
        dump_cycle_outputs(args.dump_outputs, last)

    # ---- dominant kernels (rollout+collision+cost) timed live with CUDA events -------------------
    ksteps = min(max(steps, 100), 500)
    _, eval_ms, _ = planner.replay(warmup, ksteps, vel, pose, seg[0], seg[1], time_eval=True)
    eval_us = eval_ms * 1e3 / ksteps

    # ---- end to end through the public host-buffer call (headline distribution; the loop ran above,
    # inside measure_distribution: max(K, 1000) calls, wall clock, every call moves its own cloud) ---
    esteps = len(lat)
    e2e_s = max_over_ranks(dist, e2e_wall, local)
    e2e_value = world * esteps * units_per_step / e2e_s
    psteps = 300
    lat_pageable = np.zeros(psteps)
    pageable = [np.array(pa.array[:n]) for pa, n in clouds]
    for i in range(psteps):
        t0 = time.perf_counter()
        planner.cycle_cloud(vel, pose, pageable[i % len(pageable)], seg[0], seg[1])
        lat_pageable[i] = time.perf_counter() - t0
    clocks = sampler.stop() if sampler else None
    n_cloud = clouds[0][1]
    h2d = n_cloud * 12 + 4096
    d2h = 32 + 4 * (5 * P)
    for pa, _ in clouds:
        pa.free()

    # ---- brute-force reference kernel (verification hook, outside every timed region above) -------
    brute = None
    if rank == 0 and not args.no_brute and n_cloud > 0:
        try:
            r = planner.cycle_cloud(vel, pose, pageable[0], seg[0], seg[1])
            samples = [planner.bruteforce_obstacle_costs(r.n_slots)[1:] for _ in range(3)]
            brute = {"pairs": samples[0][1], "ms_fp32_pass": float(np.median([s[0] for s in samples]))}
        except Exception as e:  # noqa: BLE001
            brute = {"error": repr(e)}
    planner.close()

    sweep = None
    if args.sweep_robots > 0:
        sweep = run_sweep(pkg, wl, kw, path, seg, world, rank, local, dist, args.sweep_robots, args.sweep_iters,
                          args.dump_outputs if args.workload == "sweep" else None)
    if rank != 0:
        if dist is not None:
            dist.destroy_process_group()
        return 0

    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass

    # ---- CPU baseline on a bounded sample (rank 0, N = 1 only), in a subprocess -------------------
    cpu, cpu_entries = None, None
    if world == 1 and not args.no_cpu:
        try:
            p = subprocess.run([sys.executable, os.path.abspath(__file__), "--cpu-baseline-only",
                                "--cpu-budget", str(args.cpu_budget)], capture_output=True, text=True, timeout=600)
            d = json.loads(p.stdout.strip().splitlines()[-1])
            cpu, cpu_entries = d["cycle"], d["entry_points"]
        except Exception as e:  # noqa: BLE001
            cpu = {"error": repr(e)}

    entries = None
    if world == 1 and not args.no_entry_points:
        try:
            entries = run_entry_points(pkg, wl, peaks, cpu_entries)
        except Exception as e:  # the headline must not depend on the other entry points
            entries = {"error": repr(e)}

    # ---- roofline ----------------------------------------------------------------------------------
    fp32_peak = pkg.measure_fp32_peak_tflops()
    S = seg[1]
    flops = algorithmic_flops(last.n_admissible, n_slots, P, n_cloud, S)
    achieved = flops / (eval_us * 1e-6) / 1e12
    step_us = total_ms * 1e3 / steps
    # Instruction issue is the roof that bounds the pruned pipeline (integer / control-flow work after
    # exact culling): warp instructions executed per cycle by the whole launch set (ncu
    # smsp__inst_executed.sum, profiles/r2_cycle_ncu_summary.json, same build and distribution; the count
    # is data dependent and comes from that capture, the TIME is this run's) against 4 schedulers x SMs x
    # SM clock. The FP32 figure of SURVEY 8(d) (brute-force-equivalent FLOPs / kernel time) is kept beside
    # it: > 1.0 by construction, evidence of exact culling, not a utilisation.
    sm_mhz = (clocks or {}).get("sm_mhz") or peaks.get("sm_max_mhz") or 1965.0
    peak_issue = 148 * 4 * sm_mhz * 1e6
    inst, inst_sweep = None, None
    try:
        ncu = json.load(open(os.path.join(ROOT, "profiles", "r2_cycle_ncu_summary.json")))
        inst = float(ncu["distributions"][HEADLINE]["warp_instructions_per_cycle"])
        inst_sweep = float(ncu["sweep"]["warp_instructions_per_robot"])
    except Exception:
        pass
    if sweep and inst_sweep:
        per_robot_s = sweep["ms_per_sweep"] * 1e-3 / max(sweep["robots_per_gpu"], 1)
        sweep["roofline"] = {"bound": "issue", "unit": "warp-instructions/s", "achieved": inst_sweep / per_robot_s,
                             "peak": peak_issue, "frac": inst_sweep / per_robot_s / peak_issue,
                             "warp_instructions_per_robot": inst_sweep,
                             "source": "count: ncu launch list of one 64-robot chunk (profiles/r2_cycle_ncu_summary.json); "
                                       "time: live (max over ranks)"}
    # DRAM traffic of one cycle's launch set from the committed `ncu --set full` capture of the same build
    # (dram__bytes_read + dram__bytes_write per kernel, first launch of each kernel; cold cache, serialised)
    traffic, traffic_by_kernel = None, None
    try:
        full = json.load(open(os.path.join(ROOT, "profiles", "r2_cycle_full_ncu_summary.json")))
        traffic_by_kernel = {}
        for k in full["kernels"]:
            name = k["kernel"].split("(")[0].replace("void ", "")
            if name not in traffic_by_kernel and k.get("dram_traffic_bytes") is not None:
                traffic_by_kernel[name] = float(k["dram_traffic_bytes"])
        traffic = sum(traffic_by_kernel.values()) if traffic_by_kernel else None
    except (OSError, KeyError, ValueError):
        pass
    roofline = {
        "kernel": "the whole launch set of one cycle (k_prep_points, k_scan_dist, k_scatter + cell classification, "
                  "k_cell_cand[_heavy], k_path_class, k_path_cand, k_dilate, k_rollout_collide, k_cost_bounds, "
                  "k_cost_split, k_cost_eval)",
        "bound": "issue", "unit": "warp-instructions/s",
        "achieved": (inst / (step_us * 1e-6)) if inst else None, "peak": peak_issue,
        "frac": (inst / (step_us * 1e-6) / peak_issue) if inst else None,
        "warp_instructions_per_cycle": inst, "step_us": step_us,
        "source": "count: ncu launch list profiles/r2_cycle_ncu_summary.json (data dependent); time: live CUDA events",
        "note": "a single control cycle is a LATENCY workload (a chain of twelve short kernels): its issue fraction is "
                "low by nature; the throughput mode of the same kernels is the sweep (roofline.sweep.roofline)",
        "traffic": traffic,
        "traffic_note": "bytes per cycle, profiles/r2_cycle_full_ncu_summary.json (ncu --set full, dense-cluster cloud, "
                        "cold cache): the 1.2 MB cloud read once plus the rows; intermediates stay in L2",
        "fp32_algorithmic": {
            "kernel": "k_rollout_collide + k_cost_bounds + k_cost_split + k_cost_eval (timed back to back on one stream)",
            "bound": "fp32", "unit": "TFLOP/s", "achieved": achieved, "peak": fp32_peak,
            "frac": (achieved / fp32_peak) if fp32_peak else None,
            "peak_source": "measured live: FP32 FMA micro-benchmark in this run (MEASURED_PEAKS.json has no FP32 figure)",
            "kernel_us": eval_us, "share_of_step": eval_us / step_us, "algorithmic_flop_per_launch": flops,
            "note": "SURVEY 8(d): brute-force-equivalent FLOPs of the reference loops / measured kernel time; > 1.0 is "
                    "expected: evidence of exact culling (grid-pruned nearest-obstacle search, branch and bound)"},
        "hbm": {"bound": "hbm", "unit": "GB/s", "peak": peaks.get("hbm_gbs"),
                "achieved": (n_cloud * 12) / (step_us * 1e-6) / 1e9,
                "note": "algorithmic bytes of a whole cycle = the cloud read once; the path is not HBM-bound"},
        "sweep": sweep, "entry_points": entries,
    }
    if brute and "ms_fp32_pass" in brute and brute["ms_fp32_pass"] > 0:
        tf = brute["pairs"] * 6.0 / (brute["ms_fp32_pass"] * 1e-3) / 1e12
        brute.update({"kernel": "k_obstacle_bruteforce (verification hook, never on the control path): minDist2D as "
                                "written, every admissible trajectory point x every cloud point, 6 FLOP per pair",
                      "achieved_tflops": tf, "frac_of_fp32_peak": (tf / fp32_peak) if fp32_peak else None,
                      "vs_pruned_cycle": brute["ms_fp32_pass"] / (total_ms / steps)})
    roofline["bruteforce_formulation"] = brute

    worst = max(family, key=lambda k: family[k]["p99_ms"])
    e2e = {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "steps": esteps, "ms_per_step": e2e_s / esteps * 1e3,
           "p50_ms": pct(lat, 50), "p90_ms": pct(lat, 90), "p99_ms": pct(lat, 99), "latency_samples": esteps,
           "p50_ms_pageable_input": pct(lat_pageable, 50), "distribution": HEADLINE,
           "worst_p99_distribution": worst, "winner_cloud0": family[HEADLINE]["winner_cloud0"],
           "admissible_cloud0": family[HEADLINE]["admissible_cloud0"], "by_distribution": family}
    if args.workload == "sweep" and sweep:
        line = {
            "metric": METRIC, "value": sweep["value"], "unit": UNIT, "n_gpus": world, "steps": sweep["iters"],
            "warmup": 1, "ms_per_step": sweep["ms_per_sweep"], "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f32+f64", "data": "synthetic", "config": config_dict("sweep"),
            "e2e": {"value": sweep["e2e_value"], "unit": UNIT,
                    "h2d_bytes_per_step": sweep["h2d_bytes_per_sweep_per_gpu"] * world,
                    "d2h_bytes_per_step": sweep["d2h_bytes_per_sweep_per_gpu"] * world,
                    "ms_per_step": sweep["e2e_ms_per_sweep"], "steps": sweep["iters"]},
            "gpu_launches": None, "roofline": roofline, "cpu_baseline": cpu, "clocks": clocks, "numa": numa,
        }
    else:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": total_ms / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32+f64", "data": "synthetic", "config": config_dict("cycle"),
            "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu,
            "clocks": clocks, "numa": numa,
        }
    emit(line)
    if dist is not None:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="cycle", choices=["cycle", "sweep"])
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-brute", action="store_true", help="skip the brute-force formulation hook")
    ap.add_argument("--no-entry-points", action="store_true", help="skip mapper / critical zone / cost evaluator")
    ap.add_argument("--no-pin", action="store_true", help="do not bind ranks to their GPU's NUMA node")
    ap.add_argument("--headline-only", action="store_true", help="measure only the headline distribution")
    ap.add_argument("--cpu-budget", type=float, default=10.0, help="seconds of oracle cost work")
    ap.add_argument("--cpu-baseline-only", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--sweep-robots", type=int, default=SWEEP_ROBOTS,
                    help="robots of the batched multi-robot sweep (config 5), 0 = skip")
    ap.add_argument("--sweep-iters", type=int, default=3)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed path returned in its last step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if args.dump_outputs and args.workload == "sweep" and args.sweep_robots <= 0:
        ap.error("--dump-outputs with --workload sweep needs --sweep-robots > 0")
    claim_stdout()
    if args.cpu_baseline_only:
        return run_cpu_baseline_only(args)
    if args.impl == "reference":
        return run_reference(args)
    return run_ours(args)


if __name__ == "__main__":
    sys.exit(main())
