"""bench.py --dump-outputs: the files written for a winner record (names, dtypes, values), the argument
checks, and on the GPU that the dump is the last timed cycle, the same from run to run."""
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TRAJ = ("vx", "vy", "omega", "x", "y")


def test_dump_writes_the_winner_record(tmp_path):
    P = 4
    rows = np.arange(5 * P - 3, dtype=np.float32) * np.float32(0.1)
    r = types.SimpleNamespace(is_found=True, cost=float(np.float32(1.25)), slot=7, n_admissible=10, n_slots=20,
                              n_points=P, vx=rows[:P - 1], vy=rows[P - 1:2 * (P - 1)],
                              omega=rows[2 * (P - 1):3 * (P - 1)], x=rows[3 * (P - 1):4 * P - 3], y=rows[4 * P - 3:])
    out = tmp_path / "dump"
    bench.dump_cycle_outputs(str(out), r)
    assert sorted(os.listdir(out)) == sorted(["winner.npy"] + [f"trajectory_{k}.npy" for k in TRAJ])
    w = np.load(out / "winner.npy")
    assert w.dtype == np.float64 and w.tolist() == [1.0, 1.25, 7.0, 10.0, 20.0, 4.0]
    for name in TRAJ:
        a = np.load(out / f"trajectory_{name}.npy")
        assert a.dtype == np.float32 and np.array_equal(a, getattr(r, name))


def test_dump_writes_the_sweep_winners(tmp_path):
    rows = [(True, float(np.float32(2.5)), 41, 300), (False, 0.0, -1, 0)]
    bench.dump_sweep_outputs(str(tmp_path), rows)
    a = np.load(tmp_path / "sweep_winners.npy")
    assert a.dtype == np.float64 and a.tolist() == [[1.0, 2.5, 41.0, 300.0], [0.0, 0.0, -1.0, 0.0]]


def test_dump_outputs_refused_outside_the_timed_cycle(tmp_path):
    out = tmp_path / "dump"
    for extra in (["--impl", "reference"], ["--workload", "sweep", "--sweep-robots", "0"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", str(out), *extra],
                           capture_output=True, text=True, timeout=120)
        assert r.returncode == 2 and "--dump-outputs" in r.stderr
    assert not out.exists()


@pytest.mark.gpu
def test_dump_is_the_last_timed_cycle(pkg, tmp_path):
    """Two short runs dump identical files, and they hold the cycle that bank slot warmup + steps - 1
    computes when replayed directly (the warm-up, latency and kernel-timing cycles end on other clouds)."""
    import workloads as wl

    warmup, steps = 3, 3
    dumps = []
    for i in range(2):
        out = tmp_path / f"dump{i}"
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                            "--warmup", str(warmup), "--headline-only", "--no-cpu", "--no-entry-points", "--no-brute",
                            "--sweep-robots", "0", "--dump-outputs", str(out)],
                           capture_output=True, text=True, timeout=900)
        assert r.returncode == 0, r.stderr[-2000:]
        assert json.loads(r.stdout.strip().splitlines()[-1])["steps"] == steps
        dumps.append({n: np.load(out / n) for n in sorted(os.listdir(out))})
    assert dumps[0].keys() == dumps[1].keys()
    for n in dumps[0]:
        assert dumps[0][n].tobytes() == dumps[1][n].tobytes(), n

    gen, w = wl.CLOUD_FAMILY[bench.HEADLINE]
    path = bench.ProductPath(pkg, wl.straight_points(20.0), 0.01, 1.0)
    seg = wl.tracked_segment(path, 0, 2.0)
    planner = bench.make_planner(pkg, wl.cfg_c2(), path)
    planner.set_weights(*(w if w is not None else (1.0, 1.0, 1.0, 1.0, 1.0)))
    planner.bank_alloc(bench.BANK, bench.N_POINTS_CLOUD)
    clouds = [gen(d, n=bench.N_POINTS_CLOUD) if bench.HEADLINE != "empty_cloud" else wl.cloud_empty()
              for d in range(bench.DISTINCT)]
    for s in range(bench.BANK):
        planner.bank_upload(s, clouds[s % bench.DISTINCT])
    _, _, r = planner.replay(warmup, steps, (1.0, 0.0, 0.0), (0.0, 0.0, 0.0), seg[0], seg[1])
    planner.close()
    got = dumps[0]
    assert got["winner.npy"].tolist() == [float(r.is_found), r.cost, r.slot, r.n_admissible, r.n_slots, r.n_points]
    for k in TRAJ:
        assert got[f"trajectory_{k}.npy"].tobytes() == np.asarray(getattr(r, k), np.float32).tobytes(), k
