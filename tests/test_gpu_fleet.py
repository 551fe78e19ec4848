"""Multi-robot DWA controller (DWAFleet / kc_fleet_*): every robot of a fleet step returns what an
independent DWA handle with the same configuration, path, state and sensor data returns (winner slot,
cost bits, admissible and slot counts, P, winner rows, every DwaInfo field, the clamped command, the goal
flag). The DWA handles are pinned to the follower oracle by test_gpu_dwa_controller.py; the oracle
checks a few fleet steps here on its own."""
import math

import numpy as np
import pytest

import workloads as wl
from orc_follower import FollowerOracle
from parity_util import assert_cycle_parity
from test_gpu_dwa_controller import OBSTACLES, PATHS, RADIUS, ROBOTS, apply_control, scenario_cfg

pytestmark = pytest.mark.gpu

INFO_FIELDS = ["closest_index", "segment_index", "seg_start", "seg_count", "n_points", "segment_position",
               "crosstrack_error", "heading_error", "horizon", "target_x", "target_y", "target_yaw"]


def transformed(pts, dx=0.0, dy=0.0, rot=0.0):
    c, s = math.cos(rot), math.sin(rot)
    return [(c * x - s * y + dx, s * x + c * y + dy) for x, y in pts]


def start_state(pts, dx=0.0, dy=0.0):
    p0, p1 = np.float32(pts[0]), np.float32(pts[1])
    yaw = float(np.arctan2(np.float32(p1[1] - p0[1]), np.float32(p1[0] - p0[0])))
    return (float(p0[0]) + dx, float(p0[1]) + dy, yaw)


def assert_robot_parity(out, fleet, r, res, dwa, tag=""):
    """fleet step output `out` of robot r == the independent handle's result `res` / state."""
    tag = f"robot {r} {tag}"
    assert bool(out["found"][r]) == res.is_found, tag
    assert out["slot"][r] == res.slot and out["n_admissible"][r] == res.n_admissible, tag
    assert out["n_slots"][r] == res.n_slots and out["n_points"][r] == res.n_points, tag
    assert np.float32(out["cost"][r]).tobytes() == np.float32(res.cost).tobytes(), tag
    traj = fleet.get_trajectory(r)
    assert traj.is_found == res.is_found and traj.slot == res.slot and traj.n_points == res.n_points, tag
    for k in ("vx", "vy", "omega", "x", "y"):
        assert np.array_equal(getattr(traj, k), getattr(res, k)), (tag, k)
    info = out["info"][r]
    for k in INFO_FIELDS:
        assert getattr(info, k) == getattr(dwa.info, k), (tag, k, getattr(info, k), getattr(dwa.info, k))
    assert tuple(out["cmd"][r]) == dwa._cmd(), tag


def make_pair(pkg, kw, paths, fp=None, tuning=()):
    cfg = pkg.planner_config(**kw)
    fleet = pkg.DWAFleet(cfg, fp, n_robots=len(paths))
    dwas = [pkg.DWA(cfg, fp) for _ in paths]
    for key, val in tuning:
        fleet.planner.set_tuning(key, val)
        for d in dwas:
            d.planner.set_tuning(key, val)
    for r, pts in enumerate(paths):
        fleet.set_current_path(r, pts)
        dwas[r].set_current_path(pts)
    return fleet, dwas


def step_both(fleet, dwas, states, vels, clouds=None, scans=None):
    fleet.set_current_states([(s[0], s[1], s[2], 0.0) for s in states])
    out = fleet.compute_velocity_commands(vels, clouds=clouds, scans=scans)
    res = []
    for r, d in enumerate(dwas):
        d.set_current_state(*states[r])
        if clouds is not None:
            res.append(d.compute_velocity_commands(vels[r], cloud=clouds[r]))
        else:
            res.append(d.compute_velocity_commands(vels[r], scan=scans[r]))
    return out, res


def twelve_paths():
    s, u, c = wl.straight_test_points(), wl.uturn_points(), wl.circle_test_points()
    return [s, u, c, transformed(s, 1.0, -2.0, 0.6), transformed(u, -3.0, 1.0, -1.1), transformed(c, 2.0, 2.0, 2.0),
            transformed(s, 0.5, 0.5, 2.9), transformed(u, 4.0, -1.0, 0.3), transformed(c, -1.0, -4.0, -0.4),
            transformed(s, -2.0, 3.0, -2.2), transformed(u, 0.0, 0.0, 1.6), transformed(c, 3.0, -3.0, 0.9)]


@pytest.mark.parametrize("prune", [1, 2])
def test_open_loop_parity_clouds(pkg, prune):
    kw = scenario_cfg(1)
    kw.update(weights=(1.0, 1.0, 1.0, 0.5, 0.25))
    paths = twelve_paths()
    fleet, dwas = make_pair(pkg, kw, paths, tuning=[(7, prune)])
    rng = np.random.default_rng(wl.SEED + 301)
    states = [start_state(p, *rng.uniform(-0.2, 0.2, 2)) for p in paths]
    vels = [(float(rng.uniform(0, 0.8)), 0.0, float(rng.uniform(-0.5, 0.5))) for _ in paths]
    for step in range(3):
        clouds = []
        for r, st in enumerate(states):
            if r % 3 == 2:
                clouds.append(np.zeros((0, 3), np.float32))
            else:
                a = rng.uniform(-math.pi, math.pi)
                clouds.append(wl.round_obstacle(st[0] + 1.2 * math.cos(st[2] + a * 0.3),
                                                st[1] + 1.2 * math.sin(st[2] + a * 0.3), 0.3))
        out, res = step_both(fleet, dwas, states, vels, clouds=clouds)
        for r in range(len(paths)):
            assert_robot_parity(out, fleet, r, res[r], dwas[r], f"step {step}")
        vels = [tuple(c) for c in out["cmd"]]
        states = [apply_control(states[r], vels[r], kw["time_step"]) for r in range(len(paths))]
    fleet.close()
    for d in dwas:
        d.close()


def test_mixed_horizons_and_segments_in_one_launch_set(pkg):
    """Robots whose horizon shrinks on a tight curve and robots near their path end share one launch
    set with full-horizon robots: per-robot P and tracked segment inside one chunk."""
    kw = scenario_cfg(1)
    tight = [(0.4 * math.cos(a), 0.4 * math.sin(a)) for a in np.linspace(0, 1.5 * math.pi, 40)]  # kappa 2.5
    straight = wl.straight_test_points()
    paths = [straight, tight, transformed(straight, 1.0, 1.0, 0.5), transformed(tight, -2.0, 0.0, 1.0),
             straight, transformed(straight, 0.0, -3.0, -0.7), wl.uturn_points(), transformed(tight, 3.0, 3.0, 0.0)]
    fleet, dwas = make_pair(pkg, kw, paths, tuning=[(12, 8)])
    states = [start_state(p) for p in paths]
    states[4] = (9.7, 0.02, 0.0)  # 0.3 m before the end of its path: short tracked segment
    end5 = transformed(straight, 0.0, -3.0, -0.7)[-1]
    states[5] = (end5[0] - 0.1, end5[1] + 0.05, -0.7)
    vels = [(0.3, 0.0, 0.0)] * len(paths)
    clouds = [wl.round_obstacle(st[0] + 1.0, st[1] + 0.3, 0.2) if r % 2 else np.zeros((0, 3), np.float32)
              for r, st in enumerate(states)]
    for step in range(2):
        out, res = step_both(fleet, dwas, states, vels, clouds=clouds)
        info = out["info"]
        assert len(set(info.n_points.tolist())) >= 2, info.n_points
        assert len(set(info.seg_count.tolist())) >= 2, info.seg_count
        assert info.n_points.min() < 40 and info.n_points.max() == 40
        for r in range(len(paths)):
            assert_robot_parity(out, fleet, r, res[r], dwas[r], f"step {step}")
        vels = [tuple(c) for c in out["cmd"]]
        states = [apply_control(states[r], vels[r], kw["time_step"]) for r in range(len(paths))]
    fleet.close()
    for d in dwas:
        d.close()


@pytest.mark.parametrize("mount", ["upright", "tilted"])
def test_scans(pkg, mount):
    kw = scenario_cfg(2)
    kw.update(weights=(1.0, 1.0, 1.0, 0.0, 0.0), sensor_position=(0.1, 0.0, 0.3))
    if mount == "tilted":
        kw.update(sensor_rotation=(0.0, math.sin(0.1), 0.0, math.cos(0.1)), octree_resolution=0.08)
    paths = twelve_paths()[:6]
    fleet, dwas = make_pair(pkg, kw, paths)
    rng = np.random.default_rng(wl.SEED + 302)
    states = [start_state(p) for p in paths]
    vels = [(0.4, 0.1, 0.2)] * len(paths)
    for step in range(2):
        scans = []
        for r in range(len(paths)):
            n = [90, 360, 0, 181, 720, 45][r]
            ranges, angles = wl.scan_360(r + 10 * step, n=max(n, 1), lo=0.6, hi=4.0)
            ranges, angles = ranges[:n].copy(), angles[:n].copy()
            if n:
                ranges[rng.integers(0, n, max(1, n // 10))] = np.inf
            scans.append((ranges, angles))
        out, res = step_both(fleet, dwas, states, vels, scans=scans)
        for r in range(len(paths)):
            assert_robot_parity(out, fleet, r, res[r], dwas[r], f"{mount} step {step}")
        vels = [tuple(c) for c in out["cmd"]]
        states = [apply_control(states[r], vels[r], kw["time_step"]) for r in range(len(paths))]
    fleet.close()
    for d in dwas:
        d.close()


@pytest.mark.parametrize("robot", sorted(ROBOTS))
def test_closed_loop(pkg, robot):
    """The 6 scenarios of test_gpu_dwa_controller.py (3 paths x obstacle on/off) as 6 robots of one
    fleet, to the goal, in lock-step with 6 independent DWA handles and the follower oracle."""
    kw = scenario_cfg(ROBOTS[robot])
    fp = pkg.follower_params(goal_dist_tolerance=0.3)
    scen = [(name, avoid) for name in sorted(PATHS) for avoid in (False, True)]
    paths = [PATHS[name]() for name, _ in scen]
    fleet, dwas = make_pair(pkg, kw, paths, fp)
    refs = []
    for pts in paths:
        ref = FollowerOracle(kw, goal_dist_tolerance=0.3)
        ref.set_current_path(pts)
        refs.append(ref)
    states = []
    for (name, _), pts in zip(scen, paths):
        st = start_state(pts)
        states.append((st[0] + 0.2, st[1], st[2]) if name == "Circle" else st)
    clouds = [wl.round_obstacle(*OBSTACLES[name], 0.3) if avoid else np.zeros((0, 3), np.float32)
              for name, avoid in scen]
    R = len(scen)
    vels = [(0.0, 0.0, 0.0)] * R
    done = [False] * R
    min_clear = [math.inf] * R
    step = 0
    while not all(done) and step < 1000:
        fleet.set_current_states([(s[0], s[1], s[2], 0.0) for s in states])
        out = fleet.compute_velocity_commands(vels, clouds=clouds)
        for r in range(R):
            if done[r]:  # frozen at its goal: the fleet keeps stepping it, its handle is left alone
                continue
            tag = f"{robot}/{scen[r]} step {step}"
            dwas[r].set_current_state(*states[r])
            res = dwas[r].compute_velocity_commands(vels[r], cloud=clouds[r])
            assert_robot_parity(out, fleet, r, res, dwas[r], tag)
            assert res.is_found, "DWA failed to find trajectory: " + tag
            if step < 4:
                refs[r].set_current_state(*states[r])
                seg = refs[r].prepare()
                assert (out["info"].seg_start[r], out["info"].seg_count[r]) == seg, tag
                oracle = refs[r].run_cycle(vels[r], seg, cloud=clouds[r])
                assert_cycle_parity(fleet.get_trajectory(r), oracle)
        goals = fleet.is_goal_reached()
        for r in range(R):
            if done[r]:
                assert goals[r]
                continue
            vels[r] = tuple(out["cmd"][r])
            states[r] = apply_control(states[r], vels[r], kw["time_step"])
            if scen[r][1]:
                c = clouds[r]
                d = np.hypot(c[:, 0].astype(np.float64) - states[r][0], c[:, 1].astype(np.float64) - states[r][1])
                min_clear[r] = min(min_clear[r], float(d.min()))
            # the goal check sees the state this step's command was computed from (as in the reference loop)
            g = dwas[r].is_goal_reached()
            assert bool(goals[r]) == g, f"{robot}/{scen[r]} step {step}"
            done[r] = g
        step += 1
    assert all(done), f"{robot}: robots {[scen[r] for r in range(R) if not done[r]]} did not reach the goal"
    for r in range(R):
        if scen[r][1]:
            assert min_clear[r] >= RADIUS, f"{scen[r]} collided with obstacle: clearance {min_clear[r]}"
    fleet.close()
    for d in dwas:
        d.close()


def test_chunks_shared_slices_and_pinned_input(pkg):
    """150 robots (several launch sets), the flat layout with robots sharing cloud slices, a robot with
    no points, page-locked against pageable input, and a sample of robots against independent handles."""
    kw = scenario_cfg(1)
    kw.update(weights=(1.0, 1.0, 1.0, 0.0, 0.0))
    R = 150
    base = twelve_paths()
    paths = [transformed(base[r % len(base)], 0.1 * (r // 12), -0.05 * (r // 12), 0.0) for r in range(R)]
    rng = np.random.default_rng(wl.SEED + 303)
    states = [start_state(p, *rng.uniform(-0.1, 0.1, 2)) for p in paths]
    vels = [(float(rng.uniform(0, 0.8)), 0.0, float(rng.uniform(-0.4, 0.4))) for _ in range(R)]
    pool = [wl.round_obstacle(st[0] + 1.0, st[1] + 0.2, 0.3) for st in states[:20]]
    flat = np.concatenate(pool)
    starts = np.concatenate([[0], np.cumsum([len(c) for c in pool])])
    offsets = np.zeros(R, np.int64)
    counts = np.zeros(R, np.int32)
    for r in range(R):
        k = (r * 7) % 20  # out of order, shared: robots r and r + 20 read the same slice
        offsets[r], counts[r] = starts[k], starts[k + 1] - starts[k]
    counts[37] = 0
    pinned = pkg.PinnedArray(flat.shape, np.float32)
    pinned.array[...] = flat
    cfg = pkg.planner_config(**kw)
    fleet = pkg.DWAFleet(cfg, n_robots=R)
    for r in range(R):
        fleet.set_current_path(r, paths[r])
    fleet.set_current_states([(s[0], s[1], s[2], 0.0) for s in states])
    a = fleet.compute_velocity_commands(vels, clouds=(pinned.array, offsets, counts))
    rows_a = {r: fleet.get_trajectory(r) for r in (0, 37, 149)}
    fleet.set_current_states([(s[0], s[1], s[2], 0.0) for s in states])
    b = fleet.compute_velocity_commands(vels, clouds=(flat, offsets, counts))
    for k in ("found", "cost", "slot", "n_points", "n_slots", "n_admissible", "cmd"):
        assert np.array_equal(a[k], b[k]), k
    for r, t in rows_a.items():
        u = fleet.get_trajectory(r)
        assert np.array_equal(t.x, u.x) and np.array_equal(t.vx, u.vx)
    for r in list(range(0, R, 13)) + [37, 63, 64, 127, 128, R - 1]:
        d = pkg.DWA(cfg)
        d.set_current_path(paths[r])
        d.set_current_state(*states[r])
        res = d.compute_velocity_commands(vels[r], cloud=flat[offsets[r]:offsets[r] + counts[r]])
        assert_robot_parity(b, fleet, r, res, d)
        d.close()
    fleet.close()
    pinned.free()


def test_errors(pkg):
    kw = scenario_cfg(1)
    cfg = pkg.planner_config(**kw)
    fleet = pkg.DWAFleet(cfg, n_robots=3)
    with pytest.raises(ValueError, match="no fleet step"):
        fleet.get_trajectory(0)
    for r in (0, 2):
        fleet.set_current_path(r, wl.straight_test_points())
    fleet.set_current_states(np.zeros((3, 4)))
    empty = [np.zeros((0, 3), np.float32)] * 3
    with pytest.raises(ValueError, match="robot 1: Pointer to global path is NULL"):
        fleet.compute_velocity_commands(np.zeros((3, 3)), clouds=empty)
    fleet.set_current_path(1, wl.uturn_points())
    with pytest.raises(IndexError):
        fleet.set_current_path(3, wl.straight_test_points())
    with pytest.raises(IndexError):
        fleet.get_trajectory(-1)
    with pytest.raises(ValueError, match="vels"):
        fleet.compute_velocity_commands(np.zeros((2, 3)), clouds=empty)
    with pytest.raises(ValueError, match="states"):
        fleet.set_current_states(np.zeros((3, 5)))
    with pytest.raises(ValueError, match="offsets"):
        fleet.compute_velocity_commands(np.zeros((3, 3)), clouds=(np.zeros((4, 3), np.float32), [0, 0], [1, 1]))
    with pytest.raises(ValueError, match="exceed"):
        fleet.compute_velocity_commands(np.zeros((3, 3)), clouds=(np.zeros((4, 3), np.float32), [0, 0, 3], [1, 1, 2]))
    out = fleet.compute_velocity_commands(np.zeros((3, 3)), clouds=empty)
    assert fleet.get_trajectory(2).n_points == out["n_points"][2] == 40
    # the C entry points check extents and robot indexes themselves
    L = pkg.lib()
    import ctypes as C
    res = (pkg.FleetResult * 3)()
    v = np.zeros((3, 3))
    off = np.array([0, -1, 0], np.int64)
    cnt = np.zeros(3, np.int32)
    rc = L.kc_fleet_compute_cloud(fleet._h, v.ctypes.data_as(C.POINTER(C.c_double)), None,
                                  off.ctypes.data_as(C.POINTER(C.c_int64)), cnt.ctypes.data_as(C.POINTER(C.c_int32)),
                                  res, None)
    assert rc == pkg.KC_ERR_INVALID_ARG and b"robot 1: bad sensor extents" in L.kc_last_error()
    out_c = pkg.CycleResult()
    assert L.kc_fleet_get_trajectory(fleet._h, 3, C.byref(out_c)) == pkg.KC_ERR_INVALID_ARG
    assert L.kc_fleet_clear_current_path(fleet._h, 5) == pkg.KC_ERR_INVALID_ARG
    fleet.close()
