"""Port vs reference sources (CPU): oracle/kompass_oracle.cpp against oracle/_ref/libkompass_ref.so,
which is the REFERENCE'S OWN translation units (path.cpp, trajectory_sampler.cpp, collision_check.cpp,
cost_evaluator.cpp, local_mapper.cpp, critical_zone_check.cpp, controller/follower/dwa.cpp) compiled
where they lie in a reference checkout (REF in oracle/Makefile) against the stand-in headers of
oracle/shim (`make -C oracle ref`). Identical bits are demanded over seeded random draws for: sizes,
path interpolation and segmentation, every sampler row (enumeration order, rollout, drop / pad), every
per-trajectory cost and the argmin, the mapper (plain, Bayesian, warp), cloud binning (both overloads)
and the critical zone. What this pins is the port's fidelity to the reference's control flow, operand widths and
operation order; the Eigen kernels (oracle/shim/Eigen) and the collision query (voxel_model.h) are
shared by both arms by construction and stay restated.

Stored record (tests/golden/oracle_vs_ref.json): the reference sources are not part of this repository,
so every value the port contributes to a comparison is also checked, in order, against a SHA-256 digest
stored per test case. The digests were recorded from the port while it matched the reference library
bit for bit on all of these cases. With the library present, both checks run. Without it, the stored
digests stand in for the reference side, and the port's own value is what `both` returns for it.
Re-record after an intended change of the port (and only after it matches the reference library again):

    KC_RECORD_ORACLE_VS_REF=1 python -m pytest tests/test_oracle_vs_ref.py"""
import hashlib
import json
import math
import os

import numpy as np
import pytest

import orc
import workloads as wl

LIVE = orc.ref_available()
RECORD = os.environ.get("KC_RECORD_ORACLE_VS_REF") == "1"
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "oracle_vs_ref.json")
_STORED = {} if RECORD else json.load(open(GOLDEN))["digests"]
_RECORDED = {}


def _canon(v):
    """Exact bytes of a value handed to a comparison: dtype, shape and bits of arrays, hex of floats."""
    if isinstance(v, np.ndarray):
        a = np.ascontiguousarray(v)
        return b"a%s%s:" % (a.dtype.str.encode(), str(a.shape).encode()) + a.tobytes()
    if isinstance(v, (bool, np.bool_)):
        return b"b%d" % bool(v)
    if isinstance(v, (int, np.integer)):
        return b"i%d" % int(v)
    if isinstance(v, (float, np.floating)):
        return b"f" + float(v).hex().encode()
    if v is None:
        return b"n"
    if isinstance(v, (tuple, list)):
        return b"(" + b",".join(_canon(x) for x in v) + b")"
    if isinstance(v, dict):
        return b"{" + b",".join(k.encode() + b"=" + _canon(v[k]) for k in sorted(v)) + b"}"
    if isinstance(v, orc.Path):
        return _canon({k: getattr(v, k) for k in ("n", "X", "Y", "acc", "curv", "total_length", "seg_starts")})
    raise TypeError(type(v))


class _Record:
    """The port's values of one test case, each checked against its stored digest as it is produced."""

    def __init__(self, name):
        self.name, self.got = name, []
        self.want = None if RECORD else _STORED.get(name)
        assert RECORD or self.want is not None, f"no stored record for {name}"

    def check(self, v):
        d = hashlib.sha256(_canon(v)).hexdigest()[:12]
        i = len(self.got)
        self.got.append(d)
        if not RECORD:
            assert i < len(self.want) and d == self.want[i], f"{self.name}: port value {i} differs from the stored record"


_rec = None


@pytest.fixture(autouse=True)
def _port_record(request):
    global _rec
    _rec = _RECORDED[request.node.name] = _Record(request.node.name)
    yield
    orc.set_backend("port")
    if not RECORD:
        assert len(_rec.got) == len(_rec.want), (request.node.name, len(_rec.got), len(_rec.want))


@pytest.fixture(scope="module", autouse=True)
def _write_record():
    yield
    if RECORD:
        prov = ("tests/test_oracle_vs_ref.py with KC_RECORD_ORACLE_VS_REF=1: SHA-256 (first 12 hex digits) of each port "
                "value the test compares with the reference sources, in order")
        with open(GOLDEN, "w") as f:  # one line per test case
            f.write('{"_provenance": %s,\n"digests": {\n' % json.dumps(prov))
            f.write(",\n".join("%s: %s" % (json.dumps(k), json.dumps(r.got, separators=(",", ":")))
                                for k, r in sorted(_RECORDED.items())))
            f.write("\n}}\n")


def both(fn):
    """fn() through the port (checked against the stored record), then through the reference sources
    where their library is present; without it the port's value stands on both sides."""
    orc.set_backend("port")
    a = fn()
    _rec.check(a)
    if not LIVE:
        return a, a
    orc.set_backend("ref")
    b = fn()
    orc.set_backend("port")
    return a, b


def same_bits(a, b):
    a, b = np.ascontiguousarray(a), np.ascontiguousarray(b)
    if a.shape != b.shape:
        return False
    if a.dtype == np.float32:
        return np.array_equal(a.view(np.uint32), b.view(np.uint32))
    if a.dtype == np.float64:
        return np.array_equal(a.view(np.uint64), b.view(np.uint64))
    return np.array_equal(a, b)


PATHS = {
    "global_path": wl.GLOBAL_PATH_XY,
    "circle": wl.circle_test_points(),
    "uturn": wl.uturn_points(),
    "straight": wl.straight_test_points(),
    "two_points": wl.straight_points(20.0),
    "short": [(0.0, 0.0), (0.004, 0.001)],
}


def test_sizes():
    for ct in (0, 1, 2):
        for lin in (1, 2, 3, 10, 20, 100, 224):
            for ang in (1, 2, 9, 20, 101):
                a, b = both(lambda: orc.lib().orc_num_trajectories(ct, lin, ang))
                assert a == b
    for dt, T in ((0.1, 1.0), (0.02, 1.0), (0.02, 2.0), (0.03, 1.0), (0.1, 0.25)):
        a, b = both(lambda: orc.lib().orc_num_points(dt, T))
        assert a == b


@pytest.mark.parametrize("name", list(PATHS))
@pytest.mark.parametrize("interp,seg_len", [(0.01, 1.0), (0.05, 0.7), (0.13, 3.0)])
def test_path_interpolation_and_segments(name, interp, seg_len):
    def run():
        p = orc.Path(PATHS[name], interp, seg_len, int(seg_len / interp + 1))
        return p
    a, b = both(run)
    assert a.n == b.n
    for k in ("X", "Y", "acc", "curv"):
        assert same_bits(getattr(a, k), getattr(b, k)), k
    assert np.float32(a.total_length) == np.float32(b.total_length)
    assert np.array_equal(a.seg_starts, b.seg_starts)
    # View::totalSegmentLength of a few parts
    for s, c in ((0, min(a.n, 101)), (a.n // 3, min(57, a.n - a.n // 3)), (max(0, a.n - 5), min(5, a.n))):
        if c < 2:
            continue
        orc.set_backend("port")
        la = float(np.float32(orc.lib().orc_segment_length(orc.fp(a.X), orc.fp(a.Y), s, c)))
        _rec.check(la)
        lb = la
        if LIVE:
            orc.set_backend("ref")
            lb = orc.ref_segment_length(PATHS[name], interp, s, c)
        assert np.float32(la) == np.float32(lb), (s, c, la, lb)


def _sampler_cases():
    rng = np.random.default_rng(wl.SEED + 401)
    cases = []
    for i in range(14):
        ct = int(rng.integers(0, 3))
        shape = int(rng.choice([0, 0, 2, 1]))
        dims = {0: (float(rng.uniform(0.1, 0.4)), float(rng.uniform(0.3, 1.2)), 0.0),
                1: (float(rng.uniform(0.3, 0.7)), float(rng.uniform(0.2, 0.5)), float(rng.uniform(0.3, 0.9))),
                2: (float(rng.uniform(0.15, 0.45)), 0.0, 0.0)}[shape]
        yaw = float(rng.uniform(-3, 3))
        rot = [(0.0, 0.0, math.sin(yaw / 2), math.cos(yaw / 2)), (0.0, 0.0, 0.0, 1.0), (1.0, 0.0, 0.0, 0.0),
               (0.0, 1.0, 0.0, 0.0)][int(rng.integers(0, 4))]
        kw = dict(control_type=ct, time_step=float(rng.choice([0.05, 0.1, 0.02])),
                  prediction_horizon=float(rng.choice([0.5, 1.0, 1.5])), control_horizon=float(rng.choice([0.1, 0.2, 0.3])),
                  max_linear_samples=int(rng.integers(3, 14)), max_angular_samples=int(rng.integers(3, 14)),
                  vx=(float(rng.uniform(0.5, 2.0)), float(rng.uniform(1, 10)), float(rng.uniform(1, 10))),
                  vy=(float(rng.uniform(0.3, 1.0)), float(rng.uniform(1, 5)), float(rng.uniform(1, 5))),
                  omega=(float(rng.uniform(0.5, 4.0)), float(rng.uniform(1, 10)), float(rng.uniform(1, 10))),
                  shape=shape, dims=dims, sensor_position=(float(rng.uniform(-0.2, 0.2)), float(rng.uniform(-0.1, 0.1)),
                                                         float(rng.uniform(0.0, 0.4))),
                  sensor_rotation=rot, octree_resolution=float(rng.choice([0.05, 0.1, 0.17])),
                  drop_samples=bool(rng.integers(0, 2)))
        vel = (float(rng.uniform(-0.5, 1.5)), float(rng.uniform(-0.3, 0.3)) if ct == 2 else 0.0, float(rng.uniform(-1, 1)))
        pose = (float(rng.uniform(-2, 2)), float(rng.uniform(-2, 2)), float(rng.uniform(-3, 3)))
        use_scan = bool(rng.integers(0, 2))
        cases.append((i, kw, vel, pose, use_scan))
    return cases


@pytest.mark.parametrize("case", _sampler_cases(), ids=lambda c: f"case{c[0]}")
def test_sampler_rows(case):
    i, kw, vel, pose, use_scan = case
    rng = np.random.default_rng(wl.SEED + 900 + i)
    if use_scan:
        ranges, angles = wl.scan_360(40 + i, n=360, lo=0.25, hi=4.0)
        ranges[::17] = np.inf
        sensor = dict(scan=(ranges, angles))
    else:
        r = rng.uniform(0.3, 4.0, 3000)
        a = rng.uniform(0, 2 * math.pi, 3000)
        cloud = np.stack([pose[0] + r * np.cos(a), pose[1] + r * np.sin(a), rng.uniform(-0.2, 0.8, 3000)], 1).astype(np.float32)
        sensor = dict(cloud=cloud)

    def run():
        cfg = orc.sampler_cfg(**kw)
        return orc.sampler_generate(cfg, vel, pose, **sensor)
    a, b = both(run)
    assert a["P"] == b["P"]
    na, nb = len(a["x"]), len(b["x"])
    if kw["shape"] == 1 and na != nb:
        # a box robot's heading reaches the collision query through the float rotation matrix in the
        # reference and as an angle in the port: tangency-level differences may move a slot
        assert abs(na - nb) <= max(1, na // 200)
        return
    assert na == nb, (na, nb)
    for k in ("vx", "vy", "omega", "x", "y"):
        assert same_bits(a[k], b[k]), k


def _random_samples(rng, n, P):
    t = np.arange(P) * 0.05
    x = (t[None, :] * rng.uniform(0.2, 1.5, (n, 1))).astype(np.float32)
    y = (np.sin(t[None, :] * rng.uniform(0.1, 2.0, (n, 1))) * rng.uniform(0, 1.0, (n, 1))).astype(np.float32)
    return dict(x=x, y=y, vx=rng.uniform(-1, 1, (n, P - 1)).astype(np.float32),
                vy=rng.uniform(-0.2, 0.2, (n, P - 1)).astype(np.float32),
                omega=rng.uniform(-2, 2, (n, P - 1)).astype(np.float32))


@pytest.mark.parametrize("seed", range(8))
def test_costs_and_argmin(seed):
    rng = np.random.default_rng(wl.SEED + 1300 + seed)
    n, P = int(rng.integers(20, 120)), int(rng.integers(5, 60))
    samples = _random_samples(rng, n, P)
    if seed % 4 == 0:  # constant-velocity rows: smoothness / jerk are exact zeros
        samples["vx"][:] = samples["vx"][:, :1]
        samples["vy"][:] = 0
        samples["omega"][:] = samples["omega"][:, :1]
    if seed == 5:  # ties: duplicated rows, the lowest index must win
        for k in samples:
            samples[k][7] = samples[k][3]
            samples[k][11] = samples[k][3]
    name = list(PATHS)[seed % 4]
    interp = 0.01 if seed % 2 == 0 else 0.04
    w = [float(x) for x in rng.uniform(0, 2, 5)]
    if seed == 3:
        w[2] = 0.0
    if seed == 6:
        w[0] = w[1] = 0.0
    acc = tuple(float(x) for x in rng.uniform(0.5, 5, 3))
    if seed == 2:
        acc = (acc[0], 0.0, acc[2])  # an axis without a limit is skipped (q4)
    yaw = float(rng.uniform(-1, 1))
    ccfg_kw = dict(w_path=w[0], w_goal=w[1], w_obstacles=w[2], w_smooth=w[3], w_jerk=w[4], acc_limits=acc,
                   sensor_position=(0.15, -0.05, 0.2), sensor_rotation=(0.0, 0.0, math.sin(yaw / 2), math.cos(yaw / 2)))
    pose = (float(rng.uniform(-1, 1)), float(rng.uniform(-1, 1)), float(rng.uniform(-3, 3)))
    max_range = float(rng.choice([6.0, 10.0, 12.0]))
    sensor = {}
    if seed % 3 == 0:
        ranges, angles = wl.scan_360(60 + seed, n=200, lo=0.2, hi=8.0)
        ranges[::13] = np.inf  # kept for the cost (q8)
        sensor = dict(scan=(ranges, angles))
    elif seed % 3 == 1:
        sensor = dict(cloud=wl.cloud_c2(70 + seed, n=1500))
    orc.set_backend("port")
    path = orc.Path(PATHS[name], interp, 1.0)
    seg = (int(rng.integers(0, max(1, path.n // 3))), 0)
    seg = (seg[0], int(min(path.n - seg[0], rng.integers(2, 400))))
    ccfg = orc.cost_cfg(**ccfg_kw)
    obs = orc.cost_points(ccfg, pose, **sensor) if sensor else None
    D = float(np.float32(max_range) / np.float32(3.0))
    fa, ia, ca, costs_a = orc.cost_evaluate(ccfg, samples, path, seg, obs, D)
    _rec.check((fa, ia, ca, costs_a))
    fb, ib, cb, costs_b = fa, ia, ca, costs_a
    if LIVE:
        orc.set_backend("ref")
        fb, ib, cb, costs_b = orc.ref_cost_evaluate(orc.cost_cfg(**ccfg_kw), samples, PATHS[name], interp, seg, pose,
                                                    max_range, **sensor)
    assert same_bits(costs_a, costs_b), np.flatnonzero(costs_a != costs_b)[:5]
    assert fa == fb and np.float32(ca) == np.float32(cb)
    if seed != 5:
        assert ia == ib
    else:  # the reference returns the winning ROW; duplicated rows cannot be told apart by content
        assert np.array_equal(samples["x"][ia], samples["x"][ib])
        assert ia == 3 or not np.array_equal(samples["x"][ia], samples["x"][3])


@pytest.mark.parametrize("seed", range(8))
def test_mapper_plain_bayes_warp(seed):
    rng = np.random.default_rng(wl.SEED + 1700 + seed)
    H, W = int(rng.integers(20, 140)), int(rng.integers(20, 140))
    res = float(rng.choice([0.05, 0.1, 0.2]))
    lp = (float(rng.uniform(-0.5, 0.5)), float(rng.uniform(-0.5, 0.5)), 0.0)
    lo = float(rng.uniform(-3, 3))
    n = int(rng.integers(1, 400))
    angles = rng.uniform(-math.pi, math.pi, n)
    ranges = rng.uniform(0.05, max(H, W) * res * 0.9, n)
    a, b = both(lambda: orc.mapper_scan_to_grid(H, W, res, lp, lo, angles, ranges))
    assert same_bits(a, b)
    prev = rng.uniform(0.05, 0.95, (H, W)).astype(np.float32)
    kw = dict(p_prior=float(rng.uniform(0.3, 0.7)), p_occupied=float(rng.uniform(0.55, 0.9)),
              p_empty=float(rng.uniform(0.1, 0.45)), range_sure=float(rng.uniform(0.1, 2.0)),
              range_max=float(rng.uniform(5, 20)), wall_size=float(rng.uniform(0.05, 0.4)))
    (ga, pa), (gb, pb) = both(lambda: orc.mapper_scan_to_grid_bayes(H, W, res, lp, lo, angles, ranges, prev=prev, **kw))
    assert same_bits(ga, gb) and same_bits(pa, pb)
    pos = (float(rng.uniform(-1, 1)), float(rng.uniform(-1, 1)))
    th = float(rng.uniform(-1, 1))
    wa, wb = both(lambda: orc.mapper_warp_previous(H, W, res, kw["p_prior"], pos, th, prev))
    assert same_bits(wa, wb)


def _raw_cloud(rng, n, layout):
    pts = np.stack([rng.uniform(-6, 6, n), rng.uniform(-6, 6, n), rng.uniform(-0.5, 2.5, n)], 1).astype(np.float32)
    pts[::97] = 0.0  # points at the origin are dropped
    if layout == "xyz16":
        buf = np.zeros((n, 4), np.float32)
        buf[:, :3] = pts
        return buf.view(np.int8).reshape(-1), 16, (0, 4, 8)
    step, off = 21, (3, 11, 7)  # unaligned fields
    raw = np.zeros((n, step), np.uint8)
    b = pts.view(np.uint8).reshape(n, 3, 4)
    for k in range(3):
        raw[:, off[k]:off[k] + 4] = b[:, k]
    return raw.view(np.int8).reshape(-1), step, off


@pytest.mark.parametrize("layout", ["xyz16", "unaligned"])
@pytest.mark.parametrize("seed", range(3))
def test_cloud_binning(layout, seed):
    rng = np.random.default_rng(wl.SEED + 2100 + seed)
    n = 5000
    data, step, off = _raw_cloud(rng, n, layout)
    for bins, max_z in ((360, 2.0), (1080, -1.0), (57, 1.0)):
        a, b = both(lambda: orc.pointcloud_to_laserscan(data, step, step * n, 1, n, off[0], off[1], off[2], 20.0, 0.1, max_z, bins))
        assert same_bits(a, b)
    for angle_step in (0.01, 2 * math.pi / 360, 0.37):
        (ra, aa), (rb, ab) = both(lambda: orc.pointcloud_to_laserscan_step(data, step, step * n, 1, n, off[0], off[1], off[2],
                                                                          15.0, 0.0, 2.0, angle_step))
        assert same_bits(ra, rb) and same_bits(aa, ab)


@pytest.mark.parametrize("seed", range(10))
def test_critical_zone(seed):
    rng = np.random.default_rng(wl.SEED + 2500 + seed)
    shape = int(rng.integers(0, 3))
    dims = {0: (float(rng.uniform(0.2, 0.6)), 1.0, 0.0), 1: (float(rng.uniform(0.4, 0.9)), float(rng.uniform(0.3, 0.7)), 0.5),
            2: (float(rng.uniform(0.2, 0.6)), 0.0, 0.0)}[shape]
    rot = [(0, 0, 0.99, 0.0), (0, 0, 0, 1), (1, 0, 0, 0), (0.1, -0.2, 0.6, 0.7)][seed % 4]  # un-normalised on purpose (q17)
    kw = dict(shape=shape, dims=dims, sensor_position=(float(rng.uniform(-0.3, 0.3)), float(rng.uniform(-0.2, 0.2)), 0.4),
              sensor_rotation=rot, critical_angle=float(rng.uniform(20, 330)), critical_distance=float(rng.uniform(0.1, 0.5)),
              slowdown_distance=float(rng.uniform(0.6, 1.5)))
    n = int(rng.integers(8, 720))
    angles = np.sort(rng.uniform(-math.pi, math.pi, n)) if seed % 2 else np.array([2 * math.pi * i / n for i in range(n)])
    ranges = rng.uniform(0.2, 3.0, n)
    for fwd in (True, False):
        ia, ib = both(lambda: orc.cz_indices(orc.cz_cfg(**kw), angles, fwd))
        assert np.array_equal(ia, ib)
        fa, fb = both(lambda: orc.cz_check_scan(orc.cz_cfg(**kw), angles, ranges, fwd))
        assert np.float32(fa) == np.float32(fb)
    data, step, off = _raw_cloud(rng, 4000, "xyz16" if seed % 2 else "unaligned")
    data = (data.view(np.uint8)).view(np.int8)
    for fwd in (True, False):
        fa, fb = both(lambda: orc.cz_check_cloud(orc.cz_cfg(**kw), angles, data, step, step * 4000, 1, 4000, off[0], off[1], off[2], fwd))
        assert np.float32(fa) == np.float32(fb)


def test_collision_states_share_the_voxel_model():
    """CollisionChecker::updateState / updateSensorData / checkCollisions(state) of the reference class
    over the shared voxel model: the transforms, the z offset of laser points and the frame choices are
    the reference's own."""
    rng = np.random.default_rng(wl.SEED + 2900)
    for shape, dims in ((0, (0.25, 0.6, 0.0)), (2, (0.3, 0.0, 0.0))):
        for rot in ((0, 0, 0, 1), (0, 0, math.sin(0.3), math.cos(0.3)), (1, 0, 0, 0)):
            kw = dict(shape=shape, dims=dims, sensor_position=(0.1, -0.05, 0.2), sensor_rotation=rot, octree_resolution=0.1)
            ranges, angles = wl.scan_360(3, n=720, lo=0.3, hi=3.0)
            st = np.stack([rng.uniform(-3, 3, 1500), rng.uniform(-3, 3, 1500), rng.uniform(-3.2, 3.2, 1500)], 1)
            a, b = both(lambda: orc.check_collision_states(orc.sampler_cfg(**kw), (0.2, 0.1, 0.4), st, scan=(ranges, angles))[1])
            assert np.array_equal(a, b)
            cloud = wl.cloud_c2(5, n=2000)
            for gf in (True, False):
                a, b = both(lambda: orc.check_collision_states(orc.sampler_cfg(**kw), (0.2, 0.1, 0.4), st, cloud=cloud, global_frame=gf)[1])
                assert np.array_equal(a, b)


# ---------------------------------------------------------------------------------------------
# Closed loop: the 18 scenarios of the reference's tests/dwa_test.cpp:161-362 (3 robot types x 3
# paths x obstacle on/off) driven by the REFERENCE'S OWN DWA object, in lock-step with the follower
# oracle (tests/orc_follower.py around the port): tracked state at every step, winner record (cost
# bits, rows) at every step.
# ---------------------------------------------------------------------------------------------
def _apply_control(state, cmd, dt):  # ref: controller_test_helpers.h:12-31
    x, y, yaw = state
    dx = (cmd[0] * math.cos(yaw) - cmd[1] * math.sin(yaw)) * dt
    dy = (cmd[0] * math.sin(yaw) + cmd[1] * math.cos(yaw)) * dt
    x, y, yaw = x + dx, y + dy, yaw + cmd[2] * dt
    while yaw > math.pi:
        yaw -= 2.0 * math.pi
    while yaw < -math.pi:
        yaw += 2.0 * math.pi
    return (x, y, yaw)


_CL_PATHS = {"Straight": wl.straight_test_points, "UTurn": wl.uturn_points, "Circle": wl.circle_test_points}
_CL_OBST = {"Straight": (4.0, 0.0), "UTurn": (10.0, 0.0), "Circle": (5.0, 8.5)}


@pytest.mark.parametrize("avoid", [False, True, "obstacle_cost"])
@pytest.mark.parametrize("ctrl", [0, 1, 2])
@pytest.mark.parametrize("path_name", sorted(_CL_PATHS))
def test_closed_loop_against_reference_dwa(avoid, ctrl, path_name):
    """avoid False / True: the reference's 18 scenarios with its own weights (path 1, goal 1, the rest
    0: the obstacle only acts through the collision stage), run to the goal. "obstacle_cost": the same
    obstacle with the obstacle-distance weight switched on, 150 steps in lock-step (the robot may park in
    front of the obstacle: no goal requirement)."""
    from orc_follower import FollowerOracle
    from parity_util import _split

    kw = dict(control_type=ctrl, time_step=0.1, prediction_horizon=4.0, control_horizon=0.5,
              max_linear_samples=20, max_angular_samples=20, vx=(1.0, 2.0, 2.0), vy=(1.0, 2.0, 2.0),
              omega=(2.0, 3.0, 3.0), shape=0, dims=(0.1, 0.4, 0.0), sensor_position=(0, 0, 0),
              sensor_rotation=(0, 0, 0, 1), octree_resolution=0.1, drop_samples=True,
              weights=(1.0, 1.0, 1.0 if avoid == "obstacle_cost" else 0.0, 0.0, 0.0), max_local_range=10.0)
    max_steps = 150 if avoid == "obstacle_cost" else 1000
    pts = _CL_PATHS[path_name]()
    common, ccfg = _split(kw)
    ref = orc.RefDWA(orc.sampler_cfg(**common), ccfg, goal_tol=0.3) if LIVE else None
    fol = FollowerOracle(kw, goal_dist_tolerance=0.3)
    fol.set_current_path(pts)
    _rec.check(fol.path.n)
    if ref is not None:
        assert ref.set_current_path(pts) == fol.path.n
    p0, p1 = np.float32(pts[0]), np.float32(pts[1])
    state = (float(p0[0]), float(p0[1]), float(np.arctan2(np.float32(p1[1] - p0[1]), np.float32(p1[0] - p0[0]))))
    if path_name == "Circle":
        state = (state[0] + 0.2, state[1], state[2])
    cloud = wl.round_obstacle(*_CL_OBST[path_name], 0.3) if avoid else np.zeros((0, 3), np.float32)
    vel, goal, step = (0.0, 0.0, 0.0), False, 0
    clamp = lambda v: max(min(float(v), 1.0), -1.0)
    try:
        while not goal and step < max_steps:
            fol.set_current_state(*state)
            seg = fol.prepare()
            mine = fol.run_cycle(vel, seg, cloud=cloud)
            tag = f"{ctrl}/{path_name}/{avoid} step {step}"
            assert mine["found"], tag
            cmd = (clamp(mine["vx"][0]), clamp(mine["vy"][0]), clamp(mine["omega"][0]))
            goal = fol.is_goal_reached()
            _rec.check(((fol.c_index, fol.current_segment_index), seg, fol.n_points, fol.sampler_horizon, fol.c_seglen,
                        fol.c_parallel, fol.heading_error, mine["found"], np.float32(mine["cost"]),
                        [mine[k] for k in ("vx", "vy", "omega", "x", "y")], cmd, goal))
            if ref is not None:
                ref.set_current_state(*state)
                got = ref.compute(vel, cloud)
                info = got["info"]
                assert (info.closest_index, info.segment_index) == (fol.c_index, fol.current_segment_index), tag
                assert (info.seg_start, info.seg_count) == seg, tag
                assert info.n_points == fol.n_points, tag
                assert info.horizon == fol.sampler_horizon, tag
                assert info.segment_position == fol.c_seglen, tag
                assert info.crosstrack_error == fol.c_parallel, tag
                # (the Python follower oracle takes the segment heading from numpy's float32 arctan2, which
                # can differ from glibc's atan2f by one float ulp; nothing on the DWA path consumes it)
                assert abs(info.heading_error - fol.heading_error) <= 5e-7, tag
                assert bool(info.found) == mine["found"], tag
                assert np.float32(info.cost) == np.float32(mine["cost"]), (tag, info.cost, mine["cost"])
                for k in ("vx", "vy", "omega", "x", "y"):
                    assert same_bits(got[k], mine[k]), (tag, k)
                assert tuple(info.cmd) == cmd, tag
            vel = cmd
            state = _apply_control(state, cmd, kw["time_step"])
            if ref is not None:
                assert ref.is_goal_reached() == goal, tag
            step += 1
        assert goal or avoid == "obstacle_cost", f"goal not reached after {step} steps"
    finally:
        if ref is not None:
            ref.close()
