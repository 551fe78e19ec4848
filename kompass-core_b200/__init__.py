"""kompass_core_b200 — ctypes front-end of libkompass_b200.so (sm_100a CUDA kernels behind a C-ABI).

The directory is named ``kompass-core_b200`` (not importable by name); load it with
``__graft_entry__.load_package()`` or ``tests/conftest`` which register it as module
``kompass_core_b200``.

Class names mirror the reference's Python-visible surface for this path
(ref: src/kompass_cpp/bindings/bindings_control.cpp:221-273 ``DWA``, bindings_gpu.cpp:13-68
``LocalMapperGPU`` / ``CriticalZoneCheckerGPU``, bindings_types.cpp:139-186 enums). There is no CPU
fallback: importing works anywhere, but creating any object without a CUDA device raises.
"""
import ctypes as C
import enum
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
# KOMPASS_B200_LIB: load another build of the same library (a deployment path, a profiling variant)
LIB_PATH = os.environ.get("KOMPASS_B200_LIB") or os.path.join(_HERE, "lib", "libkompass_b200.so")


class KompassB200Error(RuntimeError):
    pass


class ControlType(enum.IntEnum):  # ref: bindings_types.cpp:139-143
    ACKERMANN = 0
    DIFFERENTIAL_DRIVE = 1
    OMNI = 2


class RobotGeometry(enum.IntEnum):  # ref: bindings_types.cpp RobotGeometry / ShapeType
    CYLINDER = 0
    BOX = 1
    SPHERE = 2


class OccupancyType(enum.IntEnum):  # ref: bindings_mapping.cpp:17-20
    UNEXPLORED = -1
    EMPTY = 0
    OCCUPIED = 100


class SensorInputType(enum.IntEnum):  # ref: critical_zone_check.h:15-18
    LASERSCAN = 0
    POINTCLOUD = 1


KC_OK, KC_ERR_INVALID_ARG, KC_ERR_CUDA, KC_ERR_OOM, KC_ERR_UNSUPPORTED, KC_ERR_OUT_OF_RANGE = range(6)


class PlannerConfig(C.Structure):
    _fields_ = [
        ("control_type", C.c_int32),
        ("time_step", C.c_double),
        ("prediction_horizon", C.c_double),
        ("control_horizon", C.c_double),
        ("max_linear_samples", C.c_int32),
        ("max_angular_samples", C.c_int32),
        ("vx_max", C.c_double), ("vx_acc", C.c_double), ("vx_dec", C.c_double),
        ("vy_max", C.c_double), ("vy_acc", C.c_double), ("vy_dec", C.c_double),
        ("omega_max", C.c_double), ("omega_acc", C.c_double), ("omega_dec", C.c_double),
        ("robot_shape", C.c_int32),
        ("robot_dims", C.c_float * 3),
        ("sensor_position", C.c_float * 3),
        ("sensor_rotation", C.c_float * 4),
        ("octree_resolution", C.c_double),
        ("drop_samples", C.c_int32),
        ("num_ctrl_points", C.c_int64),
        ("w_path", C.c_double), ("w_goal", C.c_double), ("w_obstacles", C.c_double),
        ("w_smooth", C.c_double), ("w_jerk", C.c_double),
        ("max_local_range", C.c_float),
        ("max_num_threads", C.c_int32),
    ]


class CycleResult(C.Structure):
    _fields_ = [
        ("found", C.c_int32), ("cost", C.c_float), ("slot", C.c_int32), ("n_points", C.c_int32),
        ("n_slots", C.c_int32), ("n_admissible", C.c_int32),
        ("vx", C.POINTER(C.c_float)), ("vy", C.POINTER(C.c_float)), ("omega", C.POINTER(C.c_float)),
        ("x", C.POINTER(C.c_float)), ("y", C.POINTER(C.c_float)),
    ]


class Samples(C.Structure):
    _fields_ = [
        ("count", C.c_int32), ("n_points", C.c_int32),
        ("vx", C.POINTER(C.c_float)), ("vy", C.POINTER(C.c_float)), ("omega", C.POINTER(C.c_float)),
        ("x", C.POINTER(C.c_float)), ("y", C.POINTER(C.c_float)),
        ("slots", C.POINTER(C.c_int32)),
    ]


class TrajectoryView(C.Structure):  # kc_trajectory_view
    _fields_ = [("n_points", C.c_int32),
                ("vx", C.POINTER(C.c_float)), ("vy", C.POINTER(C.c_float)), ("omega", C.POINTER(C.c_float)),
                ("x", C.POINTER(C.c_float)), ("y", C.POINTER(C.c_float))]


class PathView(C.Structure):  # kc_path_view
    _fields_ = [("n", C.c_int32), ("X", C.POINTER(C.c_float)), ("Y", C.POINTER(C.c_float)),
                ("acc", C.POINTER(C.c_float)), ("total_length", C.c_float)]


CUSTOM_COST_FN = C.CFUNCTYPE(C.c_double, C.POINTER(TrajectoryView), C.POINTER(PathView), C.c_void_p)


class BatchResult(C.Structure):
    _fields_ = [("found", C.c_int32), ("cost", C.c_float), ("slot", C.c_int32),
                ("n_admissible", C.c_int32), ("n_slots", C.c_int32)]


class CollisionConfig(C.Structure):  # kc_collision_config
    _fields_ = [("robot_shape", C.c_int32), ("robot_dims", C.c_float * 3),
                ("sensor_position", C.c_float * 3), ("sensor_rotation", C.c_float * 4),
                ("octree_resolution", C.c_double)]


class MapperConfig(C.Structure):
    _fields_ = [
        ("grid_height", C.c_int32), ("grid_width", C.c_int32), ("resolution", C.c_float),
        ("laserscan_position", C.c_float * 3), ("laserscan_orientation", C.c_float),
        ("is_pointcloud", C.c_int32), ("scan_size", C.c_int32), ("angle_step", C.c_float),
        ("max_height", C.c_float), ("min_height", C.c_float), ("range_max", C.c_float),
        ("max_points_per_line", C.c_int32),
    ]


class CriticalZoneConfig(C.Structure):
    _fields_ = [
        ("input_type", C.c_int32), ("robot_shape", C.c_int32),
        ("robot_dims", C.c_float * 3), ("sensor_position", C.c_float * 3),
        ("sensor_rotation", C.c_float * 4),
        ("critical_angle", C.c_float), ("critical_distance", C.c_float),
        ("slowdown_distance", C.c_float),
        ("min_height", C.c_float), ("max_height", C.c_float), ("range_max", C.c_float),
        ("cloud_field_type", C.c_int32),
    ]


# every symbol include/kompass_b200.h declares (tests/test_abi.py checks the .so exports them all)
ABI_SYMBOLS = [
    "kc_last_error", "kc_available_accelerators", "kc_version",
    "kc_planner_create", "kc_planner_destroy", "kc_planner_set_weights",
    "kc_planner_set_octree_resolution", "kc_planner_set_drop_samples", "kc_planner_set_max_range",
    "kc_planner_set_prediction_horizon", "kc_planner_num_trajectories", "kc_planner_num_points",
    "kc_planner_set_path", "kc_planner_cycle_scan", "kc_planner_cycle_cloud",
    "kc_planner_fetch_costs", "kc_sampler_generate_scan", "kc_sampler_generate_cloud",
    "kc_cost_set_points_scan", "kc_cost_set_points_cloud", "kc_cost_evaluate",
    "kc_planner_bank_alloc", "kc_planner_bank_upload", "kc_planner_replay",
    "kc_planner_launch_count", "kc_pinned_alloc", "kc_pinned_free", "kc_planner_set_tuning", "kc_planner_debug_stats", "kc_planner_batch_cloud", "kc_planner_batch_replay",
    "kc_follower_params_default", "kc_path_prepare", "kc_dwa_create", "kc_dwa_destroy", "kc_dwa_planner",
    "kc_dwa_set_current_path", "kc_dwa_clear_current_path", "kc_dwa_set_current_state",
    "kc_dwa_set_control_limits", "kc_dwa_is_goal_reached", "kc_dwa_has_path", "kc_dwa_get_path",
    "kc_dwa_get_command", "kc_dwa_compute_scan", "kc_dwa_compute_cloud",
    "kc_dwa_add_custom_cost", "kc_dwa_clear_custom_costs", "kc_dwa_debug_velocity_search_scan",
    "kc_dwa_debug_velocity_search_cloud", "kc_dwa_get_debugging_samples",
    "kc_planner_get_max_range", "kc_planner_num_slots_last", "kc_planner_bruteforce_obstacle_costs",
    "kc_planner_debug_timeline", "kc_planner_fetch_pruned", "kc_planner_debug_stamps",
    "kc_collision_create", "kc_collision_destroy", "kc_collision_reset_octree_resolution",
    "kc_collision_get_radius", "kc_collision_update_state", "kc_collision_update_scan",
    "kc_collision_update_cloud", "kc_collision_check", "kc_collision_check_states",
    "kc_mapper_create", "kc_mapper_destroy", "kc_mapper_scan_to_grid", "kc_mapper_cloud_to_grid",
    "kc_mapper_replay", "kc_mapper_set_bayesian_params", "kc_mapper_scan_to_grid_bayesian",
    "kc_mapper_previous_grid_in_current_pose", "kc_mapper_get_previous_grid", "kc_mapper_set_previous_grid",
    "kc_pointcloud_to_laserscan", "kc_pointcloud_to_laserscan_step", "kc_mapper_cloud_to_grid_bayesian",
    "kc_critical_zone_create", "kc_critical_zone_destroy", "kc_critical_zone_check_scan",
    "kc_critical_zone_check_cloud", "kc_critical_zone_replay",
    "kc_fleet_create", "kc_fleet_destroy", "kc_fleet_planner", "kc_fleet_set_current_path",
    "kc_fleet_clear_current_path", "kc_fleet_set_current_states", "kc_fleet_set_control_limits",
    "kc_fleet_compute_cloud", "kc_fleet_compute_scan", "kc_fleet_get_trajectory", "kc_fleet_is_goal_reached",
]

_lib = None


def lib():
    """Load the CUDA library. Fails loudly when it has not been built (no fallback path)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise KompassB200Error(
                f"{LIB_PATH} is missing: build it with `python kompass-core_b200/build.py` "
                "(kompass_core_b200 has no CPU fallback)")
        L = C.CDLL(LIB_PATH)
        L.kc_last_error.restype = C.c_char_p
        L.kc_version.restype = C.c_char_p
        L.kc_planner_launch_count.restype = C.c_int64
        L.kc_planner_launch_count.argtypes = [C.c_void_p]
        L.kc_planner_destroy.argtypes = [C.c_void_p]
        L.kc_mapper_destroy.argtypes = [C.c_void_p]
        L.kc_critical_zone_destroy.argtypes = [C.c_void_p]
        L.kc_collision_destroy.argtypes = [C.c_void_p]
        L.kc_collision_get_radius.restype = C.c_float
        L.kc_collision_get_radius.argtypes = [C.c_void_p]
        L.kc_fleet_destroy.argtypes = [C.c_void_p]
        L.kc_fleet_planner.restype = C.c_void_p
        L.kc_fleet_planner.argtypes = [C.c_void_p]
        L.kc_debug_atan2f.restype = C.c_float
        L.kc_debug_atan2f.argtypes = [C.c_float, C.c_float]
        _lib = L
    return _lib


_EXC = {KC_ERR_INVALID_ARG: ValueError, KC_ERR_OUT_OF_RANGE: IndexError}


def _check(rc):
    if rc != KC_OK:
        msg = lib().kc_last_error().decode("utf-8", "replace")
        raise _EXC.get(rc, KompassB200Error)(f"kompass_b200 error {rc}: {msg}")


def _f32(a):
    return np.ascontiguousarray(a, dtype=np.float32)


def _f64(a):
    return np.ascontiguousarray(a, dtype=np.float64)


def _fp(a):
    return a.ctypes.data_as(C.POINTER(C.c_float))


def _dp(a):
    return a.ctypes.data_as(C.POINTER(C.c_double))


class PinnedArray:
    """numpy view of page-locked host memory (kc_pinned_alloc): planner inputs placed here are DMA-ed
    without a staging copy. Keep the object alive while the view is in use."""

    def __init__(self, shape, dtype=np.float32):
        L = lib()
        L.kc_pinned_alloc.restype = C.c_void_p
        L.kc_pinned_alloc.argtypes = [C.c_size_t]
        L.kc_pinned_free.argtypes = [C.c_void_p]
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        self._ptr = L.kc_pinned_alloc(n)
        if not self._ptr:
            raise KompassB200Error(L.kc_last_error().decode())
        buf = (C.c_uint8 * max(n, 1)).from_address(self._ptr)
        self.array = np.frombuffer(buf, dtype=dtype, count=int(np.prod(shape))).reshape(shape)

    def free(self):
        if getattr(self, "_ptr", None):
            self.array = None
            lib().kc_pinned_free(C.c_void_p(self._ptr))
            self._ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


def get_available_accelerators():
    """ref: bindings.cpp:47 get_available_accelerators"""
    buf = C.create_string_buffer(4096)
    lib().kc_available_accelerators(buf, 4096)
    return buf.value.decode()


def measure_fp32_peak_tflops():
    """FP32 FMA micro-benchmark (CUDA cores), the roofline denominator of the DWA kernels."""
    out = C.c_float(0)
    _check(lib().kc_debug_fp32_peak_tflops(C.byref(out)))
    return float(out.value)


def planner_config(control_type=ControlType.DIFFERENTIAL_DRIVE, time_step=0.1, prediction_horizon=1.0,
                   control_horizon=0.2, max_linear_samples=20, max_angular_samples=20,
                   vx=(1.0, 5.0, 10.0), vy=(0.0, 0.0, 0.0), omega=(4.0, 3.0, 3.0),
                   shape=RobotGeometry.CYLINDER, dims=(0.1, 0.4, 0.0), sensor_position=(0, 0, 0),
                   sensor_rotation=(0, 0, 0, 1), octree_resolution=0.1, drop_samples=True,
                   num_ctrl_points=-1, weights=(1.0, 1.0, 1.0, 1.0, 1.0), max_local_range=10.0,
                   max_num_threads=1):
    """weights = (path, goal, obstacles, smoothness, jerk)."""
    c = PlannerConfig()
    c.control_type = int(control_type)
    c.time_step, c.prediction_horizon, c.control_horizon = time_step, prediction_horizon, control_horizon
    c.max_linear_samples, c.max_angular_samples = max_linear_samples, max_angular_samples
    c.vx_max, c.vx_acc, c.vx_dec = vx
    c.vy_max, c.vy_acc, c.vy_dec = vy
    c.omega_max, c.omega_acc, c.omega_dec = omega
    c.robot_shape = int(shape)
    d = list(dims) + [0.0] * (3 - len(dims))
    c.robot_dims = (C.c_float * 3)(*d)
    c.sensor_position = (C.c_float * 3)(*sensor_position)
    c.sensor_rotation = (C.c_float * 4)(*sensor_rotation)
    c.octree_resolution = octree_resolution
    c.drop_samples = 1 if drop_samples else 0
    c.num_ctrl_points = num_ctrl_points
    c.w_path, c.w_goal, c.w_obstacles, c.w_smooth, c.w_jerk = weights
    c.max_local_range = max_local_range
    c.max_num_threads = max_num_threads
    return c


def _rows(ptr, n, m):
    if n == 0 or m == 0:
        return np.zeros((n, m), np.float32)
    return np.ctypeslib.as_array(ptr, shape=(n, m)).copy()


_Vec3 = C.c_double * 3
_cycle_cloud = None


def _cycle_cloud_fn():
    global _cycle_cloud
    if _cycle_cloud is None:
        f = lib().kc_planner_cycle_cloud
        f.argtypes = [C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_double), C.c_void_p, C.c_int32, C.c_int32,
                      C.c_int32, C.c_void_p]
        f.restype = C.c_int32
        _cycle_cloud = f
    return _cycle_cloud


class TrajSearchResult:
    """ref: include/datatypes/trajectory.h:611-618 / bindings_control.cpp:210-214
    SamplingControlResult {is_found, cost, trajectory}."""

    def __init__(self, r):
        self.is_found = bool(r.found)
        self.cost = float(np.float32(r.cost))
        self.slot = r.slot
        self.n_points = r.n_points
        self.n_slots = r.n_slots
        self.n_admissible = r.n_admissible
        P = r.n_points
        if self.is_found and P >= 2:
            # the five rows sit back to back in the library's result record (vx, vy, omega [P-1] each,
            # then x, y [P] each: kc_cycle_result in include/kompass_b200.h): one copy, five views
            rows = np.frombuffer(C.string_at(r.vx, (5 * P - 3) * 4), np.float32)
            self.vx, self.vy, self.omega = rows[:P - 1], rows[P - 1:2 * (P - 1)], rows[2 * (P - 1):3 * (P - 1)]
            self.x, self.y = rows[3 * (P - 1):4 * P - 3], rows[4 * P - 3:]
        else:
            self.vx = self.vy = self.omega = self.x = self.y = np.zeros(0, np.float32)


class Planner:
    """DWA hot path: TrajectorySampler + CostEvaluator + argmin behind one handle.

    ref: DWA::findBestPath (include/controllers/dwa.h:183-230)."""

    def __init__(self, cfg):
        self._h = C.c_void_p()
        self._owned = True
        self.cfg = cfg
        _check(lib().kc_planner_create(C.byref(cfg), C.byref(self._h)))

    @classmethod
    def _borrow(cls, handle, cfg):
        """Non-owning view of a planner that lives inside another handle (DWA.planner)."""
        p = cls.__new__(cls)
        p._h, p._owned, p.cfg = handle, False, cfg
        return p

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            if getattr(self, "_owned", True):
                lib().kc_planner_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # -- configuration -------------------------------------------------------------------------
    def set_weights(self, path, goal, obstacles, smooth, jerk):
        _check(lib().kc_planner_set_weights(self._h, C.c_double(path), C.c_double(goal),
                                            C.c_double(obstacles), C.c_double(smooth), C.c_double(jerk)))

    def set_resolution(self, res):  # ref: DWA::resetOctreeResolution
        _check(lib().kc_planner_set_octree_resolution(self._h, C.c_double(res)))

    def set_drop_samples(self, drop):
        _check(lib().kc_planner_set_drop_samples(self._h, 1 if drop else 0))

    def set_max_range(self, r):
        _check(lib().kc_planner_set_max_range(self._h, C.c_float(r)))

    def set_prediction_horizon(self, horizon):
        n = C.c_int32(0)
        _check(lib().kc_planner_set_prediction_horizon(self._h, C.c_double(horizon), C.byref(n)))
        return n.value

    @property
    def num_trajectories(self):
        return lib().kc_planner_num_trajectories(self._h)

    @property
    def num_points(self):
        return lib().kc_planner_num_points(self._h)

    @property
    def launch_count(self):
        return lib().kc_planner_launch_count(self._h)

    def set_tuning(self, key, value):
        _check(lib().kc_planner_set_tuning(self._h, int(key), C.c_int64(int(value))))

    def bruteforce_obstacle_costs(self, n_slots):
        """Verification / roofline hook: obstacle cost of every slot of the last cycle by brute force
        (N*P*M pairs). Returns (costs [n_slots], pass1_ms, pair_evaluations)."""
        costs = np.zeros(n_slots, np.float32)
        ms, tot, pairs = C.c_float(0), C.c_float(0), C.c_double(0)
        _check(lib().kc_planner_bruteforce_obstacle_costs(self._h, _fp(costs), C.byref(ms), C.byref(tot),
                                                          C.byref(pairs)))
        return costs, float(ms.value), float(pairs.value)

    def debug_timeline(self):
        """[(kernel, start_us, end_us)] of the last cycle run with set_tuning(4, 1)."""
        names = (C.c_char_p * 12)()
        a, b = (C.c_float * 12)(), (C.c_float * 12)()
        n = lib().kc_planner_debug_timeline(self._h, names, a, b, 12)
        return [(names[i].decode(), float(a[i]), float(b[i])) for i in range(max(n, 0))]

    def debug_stats(self):
        out = (C.c_int64 * 8)()
        _check(lib().kc_planner_debug_stats(self._h, out))
        return dict(pool_used=out[0], query_cells=out[1], listed_cells=out[2], generic_cells=out[3],
                    longest_list=out[4], kept_points=out[5], path_pool_used=out[6], longest_path_list=out[7])

    def set_path(self, X, Y, acc, total_length):
        X, Y, acc = _f32(X), _f32(Y), _f32(acc)
        _check(lib().kc_planner_set_path(self._h, _fp(X), _fp(Y), _fp(acc), len(X),
                                         C.c_float(total_length)))

    # -- full cycle ----------------------------------------------------------------------------
    def cycle_scan(self, vel, pose, ranges, angles, seg_start, seg_count):
        v, p, r, a = _f64(vel), _f64(pose), _f64(ranges), _f64(angles)
        res = CycleResult()
        _check(lib().kc_planner_cycle_scan(self._h, _dp(v), _dp(p), _dp(r), _dp(a), len(r),
                                           seg_start, seg_count, C.byref(res)))
        return TrajSearchResult(res)

    def cycle_cloud(self, vel, pose, xyz, seg_start, seg_count):
        # the control loop's call: as little interpreter work as possible around the C entry point
        if not (type(xyz) is np.ndarray and xyz.dtype == np.float32 and xyz.flags.c_contiguous):
            xyz = _f32(xyz)
        if xyz.size % 3:
            raise ValueError("cloud must hold xyz triples")
        v, p = _Vec3(*vel), _Vec3(*pose)
        res = CycleResult()
        rc = _cycle_cloud_fn()(self._h, v, p, xyz.__array_interface__["data"][0], xyz.size // 3, seg_start,
                               seg_count, C.byref(res))
        if rc != KC_OK:
            _check(rc)
        return TrajSearchResult(res)

    def fetch_costs(self, n_slots):
        costs = np.zeros(n_slots, np.float32)
        adm = np.zeros(n_slots, np.uint8)
        _check(lib().kc_planner_fetch_costs(self._h, _fp(costs), adm.ctypes.data_as(C.POINTER(C.c_uint8))))
        return costs, adm

    # -- sampler only --------------------------------------------------------------------------
    def fetch_pruned(self, n_slots):
        """uint8 [n_slots]: 1 where fetch_costs reports only a lower bound (slot proven unable to win)."""
        prn = np.zeros(n_slots, np.uint8)
        _check(lib().kc_planner_fetch_pruned(self._h, prn.ctypes.data_as(C.POINTER(C.c_uint8))))
        return prn

    def generate_trajectories(self, vel, pose, scan=None, cloud=None):
        v, p = _f64(vel), _f64(pose)
        s = Samples()
        if scan is not None:
            r, a = _f64(scan[0]), _f64(scan[1])
            _check(lib().kc_sampler_generate_scan(self._h, _dp(v), _dp(p), _dp(r), _dp(a), len(r), C.byref(s)))
        else:
            pts = _f32(cloud).reshape(-1, 3)
            _check(lib().kc_sampler_generate_cloud(self._h, _dp(v), _dp(p), _fp(pts), len(pts), C.byref(s)))
        n, P = s.count, s.n_points
        slots = np.ctypeslib.as_array(s.slots, shape=(n,)).copy() if n else np.zeros(0, np.int32)
        return dict(vx=_rows(s.vx, n, P - 1), vy=_rows(s.vy, n, P - 1), omega=_rows(s.omega, n, P - 1),
                    x=_rows(s.x, n, P), y=_rows(s.y, n, P), slots=slots, P=P)

    # -- cost evaluator on caller samples ------------------------------------------------------
    def set_point_scan(self, pose, scan=None, cloud=None, max_sensor_range=10.0, multiple=3.0):
        p = _f64(pose)
        if scan is not None:
            r, a = _f64(scan[0]), _f64(scan[1])
            _check(lib().kc_cost_set_points_scan(self._h, _dp(r), _dp(a), len(r), _dp(p),
                                                 C.c_float(max_sensor_range), C.c_float(multiple)))
        else:
            pts = _f32(cloud).reshape(-1, 3)
            _check(lib().kc_cost_set_points_cloud(self._h, _fp(pts), len(pts), _dp(p),
                                                  C.c_float(max_sensor_range), C.c_float(multiple)))

    def get_min_trajectory_cost(self, samples, seg_start, seg_count, custom=None):
        x, y = _f32(samples["x"]), _f32(samples["y"])
        vx, vy, om = _f32(samples["vx"]), _f32(samples["vy"]), _f32(samples["omega"])
        n, P = x.shape
        costs = np.zeros(n, np.float32)
        cu, ncu = None, 0
        if custom is not None:  # [n, n_custom] doubles: weight_k * custom_cost_k(trajectory, path)
            cua = _f64(custom).reshape(n, -1)
            cu, ncu = _dp(cua), cua.shape[1]
        res = CycleResult()
        _check(lib().kc_cost_evaluate(self._h, n, P, _fp(vx), _fp(vy), _fp(om), _fp(x), _fp(y),
                                      seg_start, seg_count, cu, ncu, _fp(costs), C.byref(res)))
        return TrajSearchResult(res), costs

    # -- measurement hooks ---------------------------------------------------------------------
    def bank_alloc(self, n_slots, max_points):
        _check(lib().kc_planner_bank_alloc(self._h, n_slots, max_points))

    def bank_upload(self, slot, xyz):
        pts = _f32(xyz).reshape(-1, 3)
        _check(lib().kc_planner_bank_upload(self._h, slot, _fp(pts), len(pts)))

    def replay(self, first_slot, n_cycles, vel, pose, seg_start, seg_count, time_eval=False):
        v, p = _f64(vel), _f64(pose)
        tot, ev = C.c_float(0), C.c_float(0)
        res = CycleResult()
        _check(lib().kc_planner_replay(self._h, first_slot, n_cycles, _dp(v), _dp(p), seg_start,
                                       seg_count, C.byref(tot), C.byref(ev) if time_eval else None,
                                       C.byref(res)))
        return tot.value, (ev.value if time_eval else None), TrajSearchResult(res)

    def batch_cloud(self, vels, poses, clouds, seg_start, seg_count, offsets=None, counts=None):
        """clouds: list of [n_r x 3] arrays (one per robot), or ONE float32 array holding every
        robot's points with `offsets` / `counts` (in points) naming each robot's slice; a PinnedArray's
        .array is DMA-ed without a staging copy."""
        if offsets is None:
            R = len(clouds)
            counts = np.array([len(c) for c in clouds], np.int32)
            offsets = np.zeros(R, np.int64)
            offsets[1:] = np.cumsum(counts[:-1])
            xyz = _f32(np.concatenate([np.asarray(c, np.float32).reshape(-1, 3) for c in clouds], axis=0))
        else:
            offsets, counts = np.ascontiguousarray(offsets, np.int64), np.ascontiguousarray(counts, np.int32)
            R = len(counts)
            xyz = _f32(clouds).reshape(-1, 3)
        v, p = _f64(vels).reshape(R, 3), _f64(poses).reshape(R, 3)
        out = (BatchResult * R)()
        _check(lib().kc_planner_batch_cloud(self._h, R, _dp(v), _dp(p), _fp(xyz),
                                            offsets.ctypes.data_as(C.POINTER(C.c_int64)),
                                            counts.ctypes.data_as(C.POINTER(C.c_int32)), seg_start,
                                            seg_count, out))
        self.batch_slots = [o.n_slots for o in out]
        return [(bool(o.found), float(np.float32(o.cost)), o.slot, o.n_admissible) for o in out]

    def batch_replay(self, n_iters, R):
        tot = C.c_float(0)
        out = (BatchResult * R)()
        _check(lib().kc_planner_batch_replay(self._h, n_iters, C.byref(tot), out))
        return tot.value, [(bool(o.found), float(np.float32(o.cost)), o.slot, o.n_admissible) for o in out]


class FollowerParams(C.Structure):  # ref: follower.h:24-75 FollowerParameters
    _fields_ = [("max_point_interpolation_distance", C.c_double), ("lookahead_distance", C.c_double),
                ("goal_dist_tolerance", C.c_double), ("path_segment_length", C.c_double),
                ("goal_orientation_tolerance", C.c_double), ("loosing_goal_distance", C.c_double),
                ("curvature_horizon_tolerance", C.c_double)]


class DwaInfo(C.Structure):
    _fields_ = [("closest_index", C.c_int32), ("segment_index", C.c_int32), ("seg_start", C.c_int32),
                ("seg_count", C.c_int32), ("n_points", C.c_int32), ("_pad", C.c_int32),
                ("segment_position", C.c_double), ("crosstrack_error", C.c_double),
                ("heading_error", C.c_double), ("horizon", C.c_double), ("target_x", C.c_double),
                ("target_y", C.c_double), ("target_yaw", C.c_double)]


def follower_params(**kw):
    p = FollowerParams()
    lib().kc_follower_params_default(C.byref(p))
    for k, v in kw.items():
        if not hasattr(p, k):
            raise KeyError(k)
        setattr(p, k, float(v))
    return p


def path_prepare(points, interpolate=True, max_point_interpolation_distance=0.01, path_segment_length=1.0,
                 max_points_per_segment=None):
    """Path::interpolate(LINEAR) + Path::segment (host only). Returns dict X, Y, acc, curvature,
    seg_starts, total_length."""
    pts = np.asarray(points, dtype=np.float32)
    x, y = _f32(pts[:, 0]), _f32(pts[:, 1])
    if max_points_per_segment is None:  # ref: follower.cpp:54-59
        max_points_per_segment = int(path_segment_length / max_point_interpolation_distance + 1)
    cap = 1 << 20
    X, Y, acc, K = (np.zeros(cap, np.float32) for _ in range(4))
    seg = np.zeros(cap, np.int32)
    n, ns, tot = C.c_int32(0), C.c_int32(0), C.c_float(0)
    _check(lib().kc_path_prepare(_fp(x), _fp(y), len(x), 1 if interpolate else 0,
                                 C.c_double(max_point_interpolation_distance), C.c_double(path_segment_length),
                                 C.c_int64(max_points_per_segment), cap, _fp(X), _fp(Y), _fp(acc), _fp(K),
                                 seg.ctypes.data_as(C.POINTER(C.c_int32)), C.byref(n), C.byref(ns),
                                 C.byref(tot)))
    return dict(X=X[:n.value].copy(), Y=Y[:n.value].copy(), acc=acc[:n.value].copy(),
                curvature=K[:n.value].copy(), seg_starts=seg[:ns.value].copy(),
                total_length=float(np.float32(tot.value)))


class DWA:
    """The reference's DWA controller as Python sees it (bindings_control.cpp:221-273, plus the
    Follower / Controller methods it inherits, :66-106): set_current_path, set_current_state,
    compute_velocity_commands(vel, LaserScan | cloud) -> SamplingControlResult, is_goal_reached,
    get_*_cmd, set_resolution. Path interpolation/segmentation, closest-point tracking, the adaptive
    horizon and the tracked segment are reproduced on the host (csrc/kc_dwa.cu); sampling, collision
    checking, cost evaluation and the argmin run on the GPU."""

    def __init__(self, cfg, follower=None):
        self._h = C.c_void_p()
        self.cfg = cfg
        _check(lib().kc_dwa_create(C.byref(cfg), C.byref(follower) if follower is not None else None,
                                   C.byref(self._h)))
        lib().kc_dwa_planner.restype = C.c_void_p
        lib().kc_dwa_planner.argtypes = [C.c_void_p]
        self.planner = Planner._borrow(C.c_void_p(lib().kc_dwa_planner(self._h)), cfg)
        self.info = None
        self._customs = []       # ctypes thunks must outlive the native handle
        self._callback_error = None
        self._path_cache = None

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().kc_dwa_destroy(self._h)
            self._h = C.c_void_p()
            self.planner._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_current_path(self, points, interpolate=True):
        pts = np.asarray(points, dtype=np.float32)
        x, y = _f32(pts[:, 0]), _f32(pts[:, 1])
        _check(lib().kc_dwa_set_current_path(self._h, _fp(x), _fp(y), len(x), 1 if interpolate else 0))

    def clear_current_path(self):
        _check(lib().kc_dwa_clear_current_path(self._h))

    def set_current_state(self, x, y, yaw, speed=0.0):
        _check(lib().kc_dwa_set_current_state(self._h, C.c_double(x), C.c_double(y), C.c_double(yaw),
                                              C.c_double(speed)))

    def set_control_limits(self, vx_max, vy_max, omega_max):
        """Controller::setLinearControlLimits / setAngularControlLimits (max values only)."""
        _check(lib().kc_dwa_set_control_limits(self._h, C.c_double(vx_max), C.c_double(vy_max),
                                               C.c_double(omega_max)))

    def is_goal_reached(self):
        r = C.c_int32(0)
        _check(lib().kc_dwa_is_goal_reached(self._h, C.byref(r)))
        return bool(r.value)

    def has_path(self):
        lib().kc_dwa_has_path.argtypes = [C.c_void_p]
        return bool(lib().kc_dwa_has_path(self._h))

    def get_current_path(self):
        X, Y, K = C.POINTER(C.c_float)(), C.POINTER(C.c_float)(), C.POINTER(C.c_float)()
        n, ns, tot = C.c_int32(0), C.c_int32(0), C.c_float(0)
        _check(lib().kc_dwa_get_path(self._h, C.byref(X), C.byref(Y), C.byref(K), C.byref(n), C.byref(ns),
                                     C.byref(tot)))
        return dict(X=_rows(X, 1, n.value)[0], Y=_rows(Y, 1, n.value)[0], curvature=_rows(K, 1, n.value)[0],
                    n_segments=ns.value, total_length=float(np.float32(tot.value)))

    def _cmd(self):
        c = (C.c_double * 3)()
        _check(lib().kc_dwa_get_command(self._h, c))
        return c[0], c[1], c[2]

    def get_vx_cmd(self):
        return self._cmd()[0]

    def get_vy_cmd(self):
        return self._cmd()[1]

    def get_omega_cmd(self):
        return self._cmd()[2]

    def set_resolution(self, res):
        self.planner.set_resolution(res)

    def add_custom_cost(self, weight, fn):
        """ref: bindings_control.cpp:256-257 add_custom_cost -> DWA::addCustomCost (dwa.cpp:147-150).
        fn(trajectory, reference_path) -> float; trajectory: dict of float32 arrays vx, vy, omega
        [P-1] and x, y [P]; reference_path: dict X, Y, acc, total_length (the interpolated path).
        Called once per admissible trajectory on the calling thread during
        compute_velocity_commands; an exception raised by fn is re-raised from that call."""
        def thunk(tv, pv, _user):
            if self._callback_error is not None:
                return 0.0
            try:
                t, p = tv.contents, pv.contents
                P = t.n_points
                traj = dict(vx=_rows(t.vx, 1, P - 1)[0], vy=_rows(t.vy, 1, P - 1)[0],
                            omega=_rows(t.omega, 1, P - 1)[0], x=_rows(t.x, 1, P)[0], y=_rows(t.y, 1, P)[0])
                if self._path_cache is None:
                    self._path_cache = dict(X=_rows(p.X, 1, p.n)[0], Y=_rows(p.Y, 1, p.n)[0],
                                            acc=_rows(p.acc, 1, p.n)[0],
                                            total_length=float(np.float32(p.total_length)))
                return float(fn(traj, self._path_cache))
            except BaseException as e:  # noqa: BLE001 - must not unwind through the C frames
                self._callback_error = e
                return 0.0
        c_fn = CUSTOM_COST_FN(thunk)
        _check(lib().kc_dwa_add_custom_cost(self._h, C.c_double(weight), c_fn, None))
        self._customs.append(c_fn)

    def clear_custom_costs(self):
        _check(lib().kc_dwa_clear_custom_costs(self._h))
        self._customs.clear()

    def _sensor_call(self, scan_fn, cloud_fn, v, scan, cloud, *tail):
        if scan is not None:
            r, a = _f64(scan[0]), _f64(scan[1])
            if len(r) != len(a):
                raise ValueError("LaserScan ranges and angles must have the same size")
            rc = scan_fn(self._h, _dp(v), _dp(r), _dp(a), len(r), *tail)
        else:
            pts = _f32(cloud if cloud is not None else np.zeros((0, 3), np.float32)).reshape(-1, 3)
            rc = cloud_fn(self._h, _dp(v), _fp(pts), len(pts), *tail)
        return rc

    def compute_velocity_commands(self, vel, scan=None, cloud=None):
        """vel = (vx, vy, omega); scan = (ranges, angles) or cloud = [n x 3] points.
        ref: bindings_control.cpp:239-254 -> DWA::computeVelocityCommandsSet (dwa.h:130-139)."""
        v = _f64(vel)
        res, info = CycleResult(), DwaInfo()
        self._path_cache = None
        rc = self._sensor_call(lib().kc_dwa_compute_scan, lib().kc_dwa_compute_cloud, v, scan, cloud,
                               C.byref(res), C.byref(info))
        if self._callback_error is not None:
            e, self._callback_error = self._callback_error, None
            raise e
        _check(rc)
        self.info = info
        return TrajSearchResult(res)

    def debug_velocity_search(self, vel, scan=None, cloud=None, drop_samples=True):
        """ref: bindings_control.cpp:261-271 -> DWA::debugVelocitySearch<T> (dwa.h:147-165)."""
        v = _f64(vel)
        _check(self._sensor_call(lib().kc_dwa_debug_velocity_search_scan,
                                 lib().kc_dwa_debug_velocity_search_cloud, v, scan, cloud,
                                 1 if drop_samples else 0, None))

    def get_debugging_samples(self, full=False):
        """ref: bindings_control.cpp:260 -> DWA::getDebuggingSamples (dwa.cpp:235-243): (paths_x,
        paths_y), each [n_samples x P]. full=True returns every array of getDebuggingSamplesPure."""
        s = Samples()
        _check(lib().kc_dwa_get_debugging_samples(self._h, C.byref(s)))
        n, P = s.count, s.n_points
        if not full:
            return _rows(s.x, n, P), _rows(s.y, n, P)
        slots = np.ctypeslib.as_array(s.slots, shape=(n,)).copy() if n else np.zeros(0, np.int32)
        return dict(vx=_rows(s.vx, n, P - 1), vy=_rows(s.vy, n, P - 1), omega=_rows(s.omega, n, P - 1),
                    x=_rows(s.x, n, P), y=_rows(s.y, n, P), slots=slots, P=P)


class FleetResult(C.Structure):  # kc_fleet_result
    _fields_ = [("found", C.c_int32), ("cost", C.c_float), ("slot", C.c_int32), ("n_points", C.c_int32),
                ("n_slots", C.c_int32), ("n_admissible", C.c_int32), ("cmd", C.c_double * 3)]


def _fleet_rows(a, R, k, name):
    """[R x k] float64, C-contiguous; ValueError on any other shape."""
    a = np.asarray(a, dtype=np.float64)
    if a.shape != (R, k):
        raise ValueError(f"{name} must have shape ({R}, {k}), got {a.shape}")
    return np.ascontiguousarray(a)


def _fleet_extents(R, offsets, counts):
    offsets, counts = np.asarray(offsets), np.asarray(counts)
    if offsets.shape != (R,) or counts.shape != (R,):
        raise ValueError(f"offsets and counts must have shape ({R},), got {offsets.shape} and {counts.shape}")
    if (offsets < 0).any() or (counts < 0).any():
        raise ValueError("offsets and counts must be non-negative")
    return np.ascontiguousarray(offsets, np.int64), np.ascontiguousarray(counts, np.int32)


def fleet_pack_clouds(R, clouds):
    """clouds: a list of R [n_r x 3] arrays, or the flat form (xyz, offsets, counts) of
    Planner.batch_cloud (a PinnedArray's .array is DMA-ed without a staging copy).
    Returns (xyz [n x 3] float32, offsets int64 [R], counts int32 [R])."""
    if isinstance(clouds, tuple):
        if len(clouds) != 3:
            raise ValueError("flat clouds are (xyz, offsets, counts)")
        xyz = _f32(clouds[0])
        if xyz.size % 3:
            raise ValueError("cloud must hold xyz triples")
        xyz = xyz.reshape(-1, 3)
        offsets, counts = _fleet_extents(R, clouds[1], clouds[2])
        if R and int((offsets + counts).max()) > len(xyz):
            raise ValueError("offsets + counts exceed the cloud")
        return xyz, offsets, counts
    if len(clouds) != R:
        raise ValueError(f"expected {R} clouds, got {len(clouds)}")
    parts = []
    for c in clouds:
        c = np.asarray(c, np.float32)
        if c.size % 3:
            raise ValueError("cloud must hold xyz triples")
        parts.append(c.reshape(-1, 3))
    counts = np.array([len(c) for c in parts], np.int32)
    offsets = np.zeros(R, np.int64)
    offsets[1:] = np.cumsum(counts[:-1])
    xyz = _f32(np.concatenate(parts, axis=0)) if R else np.zeros((0, 3), np.float32)
    return xyz, offsets, counts


def fleet_pack_scans(R, scans):
    """scans: a list of R (ranges, angles) pairs, or the flat form (ranges, angles, offsets, counts).
    Returns (ranges float64, angles float64, offsets int64 [R], counts int32 [R])."""
    if isinstance(scans, tuple):
        if len(scans) != 4:
            raise ValueError("flat scans are (ranges, angles, offsets, counts)")
        r, a = _f64(scans[0]).ravel(), _f64(scans[1]).ravel()
        if len(r) != len(a):
            raise ValueError("LaserScan ranges and angles must have the same size")
        offsets, counts = _fleet_extents(R, scans[2], scans[3])
        if R and int((offsets + counts).max()) > len(r):
            raise ValueError("offsets + counts exceed the scan arrays")
        return r, a, offsets, counts
    if len(scans) != R:
        raise ValueError(f"expected {R} scans, got {len(scans)}")
    rs, angs = [], []
    for sc in scans:
        r, a = np.asarray(sc[0], np.float64).ravel(), np.asarray(sc[1], np.float64).ravel()
        if len(r) != len(a):
            raise ValueError("LaserScan ranges and angles must have the same size")
        rs.append(r)
        angs.append(a)
    counts = np.array([len(r) for r in rs], np.int32)
    offsets = np.zeros(R, np.int64)
    offsets[1:] = np.cumsum(counts[:-1])
    return _f64(np.concatenate(rs)), _f64(np.concatenate(angs)), offsets, counts


class DWAFleet:
    """R DWA controllers stepped together (include/kompass_b200.h, kc_fleet_*). Each robot has its
    own path, state and sensor data; a step returns for every robot what a DWA handle with the same
    configuration and inputs returns, from one batched launch set per chunk of robots. All robots
    share the configuration, the control limits and the planner settings (`planner`)."""

    def __init__(self, cfg, follower=None, n_robots=1):
        n_robots = int(n_robots)
        if n_robots <= 0:
            raise ValueError(f"n_robots must be positive, got {n_robots}")
        self._h = C.c_void_p()
        self.cfg, self.n_robots = cfg, n_robots
        _check(lib().kc_fleet_create(C.byref(cfg), C.byref(follower) if follower is not None else None,
                                     n_robots, C.byref(self._h)))
        self.planner = Planner._borrow(C.c_void_p(lib().kc_fleet_planner(self._h)), cfg)
        self._res = (FleetResult * n_robots)()
        self._info = (DwaInfo * n_robots)()

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().kc_fleet_destroy(self._h)
            self._h = C.c_void_p()
            self.planner._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _robot(self, r):
        r = int(r)
        if not 0 <= r < self.n_robots:
            raise IndexError(f"robot {r} out of range [0, {self.n_robots})")
        return r

    def set_current_path(self, r, points, interpolate=True):
        r = self._robot(r)
        pts = np.asarray(points, dtype=np.float32)
        x, y = _f32(pts[:, 0]), _f32(pts[:, 1])
        _check(lib().kc_fleet_set_current_path(self._h, r, _fp(x), _fp(y), len(x), 1 if interpolate else 0))

    def clear_current_path(self, r):
        _check(lib().kc_fleet_clear_current_path(self._h, self._robot(r)))

    def set_current_states(self, states):
        """states: [R x 4] (x, y, yaw, speed) or [R x 3] (speed 0)."""
        st = np.asarray(states, dtype=np.float64)
        if st.ndim == 2 and st.shape == (self.n_robots, 3):
            st = np.concatenate([st, np.zeros((self.n_robots, 1))], axis=1)
        st = _fleet_rows(st, self.n_robots, 4, "states")
        _check(lib().kc_fleet_set_current_states(self._h, _dp(st)))

    def set_control_limits(self, vx_max, vy_max, omega_max):
        _check(lib().kc_fleet_set_control_limits(self._h, C.c_double(vx_max), C.c_double(vy_max),
                                                 C.c_double(omega_max)))

    def compute_velocity_commands(self, vels, clouds=None, scans=None):
        """One step of every robot. vels: [R x 3]; clouds (list of [n_r x 3] arrays, or (xyz, offsets,
        counts)) or scans (list of (ranges, angles), or (ranges, angles, offsets, counts)). Returns a
        dict of numpy arrays [R]: found, cost, slot, n_points, n_slots, n_admissible, cmd [R x 3], and
        info (record array of the DwaInfo fields)."""
        R = self.n_robots
        v = _fleet_rows(vels, R, 3, "vels")
        if (clouds is None) == (scans is None):
            raise ValueError("pass exactly one of clouds= or scans=")
        if clouds is not None:
            xyz, off, cnt = fleet_pack_clouds(R, clouds)
            rc = lib().kc_fleet_compute_cloud(self._h, _dp(v), _fp(xyz), off.ctypes.data_as(C.POINTER(C.c_int64)),
                                              cnt.ctypes.data_as(C.POINTER(C.c_int32)), self._res, self._info)
        else:
            rr, aa, off, cnt = fleet_pack_scans(R, scans)
            rc = lib().kc_fleet_compute_scan(self._h, _dp(v), _dp(rr), _dp(aa),
                                             off.ctypes.data_as(C.POINTER(C.c_int64)),
                                             cnt.ctypes.data_as(C.POINTER(C.c_int32)), self._res, self._info)
        _check(rc)
        res = np.ctypeslib.as_array(self._res).copy()
        out = {k: res[k].copy() for k in ("found", "cost", "slot", "n_points", "n_slots", "n_admissible")}
        out["found"] = out["found"].astype(bool)
        out["cmd"] = res["cmd"].copy()
        out["info"] = np.ctypeslib.as_array(self._info).copy().view(np.recarray)
        return out

    def get_trajectory(self, r):
        """The winner of robot r's last step, as DWA.compute_velocity_commands returns it."""
        res = CycleResult()
        _check(lib().kc_fleet_get_trajectory(self._h, self._robot(r), C.byref(res)))
        return TrajSearchResult(res)

    def is_goal_reached(self):
        out = np.zeros(self.n_robots, np.int32)
        _check(lib().kc_fleet_is_goal_reached(self._h, out.ctypes.data_as(C.POINTER(C.c_int32))))
        return out.astype(bool)


class CollisionChecker:
    """ref: include/utils/collision_check.h:23-180 (SURVEY section 8 row f4): the collision checker as
    PurePursuit (pure_pursuit.cpp:154-155), the OMPL validity checker (ompl.cpp:95-97) and
    TrajectorySampler::checkStatesFeasibility (trajectory_sampler.cpp:378-408) drive it."""

    def __init__(self, robot_shape, robot_dimensions, sensor_position_body=(0, 0, 0),
                 sensor_rotation_body=(0, 0, 0, 1), octree_resolution=0.01):
        c = CollisionConfig()
        c.robot_shape = int(robot_shape)
        d = list(robot_dimensions) + [0.0] * (3 - len(robot_dimensions))
        c.robot_dims = (C.c_float * 3)(*d)
        c.sensor_position = (C.c_float * 3)(*sensor_position_body)
        c.sensor_rotation = (C.c_float * 4)(*sensor_rotation_body)
        c.octree_resolution = octree_resolution
        self._h = C.c_void_p()
        _check(lib().kc_collision_create(C.byref(c), C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().kc_collision_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def reset_octree_resolution(self, resolution):
        _check(lib().kc_collision_reset_octree_resolution(self._h, C.c_double(resolution)))

    def get_radius(self):
        return float(lib().kc_collision_get_radius(self._h))

    def update_state(self, x, y, yaw):
        _check(lib().kc_collision_update_state(self._h, C.c_double(x), C.c_double(y), C.c_double(yaw)))

    def update_sensor_data(self, scan=None, cloud=None, global_frame=True):
        """updateSensorData<T>: scan = (ranges, angles) or cloud = [n x 3] points."""
        if scan is not None:
            r, a = _f64(scan[0]), _f64(scan[1])
            if len(r) != len(a):
                raise ValueError("LaserScan ranges and angles must have the same size")
            _check(lib().kc_collision_update_scan(self._h, _dp(r), _dp(a), len(r)))
        else:
            pts = _f32(cloud if cloud is not None else np.zeros((0, 3), np.float32)).reshape(-1, 3)
            _check(lib().kc_collision_update_cloud(self._h, _fp(pts), len(pts), 1 if global_frame else 0))

    def check_collisions(self, *args):
        """check_collisions() at the current state, check_collisions((x, y, yaw)) for one state, or
        check_collisions(ranges, angles) = updateSensorData(LaserScan) + check (the three reference
        overloads, collision_check.cpp:149-162,216-246)."""
        if len(args) == 2:
            self.update_sensor_data(scan=(args[0], args[1]))
            args = ()
        if len(args) == 1:
            return bool(self.check_states([args[0]])[1][0])
        r = C.c_int32(0)
        _check(lib().kc_collision_check(self._h, C.byref(r)))
        return bool(r.value)

    def check_states(self, states):
        """Batched checkCollisions(state): states [n x 3] (x, y, yaw) -> (any, uint8 [n])."""
        st = _f64(states).reshape(-1, 3)
        out = np.zeros(len(st), np.uint8)
        anyf = C.c_int32(0)
        _check(lib().kc_collision_check_states(self._h, _dp(st), len(st),
                                               out.ctypes.data_as(C.POINTER(C.c_uint8)), C.byref(anyf)))
        return bool(anyf.value), out


class LocalMapperGPU:
    """ref: include/mapping/local_mapper_gpu.h:12-31 (ctor), :96-116 (scanToGrid overloads);
    bindings_gpu.cpp:13-37 scan_to_grid."""

    def __init__(self, grid_height, grid_width, resolution, laserscan_position, laserscan_orientation,
                 is_pointcloud, scan_size, angle_step, max_height, min_height, range_max,
                 max_points_per_line=32):
        c = MapperConfig()
        c.grid_height, c.grid_width, c.resolution = grid_height, grid_width, resolution
        c.laserscan_position = (C.c_float * 3)(*laserscan_position)
        c.laserscan_orientation = laserscan_orientation
        c.is_pointcloud = 1 if is_pointcloud else 0
        c.scan_size, c.angle_step = scan_size, angle_step
        c.max_height, c.min_height, c.range_max = max_height, min_height, range_max
        c.max_points_per_line = max_points_per_line
        self.H, self.W = grid_height, grid_width
        self._h = C.c_void_p()
        _check(lib().kc_mapper_create(C.byref(c), C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().kc_mapper_destroy(self._h)
            self._h = C.c_void_p()
        for name in ("_grid_buf", "_prob_buf"):
            buf = getattr(self, name, None)
            if buf is not None:
                buf.free()
                setattr(self, name, None)

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def _out(self, name, dtype):
        """Page-locked output buffer owned by this mapper (the DMA lands in it directly), column-major
        [H x W] like the Eigen member the reference returns a reference to."""
        buf = getattr(self, name, None)
        if buf is None:
            buf = PinnedArray((self.W, self.H), dtype)
            setattr(self, name, buf)
        return buf.array

    def scan_to_grid(self, *args, copy=True):
        """scan_to_grid(angles, ranges) or scan_to_grid(data, point_step, row_step, height, width,
        x_offset, y_offset, z_offset) -> int32 grid [H, W] (Eigen::MatrixXi semantics).
        copy=False returns a view of the mapper's own buffer, reused by the next call — what the
        reference binding returns (rv_policy::reference_internal, bindings_gpu.cpp:22-37)."""
        grid = self._out("_grid_buf", np.int32)
        gp = grid.ctypes.data_as(C.POINTER(C.c_int32))
        if len(args) == 2:
            a, r = _f64(args[0]), _f64(args[1])
            _check(lib().kc_mapper_scan_to_grid(self._h, _dp(a), _dp(r), len(a), gp))
        else:
            data, ps, rs, h, w, xo, yo, zo = args
            d = np.ascontiguousarray(data, dtype=np.int8)
            _check(lib().kc_mapper_cloud_to_grid(self._h, d.ctypes.data_as(C.POINTER(C.c_int8)),
                                                 C.c_int64(d.size), ps, rs, h, w, C.c_float(xo),
                                                 C.c_float(yo), C.c_float(zo), gp))
        return grid.copy().T if copy else grid.T

    # -- Bayesian mapper (ref: LocalMapper::scanToGridBaysian / getPreviousGridInCurrentPose) ------
    def set_bayesian_params(self, p_prior=0.5, p_occupied=0.6, p_empty=0.4, range_sure=1.0, wall_size=0.2):
        _check(lib().kc_mapper_set_bayesian_params(self._h, C.c_float(p_prior), C.c_float(p_occupied),
                                                   C.c_float(p_empty), C.c_float(range_sure),
                                                   C.c_float(wall_size)))

    def scan_to_grid_baysian(self, *args, copy=True):
        """scan_to_grid_baysian(angles, ranges) or (data, point_step, row_step, height, width,
        x_offset, y_offset, z_offset) -> (grid int32 [H, W], probabilities float32 [H, W]).
        ref: LocalMapper::scanToGridBaysian, both overloads (local_mapper.cpp:222-264)."""
        grid = self._out("_grid_buf", np.int32)
        prob = self._out("_prob_buf", np.float32)
        gp = grid.ctypes.data_as(C.POINTER(C.c_int32))
        if len(args) == 2:
            a, r = _f64(args[0]), _f64(args[1])
            _check(lib().kc_mapper_scan_to_grid_bayesian(self._h, _dp(a), _dp(r), len(a), gp, _fp(prob)))
        else:
            data, ps, rs, h, w, xo, yo, zo = args
            d = np.ascontiguousarray(data, dtype=np.int8)
            _check(lib().kc_mapper_cloud_to_grid_bayesian(
                self._h, d.ctypes.data_as(C.POINTER(C.c_int8)), C.c_int64(d.size), ps, rs, h, w,
                C.c_float(xo), C.c_float(yo), C.c_float(zo), gp, _fp(prob)))
        return (grid.copy().T, prob.copy().T) if copy else (grid.T, prob.T)

    def get_previous_grid_in_current_pose(self, current_position_in_previous_pose,
                                          current_orientation_in_previous_pose):
        p = current_position_in_previous_pose
        _check(lib().kc_mapper_previous_grid_in_current_pose(self._h, C.c_float(p[0]), C.c_float(p[1]),
                                                             C.c_double(current_orientation_in_previous_pose)))

    def get_previous_grid(self):
        prob = np.zeros((self.W, self.H), np.float32)
        _check(lib().kc_mapper_get_previous_grid(self._h, _fp(prob)))
        return prob.T

    def set_previous_grid(self, prob):
        p = np.ascontiguousarray(np.asarray(prob, np.float32).T)
        assert p.shape == (self.W, self.H)
        _check(lib().kc_mapper_set_previous_grid(self._h, _fp(p)))

    def replay(self, n_iters):
        tot = C.c_float(0)
        _check(lib().kc_mapper_replay(self._h, n_iters, C.byref(tot)))
        return tot.value


def pointcloud_to_laserscan(data, point_step, row_step, height, width, x_offset, y_offset, z_offset,
                            max_range, min_z, max_z, num_bins):
    """ref: include/utils/pointcloud.h:205-259 (num_bins overload)."""
    d = np.ascontiguousarray(data, dtype=np.int8)
    out = np.zeros(num_bins, np.float64)
    _check(lib().kc_pointcloud_to_laserscan(d.ctypes.data_as(C.POINTER(C.c_int8)), C.c_int64(d.size),
                                            point_step, row_step, height, width, x_offset, y_offset,
                                            z_offset, C.c_double(max_range), C.c_double(min_z),
                                            C.c_double(max_z), num_bins, _dp(out)))
    return out


def pointcloud_to_laserscan_step(data, point_step, row_step, height, width, x_offset, y_offset, z_offset,
                                 max_range, min_z, max_z, angle_step):
    """ref: include/utils/pointcloud.h:116-177 (angle_step overload) -> (ranges, angles)."""
    d = np.ascontiguousarray(data, dtype=np.int8)
    cap = int(np.ceil(2.0 * np.pi / angle_step)) + 2 if angle_step > 0 else 1
    ranges, angles, n = np.zeros(cap, np.float64), np.zeros(cap, np.float64), C.c_int32(0)
    _check(lib().kc_pointcloud_to_laserscan_step(
        d.ctypes.data_as(C.POINTER(C.c_int8)), C.c_int64(d.size), point_step, row_step, height, width,
        x_offset, y_offset, z_offset, C.c_double(max_range), C.c_double(min_z), C.c_double(max_z),
        C.c_double(angle_step), cap, _dp(ranges), _dp(angles), C.byref(n)))
    return ranges[:n.value].copy(), angles[:n.value].copy()


class CriticalZoneCheckerGPU:
    """ref: include/utils/critical_zone_check_gpu.h:17-60 (ctor), bindings_gpu.cpp:42-68 check."""

    def __init__(self, input_type, robot_shape, robot_dimensions, sensor_position_body,
                 sensor_rotation_body, critical_angle, critical_distance, slowdown_distance, angles,
                 min_height, max_height, range_max, cloud_field_type=7):
        c = CriticalZoneConfig()
        c.input_type, c.robot_shape = int(input_type), int(robot_shape)
        d = list(robot_dimensions) + [0.0] * (3 - len(robot_dimensions))
        c.robot_dims = (C.c_float * 3)(*d)
        c.sensor_position = (C.c_float * 3)(*sensor_position_body)
        c.sensor_rotation = (C.c_float * 4)(*sensor_rotation_body)
        c.critical_angle, c.critical_distance, c.slowdown_distance = critical_angle, critical_distance, slowdown_distance
        c.min_height, c.max_height, c.range_max = min_height, max_height, range_max
        c.cloud_field_type = cloud_field_type
        a = _f64(angles)
        self.n_angles = len(a)
        self._h = C.c_void_p()
        _check(lib().kc_critical_zone_create(C.byref(c), _dp(a), len(a), C.byref(self._h)))

    def close(self):
        if getattr(self, "_h", None) and self._h.value:
            lib().kc_critical_zone_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def check(self, *args):
        """check(ranges, forward) or check(data, point_step, row_step, height, width, x_offset,
        y_offset, z_offset, forward) -> slowdown factor in [0, 1]."""
        out = C.c_float(0)
        if len(args) == 2:
            r = _f64(args[0])
            _check(lib().kc_critical_zone_check_scan(self._h, _dp(r), len(r), 1 if args[1] else 0,
                                                     C.byref(out)))
        else:
            data, ps, rs, h, w, xo, yo, zo, fwd = args
            d = np.ascontiguousarray(data, dtype=np.int8)
            _check(lib().kc_critical_zone_check_cloud(self._h, d.ctypes.data_as(C.POINTER(C.c_int8)),
                                                      C.c_int64(d.size), ps, rs, h, w, xo, yo, zo,
                                                      1 if fwd else 0, C.byref(out)))
        return float(np.float32(out.value))

    def replay(self, n_iters):
        tot = C.c_float(0)
        _check(lib().kc_critical_zone_replay(self._h, n_iters, C.byref(tot)))
        return tot.value
