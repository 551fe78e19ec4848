"""CPU-side checks of the multi-robot DWA controller (kc_fleet_* / DWAFleet): arguments are rejected
before any device use, creation fails loudly without a device, and the Python front-end checks shapes
and sensor layouts before it calls the library."""
import ctypes as C

import numpy as np
import pytest


def _create(pkg, cfg, n):
    h = C.c_void_p()
    rc = pkg.lib().kc_fleet_create(C.byref(cfg) if cfg is not None else None, None, n, C.byref(h))
    return rc, h


def test_create_fails_without_device(pkg):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    rc, h = _create(pkg, pkg.planner_config(), 4)
    assert rc == pkg.KC_ERR_CUDA and not h.value
    with pytest.raises(pkg.KompassB200Error, match="no usable CUDA device"):
        pkg.DWAFleet(pkg.planner_config(), n_robots=4)


@pytest.mark.parametrize("n", [0, -3])
def test_bad_robot_count_and_null_config(pkg, n):
    rc, h = _create(pkg, pkg.planner_config(), n)
    assert rc == pkg.KC_ERR_INVALID_ARG and not h.value
    assert b"n_robots" in pkg.lib().kc_last_error()
    rc, h = _create(pkg, None, 4)
    assert rc == pkg.KC_ERR_INVALID_ARG and b"null config" in pkg.lib().kc_last_error()
    with pytest.raises(ValueError, match="n_robots"):
        pkg.DWAFleet(pkg.planner_config(), n_robots=n)


def test_null_handle_calls(pkg):
    L = pkg.lib()
    assert L.kc_fleet_set_control_limits(None, C.c_double(1), C.c_double(1), C.c_double(1)) == pkg.KC_ERR_INVALID_ARG
    assert L.kc_fleet_is_goal_reached(None, None) == pkg.KC_ERR_INVALID_ARG
    assert L.kc_fleet_get_trajectory(None, 0, None) == pkg.KC_ERR_INVALID_ARG
    assert not L.kc_fleet_planner(None)


def test_pack_clouds(pkg):
    a, b = np.ones((4, 3), np.float32), np.zeros((0, 3))
    xyz, off, cnt = pkg.fleet_pack_clouds(2, [a, b])
    assert xyz.shape == (4, 3) and xyz.dtype == np.float32
    assert off.tolist() == [0, 4] and cnt.tolist() == [4, 0]
    flat = np.arange(30, dtype=np.float32).reshape(10, 3)
    xyz, off, cnt = pkg.fleet_pack_clouds(3, (flat, [0, 0, 6], [3, 3, 4]))
    assert np.shares_memory(xyz, flat) and off.dtype == np.int64 and cnt.dtype == np.int32
    with pytest.raises(ValueError, match="expected 3 clouds"):
        pkg.fleet_pack_clouds(3, [a, b])
    with pytest.raises(ValueError, match="xyz triples"):
        pkg.fleet_pack_clouds(1, [np.ones(4)])
    with pytest.raises(ValueError, match="shape"):
        pkg.fleet_pack_clouds(3, (flat, [0, 0], [1, 1]))
    with pytest.raises(ValueError, match="non-negative"):
        pkg.fleet_pack_clouds(2, (flat, [0, -1], [1, 1]))
    with pytest.raises(ValueError, match="exceed"):
        pkg.fleet_pack_clouds(2, (flat, [0, 8], [1, 3]))


def test_pack_scans(pkg):
    r, a = np.ones(5), np.linspace(0, 1, 5)
    rr, aa, off, cnt = pkg.fleet_pack_scans(2, [(r, a), (r[:2], a[:2])])
    assert len(rr) == len(aa) == 7 and off.tolist() == [0, 5] and cnt.tolist() == [5, 2]
    with pytest.raises(ValueError, match="same size"):
        pkg.fleet_pack_scans(1, [(r, a[:3])])
    with pytest.raises(ValueError, match="same size"):
        pkg.fleet_pack_scans(1, (r, a[:3], [0], [3]))
    with pytest.raises(ValueError, match="expected 2 scans"):
        pkg.fleet_pack_scans(2, [(r, a)])
    with pytest.raises(ValueError, match="exceed"):
        pkg.fleet_pack_scans(2, (r, a, [0, 4], [2, 2]))


def test_velocity_and_state_shapes(pkg):
    fleet = pkg.DWAFleet.__new__(pkg.DWAFleet)  # argument checks only: no native handle
    fleet.n_robots, fleet._h = 3, C.c_void_p()
    with pytest.raises(ValueError, match=r"vels must have shape \(3, 3\)"):
        fleet.compute_velocity_commands(np.zeros((3, 2)), clouds=[np.zeros((0, 3))] * 3)
    with pytest.raises(ValueError, match="exactly one"):
        fleet.compute_velocity_commands(np.zeros((3, 3)))
    with pytest.raises(ValueError, match=r"states must have shape \(3, 4\)"):
        fleet.set_current_states(np.zeros((2, 4)))
    with pytest.raises(IndexError):
        fleet.set_current_path(3, [(0, 0), (1, 0)])
    with pytest.raises(IndexError):
        fleet.get_trajectory(-1)
