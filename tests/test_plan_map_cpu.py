"""CPU: cost maps (rk_plan_rollout_map) -- the cell lookup's edge cases on the host restatement (tests/plan_map_ref.py),
its equality with the moving-disc cost for an all-zero grid, the new argument errors, and the wall scenario on the port:
without the map robots drive into the wall, with it no executed tick lies in a wall cell and the robots reach their
goals through the gap."""
import ctypes as C

import numpy as np
import pytest

import plan_fleet_ref as pfr
import plan_map_ref as pmr
import plan_ref as pr
import roboken_fmskf_robot_controller_b200 as rk
from roboken_fmskf_robot_controller_b200 import _cabi, build
from test_plan_fleet_cpu import _buf, _obst, _static, _trace

f32 = np.float32
INF = np.inf


@pytest.fixture(scope="module")
def lib():
    build.build()
    return rk.load()


def _one(x, y, cells, k=0, x0=0.0, y0=0.0, inv_res=1.0, outside=7.0, w_map=1.0, O=0.0):
    """O after one map term at one point (a map of cells [n_maps, H, W] and map index k for that one candidate)."""
    mp = pmr.HostMap(np.asarray(cells, dtype=np.float32), None, f32(x0), f32(y0), f32(inv_res), f32(outside), f32(w_map))
    return pmr.map_term(np.array([O], dtype=np.float32), np.array([x], dtype=np.float32), np.array([y], dtype=np.float32), mp,
                        np.array([k]))[0]


def test_lookup_edges():
    cells = np.arange(1, 13, dtype=np.float32).reshape(1, 3, 4)  # cell (ix, iy) = 1 + iy*4 + ix
    x0, y0 = f32(-0.5), f32(0.25)
    kw = dict(x0=x0, y0=y0, inv_res=2.0, outside=100.0)
    assert _one(x0, y0, cells, **kw) == 1  # x exactly x0, y exactly y0: cell (0, 0)
    below = np.nextafter(f32(4.0), f32(0)) / f32(2.0) + x0  # u just below width
    u = (f32(below) - x0) * f32(2.0)
    assert u < 4 and _one(below, y0, cells, **kw) == 4
    assert _one(x0 + f32(2.0), y0, cells, **kw) == 100  # u == width: off the grid
    assert _one(np.nextafter(x0, f32(-1)), y0, cells, **kw) == 100  # u < 0
    assert _one(x0, y0 + f32(1.5), cells, **kw) == 100  # v == height
    assert _one(x0 + f32(1.0), y0 + f32(1.0), cells, **kw) == 1 + 2 * 4 + 2
    assert _one(np.nan, y0, cells, **kw) == 100 and _one(x0, np.nan, cells, **kw) == 100  # NaN reads outside
    assert _one(np.nan, y0, cells, **dict(kw, outside=INF)) == INF


def test_cells_that_add_nothing_and_hard_walls():
    for c in (np.nan, -1.0, 0.0, -0.0, -INF):
        for w in (3.0, INF):
            got = _one(0.5, 0.5, [[[c]]], w_map=w, O=2.0)
            assert got == f32(2.0), (c, w)
    assert _one(0.5, 0.5, [[[INF]]], w_map=3.0) == INF
    assert _one(0.5, 0.5, [[[1e-30]]], w_map=INF) == INF
    assert _one(0.5, 0.5, [[[0.0]]], w_map=INF, O=1.0) == 1  # never 0 * inf
    assert _one(5.0, 0.5, [[[0.0]]], outside=INF, w_map=2.0) == INF  # +inf outside
    assert _one(5.0, 0.5, [[[0.0]]], outside=-INF, w_map=INF) == 0
    assert _one(0.5, 0.5, [[[0.25]]], w_map=3.0, O=1.0) == f32(1.0) + f32(3.0) * f32(0.25)


def test_map_index_out_of_range_adds_nothing():
    cells = np.ones((2, 1, 1), dtype=np.float32)
    cells[1] = 5.0
    for k, exp in ((-1, 0.0), (2, 0.0), (1 << 30, 0.0), (0, 1.0), (1, 5.0)):
        assert _one(0.5, 0.5, cells, k=k, outside=9.0) == exp, k
    assert _one(7.0, 0.5, cells, k=-1, outside=INF) == 0  # not even `outside`


@pytest.mark.parametrize("P", [1, 4, 12])
@pytest.mark.parametrize("m", [0, 3])
def test_all_zero_grid_is_the_moving_cost(P, m):
    rng = np.random.default_rng(20 * P + m)
    R, S, K = 6, 5, 24
    tr = _trace(rng, K, R * S)
    obs = np.ascontiguousarray(np.broadcast_to(_static(rng, m, R), (K // P, m, R, 4)))
    mp = pmr.HostMap(np.zeros((2, 8, 8), np.float32), np.array([0, 1, -1, 2, 1, 0], np.int32), f32(-0.2), f32(-0.2), f32(20.0), f32(0.0),
                     f32(INF))
    got = pmr.map_obstacle_cost(tr, obs, S, P, 7.0, mp)
    np.testing.assert_array_equal(got.view(np.uint32), pfr.moving_obstacle_cost(tr, obs, S, P, 7.0).view(np.uint32))


def test_discs_and_map_share_one_accumulator():
    """Discs first, then the map, checkpoint by checkpoint, into one O: not the sum of two separate sums."""
    R, S, K, P = 1, 1, 2, 1
    tr = np.zeros((K, 16, 1), dtype=np.uint32)  # the candidate sits at (0, 0) at both checkpoints
    obs = np.zeros((K, 1, 1, 4), dtype=np.float32)
    obs[:, 0, 0, 2] = 1.0  # pen = 1 at each checkpoint, w_obst = 1
    mp = pmr.HostMap(np.full((1, 1, 1), 2.0 ** -23, np.float32), None, f32(-1), f32(-1), f32(0.5), f32(0), f32(1.0))
    got = pmr.map_obstacle_cost(tr, obs, S, P, 1.0, mp)
    inter = f32(0)
    for _ in range(K):
        inter = (inter + f32(1)) + f32(2.0 ** -23)
    sep = f32(2) + (f32(2.0 ** -23) + f32(2.0 ** -23))
    assert got[0] == inter and inter != sep


def _map(d_cells, d_map_of=None, n=1, w=4, h=4, x0=0.0, y0=0.0, inv=20.0, outside=INF, w_map=1.0):
    m = _cabi.PlanMap()
    m.d_cells, m.d_map_of, m.n_maps, m.width, m.height = d_cells, d_map_of, n, w, h
    m.x0, m.y0, m.inv_res, m.outside, m.w_map = x0, y0, inv, outside, w_map
    return m


def test_map_argument_errors(lib):
    p = rk.default_params()
    c = _cabi.PlanCost()
    keep, a = _buf(4096)
    c.d_ref = a.value
    roll = lib.rk_plan_rollout_map
    ok_o = _obst(a.value, 0, 5, 1.0)
    cells = a.value + 1024
    bad = {
        "d_cells NULL": _map(None),
        "d_cells misaligned": _map(cells + 2),
        "d_map_of misaligned": _map(cells, a.value + 2050),
        "n_maps 0": _map(cells, n=0),
        "width 0": _map(cells, w=0),
        "height < 0": _map(cells, h=-3),
        "width > 2^24": _map(cells, w=(1 << 24) + 1),
        "height > 2^24": _map(cells, h=(1 << 24) + 1),
        "n_maps * height * width >= 2^31": _map(cells, n=2, w=1 << 15, h=1 << 15),
        "inv_res 0": _map(cells, inv=0.0),
        "inv_res < 0": _map(cells, inv=-20.0),
        "inv_res inf": _map(cells, inv=INF),
        "inv_res NaN": _map(cells, inv=np.nan),
        "x0 inf": _map(cells, x0=-INF),
        "y0 NaN": _map(cells, y0=np.nan),
        "outside NaN": _map(cells, outside=np.nan),
        "w_map < 0": _map(cells, w_map=-1.0),
        "w_map NaN": _map(cells, w_map=np.nan),
    }
    for what, mp in bad.items():
        assert roll(C.byref(p), a, 1, 4, a, 2, 10, C.byref(c), C.byref(ok_o), C.byref(mp), None, a, None) == 1, what
        assert b"rk_plan_rollout_map" in lib.rk_last_error(), f"{what}: no message"
    good = _map(cells, a.value + 2048, outside=INF, w_map=INF)
    moving_bad = {
        "obst NULL": (None, None),
        "m < 0": (_obst(a.value, -1, 10, 1.0), None),
        "P < 1": (_obst(a.value, 0, 0, 1.0), None),
        "seg_len % P != 0": (_obst(a.value, 0, 3, 1.0), None),
        "w_obst NaN": (_obst(a.value, 0, 5, float("nan")), None),
        "m > 0, d_obs misaligned": (_obst(a.value + 8, 2, 5, 1.0), None),
        "d_path misaligned": (ok_o, a.value + 4),
    }
    for what, (o, path) in moving_bad.items():
        assert roll(C.byref(p), a, 1, 4, a, 2, 10, C.byref(c), None if o is None else C.byref(o), C.byref(good), path, a, None) == 1, what
        assert b"rk_plan_rollout_map" in lib.rk_last_error(), f"{what}: no message"
    assert roll(None, a, 1, 4, a, 2, 10, C.byref(c), C.byref(ok_o), C.byref(good), None, a, None) == 1
    assert roll(C.byref(p), a, -1, 4, a, 2, 10, C.byref(c), C.byref(ok_o), C.byref(good), None, a, None) == 1
    # R == 0 is a no-op, with or without a map (the scalar checks still apply)
    assert roll(C.byref(p), None, 0, 4, None, 2, 10, C.byref(c), C.byref(ok_o), C.byref(_map(None)), None, None, None) == 0
    assert roll(C.byref(p), None, 0, 4, None, 2, 10, C.byref(c), C.byref(ok_o), None, None, None, None) == 0
    assert roll(C.byref(p), None, 0, 4, None, 2, 10, C.byref(c), C.byref(ok_o), C.byref(_map(cells, w_map=-1.0)), None, None, None) == 1


def test_map_entry_fails_without_a_device(lib):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    p = rk.default_params()
    c = _cabi.PlanCost()
    keep, a = _buf(1 << 16)
    c.d_ref = a.value
    mp = _map(a.value + 40960)
    assert lib.rk_plan_rollout_map(C.byref(p), a, 1, 4, C.c_void_p(a.value + 32768), 2, 10, C.byref(c), C.byref(_obst(None, 0, 5, 0.0)),
                                   C.byref(mp), None, a, None) == 2
    assert b"no CPU fallback" in lib.rk_last_error()


# The wall scenario (plan_map_ref.WALL) on the port.  Observed: without the map every robot drives into its wall within 12
# steps; with it no executed tick lies in a wall cell, and after 40 argmin steps the robots end 17 - 57 mm from their
# goals.  Under CEM (plan_map_ref.WALL_CEM) no robot enters a wall either, but the elite refit can stall in front of the
# wall, where every sideways move first takes a robot farther from a goal straight behind it: robot 3 stays 0.55 m away.
WALL_GOAL_TOLERANCE_M = 0.1


def _executed(out):
    return np.concatenate([o[3] for o in out], axis=0)


def test_wall_entered_without_the_map():
    out, g, wall, origin = pmr.wall_loop(use_map=False, steps=12)
    hit = pmr.in_wall(_executed(out), wall, origin).any(axis=0)
    assert hit.all(), f"robots that entered a wall cell without the map: {hit}; the scenario tests nothing"


def test_wall_avoided_and_goals_reached_with_the_map():
    out, g, wall, origin = pmr.wall_loop(steps=40)
    pos = _executed(out)
    assert not pmr.in_wall(pos, wall, origin).any(), "an executed tick lies in a wall cell"
    d = pr.distances(out[-1][2], pmr.WALL["R"], g)
    assert (d < WALL_GOAL_TOLERANCE_M).all(), f"distances to the goals: {d}"
    assert (pos[-1, :, 1] > 0.05).all(), "every robot ends north of the wall"


def test_wall_avoided_under_cem():
    out, g, wall, origin = pmr.wall_loop(cem=pmr.WALL_CEM, steps=40)
    assert not pmr.in_wall(_executed(out), wall, origin).any(), "an executed tick lies in a wall cell"
    d = pr.distances(out[-1][2], pmr.WALL["R"], g)
    assert (d < WALL_GOAL_TOLERANCE_M).sum() >= 3, f"distances to the goals: {d}"
