"""CPU: cost-map inflation (rk_plan_inflate) -- the two host restatements of the distance agree on every edge case of the
definition and reproduce the one-cell grids the map and field scenarios write by hand, inflation_table's values worked
out by hand, the struct layout, every argument error and the no-device error, and on the port the narrow-gap scenario:
a point robot takes the gap straight ahead and its body overlaps a wall, while on the inflated map no body does."""
import ctypes as C
import math

import numpy as np
import pytest

import plan_field_ref as pf
import plan_inflate_ref as pi
import plan_map_ref as pmr
import plan_ref as pr
import roboken_fmskf_robot_controller_b200 as rk
from roboken_fmskf_robot_controller_b200 import _cabi, build
from roboken_fmskf_robot_controller_b200.planner import inflation_table
from test_plan_fleet_cpu import _buf
from test_plan_map_cpu import _map

f32 = np.float32
INF = np.inf


@pytest.fixture(scope="module")
def lib():
    build.build()
    return rk.load()


@pytest.mark.parametrize("name", list(pi.cases()))
def test_brute_force_and_edt_agree(name):
    cells, outside, lethal, table = pi.cases()[name]
    a = pi.d2_brute(cells, outside, lethal)
    b = pi.d2_edt(cells, outside, lethal)
    np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(pi.apply(cells, a, table).view(np.uint32), pi.apply(cells, b, table).view(np.uint32))


def test_definition_by_hand():
    c = np.zeros((1, 5, 6), np.float32)
    c[0, 2, 3] = 1.0
    d2 = pi.d2_brute(c, 0.0, 1.0)[0]
    assert d2[2, 3] == 0 and d2[2, 4] == 1 and d2[3, 4] == 2 and d2[0, 0] == 4 + 9
    # off the grid: the axial distance to the ring, only when outside >= lethal
    e = pi.d2_brute(np.zeros((1, 5, 6), np.float32), 1.0, 1.0)[0]
    assert e[0, 0] == 1 and e[2, 2] == 9 and e[2, 3] == 9 and e[4, 5] == 1
    assert (pi.d2_brute(np.zeros((1, 5, 6), np.float32), 0.999, 1.0) == pi.NONE).all()
    # the output rule: larger wins, NaN takes the table, signed zeros keep the source, beyond the table the source
    cells = np.array([[[2.0, -0.0, np.nan, 0.5, 0.5]]], np.float32)
    d2 = np.array([[[0, 1, 1, 2, 3]]])
    out = pi.apply(cells, d2, np.array([1.0, 0.0, 3.0], np.float32))[0, 0]
    assert out[0] == 2.0 and out[1].view(np.uint32) == f32(-0.0).view(np.uint32) and out[2] == 0.0 and out[3] == 3.0 and out[4] == 0.5


def test_one_cell_dilations_are_inflations():
    """The raw wall (1.0 on wall cells), lethal 1, outside 0 and the table [1, 1, 1]: Euclidean d2 <= 2 is the 8-neighbour
    dilation that plan_map_ref.wall_world and plan_field_ref.dead_end_world write by hand."""
    for world in (pmr.wall_world, pf.dead_end_world):
        wall, cells, _, _, _ = world(5)
        got = pi.inflate(wall.astype(np.float32), 0.0, 1.0, np.ones(3, np.float32))[0]
        np.testing.assert_array_equal(got.view(np.uint32), cells.view(np.uint32))


def test_inflation_table_by_hand():
    t = inflation_table(0.05, 0.11, 0.2, scaling=4.0, peak=0.5, lethal=254.0, device="cpu").numpy()
    # d = sqrt(d2) * 0.05 <= 0.2 up to d2 = 16 (4 * 0.05 is 0.2 in float64); lethal up to d2 = 4 (2.2 cells)
    assert t.dtype == np.float32 and len(t) == 17
    assert (t[:5] == f32(254.0)).all()
    for d2 in range(5, 17):
        assert t[d2] == f32(0.5 * math.exp(-4.0 * (math.sqrt(d2) * 0.05 - 0.11))), d2
    t = inflation_table(0.05, 0.0, 0.0, device="cpu").numpy()
    assert len(t) == 1 and t[0] == INF  # d = 0 <= inscribed
    t = inflation_table(0.1, 0.05, 0.35, device="cpu").numpy()  # scaling 0: a flat peak out to the radius
    assert len(t) == 13 and t[0] == INF and (t[1:] == f32(1.0)).all()
    t = inflation_table(1.0, 0.5, 255.5, device="cpu")
    assert t.numel() == 65281  # d2 <= 255.5^2: the largest radius the entry takes is 255 cells and a bit
    with pytest.raises(AssertionError):
        inflation_table(1.0, 0.5, 256.0, device="cpu")
    with pytest.raises(AssertionError):
        inflation_table(0.05, 0.1, -0.01, device="cpu")
    np.testing.assert_array_equal(pi.table(), inflation_table(pmr.CELL, pi.INSCRIBED, pi.RADIUS, pi.SCALING, pi.PEAK, device="cpu").numpy())


def test_lazy_exports():
    assert rk.inflation_table is inflation_table
    assert rk.CostMap is rk.planner.CostMap


def test_struct_layout():
    assert C.sizeof(_cabi.PlanInflate) == 16
    assert [_cabi.PlanInflate.__dict__[n].offset for n in ("d_table", "n_table", "lethal")] == [0, 8, 12]


def _spec(d_table, n=3, lethal=1.0):
    s = _cabi.PlanInflate()
    s.d_table, s.n_table, s.lethal = d_table, n, lethal
    return s


def test_inflate_argument_errors(lib):
    keep, a = _buf(1 << 14)
    base = a.value
    cells, table, dst, work = base, base + 1024, base + 2048, base + 4096  # a 4 x 4 map: 64 bytes of cells, 32 of work
    inflate, work_bytes = lib.rk_plan_inflate, lib.rk_plan_inflate_work_bytes

    def call(mp=_map(cells), spec=_spec(table), d=dst, w=work):
        return inflate(None if mp is None else C.byref(mp), None if spec is None else C.byref(spec), d, w, None)

    bad = {
        "map NULL": dict(mp=None),
        "map n_maps 0": dict(mp=_map(cells, n=0)),
        "map height 0": dict(mp=_map(cells, h=0)),
        "map width > 2^24": dict(mp=_map(cells, w=(1 << 24) + 1)),
        "map n_maps * height * width >= 2^31": dict(mp=_map(cells, n=2, w=1 << 15, h=1 << 15)),
        "map inv_res 0": dict(mp=_map(cells, inv=0.0)),
        "map y0 NaN": dict(mp=_map(cells, y0=np.nan)),
        "map outside NaN": dict(mp=_map(cells, outside=np.nan)),
        "map d_cells NULL": dict(mp=_map(None)),
        "map d_cells misaligned": dict(mp=_map(cells + 2)),
        "map d_map_of misaligned": dict(mp=_map(cells, base + 6)),
        "spec NULL": dict(spec=None),
        "n_table 0": dict(spec=_spec(table, n=0)),
        "n_table < 0": dict(spec=_spec(table, n=-1)),
        "n_table 65537": dict(spec=_spec(table, n=65537)),
        "lethal NaN": dict(spec=_spec(table, lethal=np.nan)),
        "lethal 0": dict(spec=_spec(table, lethal=0.0)),
        "lethal -0": dict(spec=_spec(table, lethal=-0.0)),
        "lethal -inf": dict(spec=_spec(table, lethal=-INF)),
        "d_table NULL": dict(spec=_spec(None)),
        "d_table misaligned": dict(spec=_spec(table + 2)),
        "d_dst NULL": dict(d=None),
        "d_dst misaligned": dict(d=dst + 1),
        "d_work NULL": dict(w=None),
        "d_work misaligned": dict(w=work + 2),
        "d_dst overlaps the cells": dict(d=cells + 60),
        "d_dst is the cells": dict(d=cells),
        "d_dst overlaps d_work": dict(d=work - 60),
        "d_dst overlaps the table": dict(d=table + 8),
        "d_work overlaps the cells": dict(w=cells + 32),
        "d_work overlaps the table": dict(spec=_spec(work + 28, n=2)),
    }
    for what, kw in bad.items():
        assert call(**kw) == 1, what
        assert b"rk_plan_inflate" in lib.rk_last_error(), f"{what}: no message"
    assert work_bytes(1, 4, 4) == 32 and work_bytes(1, 3, 1) == 8 and work_bytes(3, 7, 5) == 212
    for bad_size in ((0, 4, 4), (1, 0, 4), (1, 4, -1), (1, (1 << 24) + 1, 1), (2, 1 << 15, 1 << 15)):
        assert work_bytes(*bad_size) == 0, bad_size


def test_inflate_fails_without_a_device(lib):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    keep, a = _buf(1 << 14)
    assert lib.rk_plan_inflate(C.byref(_map(a.value)), C.byref(_spec(a.value + 1024, n=3, lethal=INF)), a.value + 2048, a.value + 4096, None) == 2
    assert b"no CPU fallback" in lib.rk_last_error()


# The narrow-gap scenario on the port (plan_field_ref.field_loop with each robot's lane field).  Observed: the point
# robots cross the wall band within 10 mm of their lane's line and come 23 - 86 mm from a wall cell; on the inflated map
# they cross through the wide gaps on the lane boundaries, at least 0.25 m from every wall cell, and end 51 - 89 mm from
# their goals.
NARROW = dict(pf.WALL_FIELD, steps=60)


def _play(world, cem):
    out, g, wall, origin, _ = pf.field_loop(NARROW, world, cem=cem)
    pos = np.concatenate([o[3] for o in out], axis=0)  # [ticks, R, 2]
    return pi.wall_clearance(pos, wall, origin), pos, pr.distances(out[-1][2], NARROW["R"], g)


@pytest.mark.parametrize("cem", [None, pmr.WALL_CEM], ids=["argmin", "cem"])
def test_point_robot_takes_the_narrow_gap(cem):
    clear, pos, _ = _play(pi.point_robot_world, cem)
    crossing = np.abs(pos[..., 1]).argmin(axis=0)
    x = pos[crossing, np.arange(NARROW["R"]), 0]
    assert (np.abs(x - np.arange(NARROW["R"])) < 0.1).all(), f"the robots must cross on their lane's line: {x}"
    assert (clear.min(axis=0) < pi.BODY_M).all(), f"every body must overlap a wall: {clear.min(axis=0)}"


@pytest.mark.parametrize("cem", [None, pmr.WALL_CEM], ids=["argmin", "cem"])
def test_inflated_map_keeps_every_body_clear(cem):
    clear, _, d = _play(pi.narrow_gap_world, cem)
    assert clear.min() >= pi.BODY_M, f"least clearance per robot: {clear.min(axis=0)}"
    assert (d < 0.1).all(), f"distances to the goals: {d}"
