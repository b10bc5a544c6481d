"""GPU: cost-map inflation (rk_plan_inflate through planner.CostMap.inflate) against the host restatement
tests/plan_inflate_ref.py, bit for bit: every edge case of the definition, random worlds whose sizes are no multiple of a
block or a tile, three maps with the largest table, 800 x 800 random walls, two calls, the one-cell grids the map and
field scenarios write by hand, and the narrow-gap planning loop on the inflated map under argmin and CEM, step by step."""
import numpy as np
import pytest
import torch

import plan_field_ref as pf
import plan_fleet_ref as pfr
import plan_inflate_ref as pi
import plan_map_ref as pmr
from roboken_fmskf_robot_controller_b200 import _cabi
from roboken_fmskf_robot_controller_b200.planner import CostMap, VehiclePlanner, inflation_table
from roboken_fmskf_robot_controller_b200.vehicle import VehicleBatch
from test_plan_gpu import _u32

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _device(cells, outside, lethal, table, origin=(0.0, 0.0)):
    cm = CostMap(torch.from_numpy(np.ascontiguousarray(cells, np.float32)).to(DEV), origin, pmr.CELL, outside=float(outside))
    out = cm.inflate(torch.from_numpy(np.ascontiguousarray(table, np.float32)).to(DEV), lethal=float(lethal))
    torch.cuda.synchronize()
    assert (out.x0, out.y0, out.inv_res, out.outside, out.map_of) == (cm.x0, cm.y0, cm.inv_res, cm.outside, cm.map_of)
    return out.cells.cpu().numpy()


def _check(cells, outside, lethal, table):
    got = _device(cells, outside, lethal, table)
    exp = pi.inflate(cells, outside, lethal, table)
    np.testing.assert_array_equal(got.view(np.uint32), exp.view(np.uint32))
    return got


@pytest.mark.parametrize("name", list(pi.cases()))
def test_inflate_bit_exact_on_the_edge_cases(name):
    _check(*pi.cases()[name])


@pytest.mark.parametrize("shape,n_table,outside", [((1, 131, 259), 50, np.inf), ((2, 65, 129), 401, 0.0), ((1, 300, 7), 2000, np.inf),
                                                    ((3, 7, 300), 10, np.inf), ((1, 1, 1000), 626, 0.0), ((1, 1000, 1), 626, np.inf)])
def test_inflate_random_worlds(shape, n_table, outside):
    rng = np.random.default_rng(sum(shape) + n_table)
    cells = pi._random(rng, shape, obst=0.01)
    table = np.sort(rng.uniform(0.0, 4.0, n_table).astype(np.float32))[::-1].copy()
    _check(cells, outside, 1.0, table)


def test_inflate_three_maps_largest_table():
    """n_table = 65536: rmax = 255, wider than the maps, so every obstacle of a map counts."""
    rng = np.random.default_rng(65536)
    cells = np.stack([pi._random(rng, (230, 270), obst=o) for o in (0.0005, 0.0, 0.00005)])
    table = np.linspace(5.0, 0.001, 65536).astype(np.float32)
    for outside in (0.0, np.inf):
        _check(cells, outside, 1.0, table)


def _random_walls(n, rng):
    g = np.zeros((n, n), np.float32)
    for _ in range(n * n // 160):
        h, w = (rng.integers(1, 5), rng.integers(4, 41))[:: 1 if rng.random() < 0.5 else -1]
        y, x = rng.integers(0, n - h), rng.integers(0, n - w)
        g[y:y + h, x:x + w] = 1.0
    return g


@pytest.mark.parametrize("radius_cells", [4, 10, 40])
def test_inflate_800_random_walls_and_twice(radius_cells):
    cells = _random_walls(800, np.random.default_rng(800 + radius_cells))[None]
    table = inflation_table(0.05, 0.2, radius_cells * 0.05 + 1e-9, scaling=3.0, device="cpu").numpy()
    got = _check(cells, np.inf, 1.0, table)
    again = _device(cells, np.inf, 1.0, table)
    np.testing.assert_array_equal(again.view(np.uint32), got.view(np.uint32))


def test_one_cell_grids_are_the_device_inflation():
    for world in (pmr.wall_world, pf.dead_end_world):
        wall, cells, _, _, _ = world(37)
        got = _device(wall.astype(np.float32), 0.0, 1.0, np.ones(3, np.float32))
        np.testing.assert_array_equal(got[0].view(np.uint32), cells.view(np.uint32))


@pytest.mark.parametrize("mode,steps", [("argmin", 8), ("cem", 5)])
def test_narrow_gap_loop_equals_the_port(mode, steps):
    sc = dict(pf.WALL_FIELD, steps=steps)
    cem = None if mode == "argmin" else pmr.WALL_CEM
    exp, g, wall, origin, hf = pf.field_loop(sc, pi.narrow_gap_world, cem=cem, steps=steps)
    Rw, n_seg, seg_len, P = sc["R"], sc["n_seg"], sc["seg_len"], sc["P"]
    _, cells, _, start, _ = pi.narrow_gap_world(Rw)
    raw = CostMap(torch.from_numpy(wall.astype(np.float32)).to(DEV), origin, pmr.CELL)
    cm = raw.inflate(inflation_table(pmr.CELL, pi.INSCRIBED, pi.RADIUS, pi.SCALING, pi.PEAK, device=DEV), lethal=1.0)
    np.testing.assert_array_equal(_u32(cm.cells).reshape(cells.shape), cells.view(np.uint32))
    robots = VehicleBatch(Rw, DEV)
    robots.load_state_soa(pfr.start_states(start))
    pl = VehiclePlanner(Rw, sc["S"] if cem is None else cem["S"], n_seg, seg_len, DEV, sigma=sc["sigma"], seed=sc["seed"])
    offs = np.stack([np.arange(Rw) * 20, np.zeros(Rw, np.int64)], axis=1).astype(np.int32)
    ctg = cm.cost_to_go(g, size=(cells.shape[0], 20), offsets=offs, lethal=1.0, field_of=torch.arange(Rw, dtype=torch.int32, device=DEV))
    torch.cuda.synchronize()
    np.testing.assert_array_equal(_u32(ctg.field).reshape(hf.field.shape), hf.field.view(np.uint32))
    ref = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(g, (n_seg, Rw, 2)))).to(DEV)
    w = (sc["w_pos"], sc["w_goal"], sc["w_cur"])
    kw = dict(shift=0, check_period=P, costmap=cm, w_map=sc["w_map"], field=ctg, w_field=sc["w_field"])
    for it in range(steps):
        if cem is None:
            pl.plan(robots, ref, *w, lam=0.0, seed=sc["seed"] + it, **kw)
        else:
            pl.plan_cem(robots, ref, *w, cem["iters"], cem["elite"], cem["alpha"], cem["sigma_min"], seed=sc["seed"] + it, **kw)
        robots.rollout(seg_len, sensor_mode=_cabi.RK_SENSOR_PLANT, cmd=pl.first_command(), seg_len=seg_len)
        torch.cuda.synchronize()
        costs, ebest, estate, _ = exp[it]
        np.testing.assert_array_equal(_u32(pl.cost), costs[-1].view(np.uint32), err_msg=f"step {it}: costs")
        np.testing.assert_array_equal(pl.best.cpu().numpy(), ebest, err_msg=f"step {it}: best")
        np.testing.assert_array_equal(_u32(robots.state), estate, err_msg=f"step {it}: executed states")
