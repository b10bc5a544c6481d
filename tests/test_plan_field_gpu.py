"""GPU: cost-to-go fields (rk_plan_cost_to_go through planner.CostMap.cost_to_go, and the closed planning loops with
rk_plan_rollout_field) against the host restatement tests/plan_field_ref.py.  The builder is compared bit for bit with
the float32 Dijkstra on every edge case of the definition, a serpentine maze whose one path crosses many tiles, windows
that are not a multiple of the tile, several maps and 4096 lane windows; two calls give the same bits.  The checks that
need torch.profiler are in test_vdt_instances_field_gpu.py."""
import numpy as np
import pytest
import torch

import plan_field_ref as pf
import plan_map_ref as pmr
import plan_ref as pr
from roboken_fmskf_robot_controller_b200 import _cabi
from roboken_fmskf_robot_controller_b200.planner import CostMap, VehiclePlanner
from roboken_fmskf_robot_controller_b200.vehicle import VehicleBatch
from test_plan_gpu import _u32

import plan_fleet_ref as pfr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _device_build(mp, spec, goals, fw, fh, offs, fm):
    cm = CostMap(torch.from_numpy(np.ascontiguousarray(mp.cells)).to(DEV), (float(mp.x0), float(mp.y0)), pf.CELL, outside=float(mp.outside))
    assert cm.inv_res == np.float32(mp.inv_res)
    ctg = cm.cost_to_go(np.asarray(goals, np.float32), size=(fh, fw), offsets=offs, k_cost=float(spec.k_cost), lethal=float(spec.lethal),
                        field_map=fm)
    torch.cuda.synchronize()
    return ctg.field.cpu().numpy(), ctg.rounds


@pytest.mark.parametrize("name", list(pf.builder_cases()))
def test_builder_bit_exact_on_the_edge_cases(name):
    mp, spec, goals, fw, fh, offs, fm = pf.builder_cases()[name]
    got, _ = _device_build(mp, spec, goals, fw, fh, offs, fm)
    exp = pf.build(mp, spec, goals, fw, fh, offs, fm)
    np.testing.assert_array_equal(got.view(np.uint32), exp.view(np.uint32))


@pytest.mark.parametrize("n", [100, 77])
def test_builder_on_a_serpentine_maze(n):
    """The one path crosses every tile row back and forth: many rounds, and n = 77 is not a multiple of the tile."""
    mp = pmr.host_map(pf.serpentine(n), (0.0, 0.0), 0.0)
    spec = pf.spec_for(pf.CELL, 0.0, np.inf)
    goals = [[0.025, 0.025], [(n - 0.5) * pf.CELL, (n - 0.5) * pf.CELL]]
    got, rounds = _device_build(mp, spec, goals, n, n, None, None)
    exp = pf.build(mp, spec, goals, n, n)
    np.testing.assert_array_equal(got.view(np.uint32), exp.view(np.uint32))
    assert rounds > 2, rounds
    again, rounds2 = _device_build(mp, spec, goals, n, n, None, None)
    np.testing.assert_array_equal(again.view(np.uint32), got.view(np.uint32))
    assert rounds2 == rounds


def test_builder_random_world_several_maps():
    rng = np.random.default_rng(17)
    cells = np.stack([pf._grid(rng, (70, 90), lethal_frac=0.3) for _ in range(2)])
    mp = pmr.host_map(cells, (-1.0, -2.0), 0.0, outside=0.0)
    spec = pf.spec_for(pf.CELL, 1.5, 1.0)
    goals = np.stack([rng.uniform(-1.0, 3.5, 8), rng.uniform(-2.0, 1.5, 8)], axis=1).astype(np.float32)
    offs = rng.integers(-10, 40, (8, 2)).astype(np.int32)
    fm = np.array([0, 1, 1, 0, 2, 0, 1, -3], np.int32)
    got, _ = _device_build(mp, spec, goals, 61, 45, offs, fm)
    np.testing.assert_array_equal(got.view(np.uint32), pf.build(mp, spec, goals, 61, 45, offs, fm).view(np.uint32))


def test_builder_on_4096_lane_windows():
    R = 4096
    wall, cells, origin, _, goals = pmr.wall_world(R)
    mp0, spec, offs, exp = pf.lane_fields(cells, origin, goals, R)
    got, _ = _device_build(mp0, spec, goals, 20, cells.shape[0], offs, None)
    np.testing.assert_array_equal(got.view(np.uint32), exp.view(np.uint32))


@pytest.mark.parametrize("world,mode,steps", [("wall", "cem", 6), ("dead_end", "argmin", 8), ("dead_end", "cem", 5)])
def test_field_loop_equals_the_host_restatement(world, mode, steps):
    sc = pf.WALL_FIELD if world == "wall" else pf.DEAD_END
    make = pmr.wall_world if world == "wall" else pf.dead_end_world
    cem = None if mode == "argmin" else pmr.WALL_CEM
    exp, g, wall, origin, hf = pf.field_loop(sc, make, cem=cem, steps=steps)
    Rw, n_seg, seg_len, P = sc["R"], sc["n_seg"], sc["seg_len"], sc["P"]
    _, cells, origin, start, _ = make(Rw)
    robots = VehicleBatch(Rw, DEV)
    robots.load_state_soa(pfr.start_states(start))
    pl = VehiclePlanner(Rw, sc["S"] if cem is None else cem["S"], n_seg, seg_len, DEV, sigma=sc["sigma"], seed=sc["seed"])
    cm = CostMap(torch.from_numpy(cells).to(DEV), origin, pmr.CELL)
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


def test_planner_field_without_a_map():
    """rollout(field=..., costmap=None): the field term alone, checkpoints every seg_len ticks."""
    sc = pf.DEAD_END
    Rw, n_seg, seg_len = sc["R"], sc["n_seg"], sc["seg_len"]
    _, cells, origin, start, g = pf.dead_end_world(Rw)
    state = pfr.start_states(start)
    robots = VehicleBatch(Rw, DEV)
    robots.load_state_soa(state)
    pl = VehiclePlanner(Rw, 16, n_seg, seg_len, DEV, sigma=sc["sigma"], seed=3)
    cm = CostMap(torch.from_numpy(cells).to(DEV), origin, pmr.CELL)
    offs = np.stack([np.arange(Rw) * 20, np.zeros(Rw, np.int64)], axis=1).astype(np.int32)
    ctg = cm.cost_to_go(g, size=(cells.shape[0], 20), offsets=offs, lethal=1.0, field_of=torch.arange(Rw, dtype=torch.int32, device=DEV))
    ref_np = np.ascontiguousarray(np.broadcast_to(g, (n_seg, Rw, 2)))
    pl.sample(seed=9)
    cost = pl.rollout(robots, torch.from_numpy(ref_np).to(DEV), 0.0, 1.0, 1e-9, field=ctg, w_field=10.0).clone()
    torch.cuda.synchronize()
    mp0, _, _, fields = pf.lane_fields(cells, origin, g, Rw)
    hf = pf.host_field(fields, offs, mp0, 10.0, field_of=np.arange(Rw, dtype=np.int32))
    cand = np.ascontiguousarray(pl.candidates.cpu().numpy()).view(pr.CMD_DT).reshape(n_seg, Rw * 16)
    exp, _, _ = pf.candidate_costs_field(state, Rw, 16, cand, seg_len, ref_np, 0.0, 1.0, 1e-9, np.zeros((n_seg, 0, Rw, 4), np.float32), seg_len,
                                         0.0, None, hf)
    np.testing.assert_array_equal(_u32(cost), exp.view(np.uint32))
