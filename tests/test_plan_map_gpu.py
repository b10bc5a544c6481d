"""GPU: cost maps (rk_plan_rollout_map, planner.CostMap) against the host restatement tests/plan_map_ref.py -- the
planner's static-disc expansion, the closed wall loop under argmin and CEM, and a fleet step with peer discs and a map
together.  The checks that need torch.profiler (every compiled kObstMoving instantiation, and the equality with
rk_plan_rollout_moving without a map) are in test_vdt_instances_map_gpu.py, next to the instance matrix."""
import ctypes as C

import numpy as np
import pytest
import torch

import plan_fleet_ref as pfr
import plan_map_ref as pmr
import plan_ref as pr
import roboken_fmskf_robot_controller_b200 as rk
from roboken_fmskf_robot_controller_b200 import _cabi, layout, streams
from roboken_fmskf_robot_controller_b200.planner import CostMap, VehiclePlanner, fleet_peers
from roboken_fmskf_robot_controller_b200.vehicle import VehicleBatch
from test_plan_fleet_cpu import FLEET
from test_plan_fleet_gpu import _moving_discs
from test_plan_gpu import _cells, _u32
from test_plan_obst_gpu import N_SEG, R, S, SEG_LEN, W, _case

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
W_OBST = 3.0e3


def _table(src, n_ck, m, seed):
    """test_plan_fleet_gpu._moving_discs, or an empty [n_ck, 0, R, 4] table for m = 0."""
    return _moving_discs(src, n_ck, m, seed) if m else np.zeros((n_ck, 0, R, 4), dtype=np.float32)


def _world(src, n_maps, outside, seed):
    """Cost grids float32 [n_maps, 40, 24] of 5 mm cells over x in [-0.1, 0.02) + the robots' mean and y in [-0.1, 0.1) +
    theirs: robots east of the grid read `outside`.  Cells are uniform in [-0.5, 1) with 5 % NaNs and 0.5 % +inf."""
    aos = layout.soa_to_aos(src, R, layout.VS_WORDS)
    pos = aos[:, [layout.VS_POS_X, layout.VS_POS_Y]].view(np.float32)
    rng = np.random.default_rng(seed)
    cells = rng.uniform(-0.5, 1.0, (n_maps, 40, 24)).astype(np.float32)
    cells[rng.random(cells.shape) < 0.05] = np.nan
    cells[rng.random(cells.shape) < 0.005] = np.inf
    origin = (float(pos[:, 0].mean()) - 0.1, float(pos[:, 1].mean()) - 0.1)
    map_of = None
    if n_maps > 1:
        map_of = rng.integers(0, n_maps, R).astype(np.int32)
        map_of[[1, 7]], map_of[[2, 11]] = -1, n_maps  # no map term for these robots
    return cells, origin, outside, map_of


def _costmap(world):
    cells, origin, outside, map_of = world
    return CostMap(torch.from_numpy(cells).to(DEV), origin, 0.005, outside, None if map_of is None else torch.from_numpy(map_of).to(DEV))


def _host(cm, w_map):
    return pmr.HostMap(cm.cells.cpu().numpy(), None if cm.map_of is None else cm.map_of.cpu().numpy(), np.float32(cm.x0), np.float32(cm.y0),
                       np.float32(cm.inv_res), np.float32(cm.outside), np.float32(w_map))


def _map_rollout(vb, cand, ref, obs, P, w_obst, cm, w_map, params=None, path=True):
    """rk_plan_rollout_map: (cost float32 [R*S], path float32 [n_ck, R*S, 2] or None)."""
    lib = rk.load()
    n_ck = N_SEG * SEG_LEN // P
    c = _cabi.PlanCost()
    ref_d = torch.from_numpy(np.ascontiguousarray(ref)).to(DEV)
    cand_d = _cells(cand, (N_SEG, R * S))
    obs_d = torch.from_numpy(np.ascontiguousarray(obs)).to(DEV)
    cost = torch.full((R * S,), float("nan"), dtype=torch.float32, device=DEV)
    pth = torch.full((n_ck, R * S, 2), float("nan"), dtype=torch.float32, device=DEV) if path else None
    c.d_ref, c.w_pos, c.w_goal, c.w_cur = ref_d.data_ptr(), *W
    o = _cabi.PlanObstacles()
    o.d_obs, o.m, o.check_period, o.w_obst = obs_d.data_ptr(), obs.shape[1], P, w_obst
    mp = None if cm is None else cm.struct(w_map)
    _cabi.check(lib.rk_plan_rollout_map(params or rk.default_params(), vb.state.data_ptr(), R, S, cand_d.data_ptr(), N_SEG, SEG_LEN, c, o,
                                        None if mp is None else C.byref(mp), None if pth is None else pth.data_ptr(), cost.data_ptr(),
                                        torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return cost.cpu().numpy(), None if pth is None else pth.cpu().numpy()


def test_planner_static_discs_expand_to_the_4d_table():
    vb, src, ref, cand = _case(seed=8)
    P = 5
    n_ck = N_SEG * SEG_LEN // P
    pl = VehiclePlanner(R, S, N_SEG, SEG_LEN, DEV)
    pl.candidates.copy_(_cells(cand, (N_SEG, R * S)))
    cm = _costmap(_world(src, 3, np.inf, seed=5))
    static = torch.from_numpy(_moving_discs(src, 1, 3, seed=9)[0]).to(DEV)
    ref_d = torch.from_numpy(ref).to(DEV)
    a = pl.rollout(vb, ref_d, *W, obstacles=static, w_obst=W_OBST, check_period=P, costmap=cm, w_map=25.0).clone()
    b = pl.rollout(vb, ref_d, *W, obstacles=static.expand(n_ck, 3, R, 4).contiguous(), w_obst=W_OBST, check_period=P, costmap=cm,
                   w_map=25.0).clone()
    torch.cuda.synchronize()
    np.testing.assert_array_equal(_u32(a), _u32(b))
    exp, _, _ = pmr.candidate_costs_map(src, R, S, cand, SEG_LEN, ref, *W, np.repeat(static.cpu().numpy()[None], n_ck, 0), P, W_OBST,
                                        _host(cm, 25.0))
    np.testing.assert_array_equal(_u32(a), exp.view(np.uint32))
    # no obstacles: checkpoints every seg_len ticks by default, m = 0
    c = pl.rollout(vb, ref_d, *W, costmap=cm, w_map=25.0)
    torch.cuda.synchronize()
    exp, _, _ = pmr.candidate_costs_map(src, R, S, cand, SEG_LEN, ref, *W, np.zeros((N_SEG, 0, R, 4), np.float32), SEG_LEN, 0.0,
                                        _host(cm, 25.0))
    np.testing.assert_array_equal(_u32(c), exp.view(np.uint32))


@pytest.mark.parametrize("mode,steps", [("argmin", 10), ("cem", 5)])
def test_wall_loop_equals_the_host_restatement(mode, steps):
    sc = pmr.WALL
    cem = None if mode == "argmin" else pmr.WALL_CEM
    exp, g, wall, origin = pmr.wall_loop(sc, cem=cem, steps=steps)
    Rw, n_seg, seg_len, P = sc["R"], sc["n_seg"], sc["seg_len"], sc["P"]
    _, cells, origin, start, _ = pmr.wall_world(Rw)
    robots = VehicleBatch(Rw, DEV)
    robots.load_state_soa(pfr.start_states(start))
    pl = VehiclePlanner(Rw, sc["S"] if cem is None else cem["S"], n_seg, seg_len, DEV, sigma=sc["sigma"], seed=sc["seed"])
    cm = CostMap(torch.from_numpy(cells).to(DEV), origin, pmr.CELL)
    ref = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(g, (n_seg, Rw, 2)))).to(DEV)
    w = (sc["w_pos"], sc["w_goal"], sc["w_cur"])
    for it in range(steps):
        if cem is None:
            pl.plan(robots, ref, *w, lam=0.0, shift=0, seed=sc["seed"] + it, check_period=P, costmap=cm, w_map=sc["w_map"])
        else:
            pl.plan_cem(robots, ref, *w, cem["iters"], cem["elite"], cem["alpha"], cem["sigma_min"], shift=0, seed=sc["seed"] + it,
                        check_period=P, costmap=cm, w_map=sc["w_map"])
        robots.rollout(seg_len, sensor_mode=_cabi.RK_SENSOR_PLANT, cmd=pl.first_command(), seg_len=seg_len)
        torch.cuda.synchronize()
        costs, ebest, estate, _ = exp[it]
        np.testing.assert_array_equal(_u32(pl.cost), costs[-1].view(np.uint32), err_msg=f"step {it}: costs")
        np.testing.assert_array_equal(pl.best.cpu().numpy(), ebest, err_msg=f"step {it}: best")
        np.testing.assert_array_equal(_u32(robots.state), estate, err_msg=f"step {it}: executed states")


def test_fleet_step_with_peer_discs_and_a_map():
    sc = FLEET
    G, n_seg, seg_len, P, S_ = sc["G"], sc["n_seg"], sc["seg_len"], sc["P"], sc["S"]
    Rf = sc["groups"] * G
    start, g = pfr.circle_swap(sc["groups"], G, sc["circle"], sc["spacing"])
    state = pfr.start_states(start)
    cells = np.zeros((12, 12), dtype=np.float32)  # 5 cm cells over x, y in [-0.3, 0.3): group 0 only
    cells[5:7, 3:9] = 1.0  # a 0.3 m x 0.1 m table across group 0's centre, under two of its robots
    origin = (-0.3, -0.3)
    ref_np = np.ascontiguousarray(np.broadcast_to(g, (n_seg, Rf, 2)))
    # the port: predict -> peer discs -> candidates -> cost with discs and map -> argmin
    nominal = np.zeros((n_seg, Rf), dtype=pr.CMD_DT)
    discs = pfr.peer_discs(pfr.predict(state, Rf, nominal, seg_len, P), pfr.fleet_peers(Rf, G), np.float32(sc["disc"]))
    cand = streams.plan_commands_v2(nominal, S_, seed=sc["seed"], sigma=sc["sigma"])
    # group 1 is off the grid and reads `outside` = 0: no map term
    mp = pmr.host_map(cells, origin, 1.0e3, outside=0.0)
    exp, O, _ = pmr.candidate_costs_map(state, Rf, S_, cand, seg_len, ref_np, sc["w_pos"], sc["w_goal"], sc["w_cur"], discs, P, sc["w_obst"], mp)
    _, best, _ = pr.select_argmin(exp, cand, Rf, S_, 0)
    # the device
    robots = VehicleBatch(Rf, DEV)
    robots.load_state_soa(state)
    pl = VehiclePlanner(Rf, S_, n_seg, seg_len, DEV, sigma=sc["sigma"], seed=sc["seed"])
    cm = CostMap(torch.from_numpy(cells).to(DEV), origin, pmr.CELL, outside=0.0)
    path = pl.predict(robots, check_period=P)
    d = pl.peer_discs(path, fleet_peers(Rf, G, DEV), radius=sc["disc"])
    pl.plan(robots, torch.from_numpy(ref_np).to(DEV), sc["w_pos"], sc["w_goal"], sc["w_cur"], lam=0.0, shift=0, seed=sc["seed"], obstacles=d,
            w_obst=sc["w_obst"], check_period=P, costmap=cm, w_map=1.0e3)
    torch.cuda.synchronize()
    np.testing.assert_array_equal(_u32(d).reshape(discs.shape), discs.view(np.uint32))
    np.testing.assert_array_equal(_u32(pl.cost), exp.view(np.uint32))
    np.testing.assert_array_equal(pl.best.cpu().numpy(), best)
    assert (O > 0).any() and (O == 0).any(), "the table must price some candidates, not all"
