"""GPU: keep-out discs in the planner's candidate cost (rk_plan_rollout_obstacles) against the host restatement
tests/plan_obst_ref.py -- bit for bit on every rollout kernel, the equalities with rk_plan_rollout, w_obst = +inf with
selection, and the closed planning loop through VehiclePlanner with discs."""
import numpy as np
import pytest
import torch

import plan_obst_ref as por
import plan_ref as pr
import roboken_fmskf_robot_controller_b200 as rk
from roboken_fmskf_robot_controller_b200 import _cabi, layout, streams
from roboken_fmskf_robot_controller_b200.planner import VehiclePlanner
from roboken_fmskf_robot_controller_b200.vehicle import VehicleBatch
from test_plan_cpu import PLAN_GOAL_TOLERANCE_M, _nominal
from test_plan_gpu import _cells, _mid_move_states, _params, _plan_rollout, _select, _u32
from test_plan_obst_cpu import CHECK_PERIOD, obstacle_scenario

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
R, S, N_SEG, SEG_LEN = 24, 20, 4, 25
W = (1.0, 10.0, 1e-8)


def _discs(src, m, seed):
    """m discs per robot, float32 [m, R, 4]: centres up to 60 mm from the robot's current position (the candidates travel
    a few tens of mm in 100 ticks), radii 5 - 25 mm, so that some candidates enter some discs and others none; robot 3's
    disc 0 has a NaN radius and robot 5's a NaN centre."""
    aos = layout.soa_to_aos(src, R, layout.VS_WORDS)
    pos = aos[:, [layout.VS_POS_X, layout.VS_POS_Y]].view(np.float32)
    rng = np.random.default_rng(seed)
    obs = np.zeros((m, R, 4), dtype=np.float32)
    obs[:, :, :2] = pos[None] + rng.uniform(-0.06, 0.06, (m, R, 2))
    obs[:, :, 2] = rng.uniform(0.005, 0.025, (m, R))
    obs[0, 3, 2] = np.nan
    obs[0, 5, 0] = np.nan
    return obs


def _obst_rollout(vb, cand, ref, obs, P, w_obst, params=None, m=None, null=False):
    lib = rk.load()
    c = _cabi.PlanCost()
    ref_d = torch.from_numpy(np.ascontiguousarray(ref)).to(DEV)
    cand_d = _cells(cand, (N_SEG, R * S))
    obs_d = torch.from_numpy(np.ascontiguousarray(obs)).to(DEV)
    cost = torch.full((R * S,), float("nan"), dtype=torch.float32, device=DEV)
    c.d_ref, c.w_pos, c.w_goal, c.w_cur = ref_d.data_ptr(), *W
    o = _cabi.PlanObstacles()
    o.d_obs, o.m, o.check_period, o.w_obst = obs_d.data_ptr(), obs.shape[0] if m is None else m, P, w_obst
    _cabi.check(lib.rk_plan_rollout_obstacles(params or rk.default_params(), vb.state.data_ptr(), R, S, cand_d.data_ptr(), N_SEG, SEG_LEN,
                                              c, None if null else o, cost.data_ptr(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return cost.cpu().numpy()


def _case(seed=4):
    vb = _mid_move_states(R, seed=seed)
    src = _u32(vb.state).copy()
    ref = np.random.default_rng(1).uniform(-0.5, 0.5, (N_SEG, R, 2)).astype(np.float32)
    cand = streams.plan_commands_v2(_nominal(N_SEG, R), S, seed=5)
    return vb, src, ref, cand


@pytest.mark.parametrize("m", [1, 7])
@pytest.mark.parametrize("P", [1, 5, SEG_LEN])
@pytest.mark.parametrize("variant", ["default", "force_transcription", "scalar", "kd", "transcription"])
def test_obstacle_costs_bit_exact_vs_port(variant, P, m):
    vb, src, ref, cand = _case()
    obs = _discs(src, m, seed=10 * m + P)
    w_obst = 3.0e3
    lib, p = rk.load(), _params(variant)
    try:
        if variant == "force_transcription":
            lib.rk_set_option(_cabi.RK_OPT_FORCE_TRANSCRIPTION, 1)
        if variant == "scalar":
            lib.rk_set_option(_cabi.RK_OPT_FAST_PACKED, 0)
        got = _obst_rollout(vb, cand, ref, obs, P, w_obst, params=p)
    finally:
        lib.rk_set_option(_cabi.RK_OPT_FORCE_TRANSCRIPTION, 0)
        lib.rk_set_option(_cabi.RK_OPT_FAST_PACKED, 1)
    assert np.array_equal(_u32(vb.state), src), "rk_plan_rollout_obstacles wrote the source states"
    exp, O = por.candidate_costs_obst(src, R, S, cand, SEG_LEN, ref, *W, obs, P, w_obst, params=p)
    assert (O == 0).any() and (O > 0).any(), "the discs must be entered by some candidates and missed by others"
    np.testing.assert_array_equal(got.view(np.uint32), exp.view(np.uint32))


@pytest.mark.parametrize("variant", ["default", "scalar", "transcription"])
def test_without_discs_is_the_plan_rollout(variant):
    vb, src, ref, cand = _case(seed=6)
    obs = _discs(src, 3, seed=2)
    lib, p = rk.load(), _params(variant)
    try:
        if variant == "scalar":
            lib.rk_set_option(_cabi.RK_OPT_FAST_PACKED, 0)
        plain = _plan_rollout(vb, R, S, cand, N_SEG, SEG_LEN, ref, W, params=p)
        for kw in (dict(m=0), dict(null=True), dict()):  # m = 0, obst = NULL, w_obst = 0 with the discs present
            got = _obst_rollout(vb, cand, ref, obs, 5, 0.0, params=p, **kw)
            np.testing.assert_array_equal(got.view(np.uint32), plain.view(np.uint32), err_msg=str(kw or "w_obst = 0"))
    finally:
        lib.rk_set_option(_cabi.RK_OPT_FAST_PACKED, 1)
    assert np.array_equal(_u32(vb.state), src)


@pytest.mark.parametrize("P", [1, 5])
def test_infinite_weight_is_a_hard_constraint(P):
    vb, src, ref, cand = _case(seed=7)
    obs = _discs(src, 6, seed=21)  # a seed that leaves some robots with both clean and penetrating candidates
    got = _obst_rollout(vb, cand, ref, obs, P, float("inf"))
    plain = _plan_rollout(vb, R, S, cand, N_SEG, SEG_LEN, ref, W)
    _, O = por.candidate_costs_obst(src, R, S, cand, SEG_LEN, ref, *W, obs, P, np.float32(1.0))
    hit = O > 0
    assert hit.any() and (~hit).any()
    assert (got[hit] == np.inf).all()
    np.testing.assert_array_equal(got[~hit].view(np.uint32), plain[~hit].view(np.uint32))
    _, best, _ = _select(got, cand, R, S, N_SEG, 0.0, 1)
    clean = (~hit).reshape(R, S)
    assert (clean.any(axis=1) & ~clean.all(axis=1)).any(), "no robot has both clean and penetrating candidates"
    for r in range(R):
        if clean[r].any():
            assert clean[r, best[r]], f"robot {r}: picked a penetrating candidate over a clean one"


def test_closed_loop_with_discs_equals_the_host_restatement():
    sc = pr.SCENARIO
    Rs, n_seg, seg_len = sc["R"], sc["n_seg"], sc["seg_len"]
    disc, keep_out = obstacle_scenario()
    exp, g = por.plan_loop_obst(keep_out, np.inf, CHECK_PERIOD)
    ref = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(g, (n_seg, Rs, 2)))).to(DEV)
    obs = torch.from_numpy(keep_out).to(DEV)
    vb = VehicleBatch(Rs, DEV)
    pl = VehiclePlanner(Rs, sc["S"], n_seg, seg_len, DEV, sigma=sc["sigma"], seed=sc["seed"])
    tr = torch.zeros((seg_len, _cabi.RK_VDT_TRACE_WORDS, Rs), dtype=torch.int32, device=DEV)
    executed = []
    for it in range(sc["steps"]):
        pl.plan(vb, ref, sc["w_pos"], sc["w_goal"], sc["w_cur"], lam=0.0, shift=0, seed=sc["seed"] + it, obstacles=obs, w_obst=float("inf"),
                check_period=CHECK_PERIOD)
        vb.rollout(seg_len, sensor_mode=_cabi.RK_SENSOR_PLANT, cmd=pl.first_command(), seg_len=seg_len, trace=tr)
        torch.cuda.synchronize()
        ecost, ebest, estate, _ = exp[it]
        np.testing.assert_array_equal(_u32(pl.cost), ecost.view(np.uint32), err_msg=f"step {it}: costs")
        np.testing.assert_array_equal(pl.best.cpu().numpy(), ebest, err_msg=f"step {it}: best")
        np.testing.assert_array_equal(_u32(vb.state), estate, err_msg=f"step {it}: executed states")
        t = _u32(tr)
        executed.append((None, None, None, np.stack([t[:, 0].view(np.float32), t[:, 1].view(np.float32)], axis=2)))
    clear = por.min_clearance(executed, disc)
    assert (clear > 0).all(), f"an executed tick inside a disc: clearance {clear}"
    assert (pr.distances(_u32(vb.state), Rs, g) < PLAN_GOAL_TOLERANCE_M).all()
