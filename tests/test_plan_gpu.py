"""GPU: the sampling planner (rk_plan_sample_commands / rk_plan_rollout / rk_plan_select) against its definitions --
bit for bit against streams.plan_commands_v2 and the port (tests/plan_ref.py), on every rollout kernel, and the whole
closed planning loop against the host restatement."""
import numpy as np
import pytest
import torch

import plan_ref as pr
import workloads as wl
import roboken_fmskf_robot_controller_b200 as rk
from roboken_fmskf_robot_controller_b200 import _cabi, layout, streams
from roboken_fmskf_robot_controller_b200.planner import VehiclePlanner
from roboken_fmskf_robot_controller_b200.vehicle import VehicleBatch
from test_plan_cpu import PLAN_GOAL_TOLERANCE_M, _nominal

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _dev(a):
    return torch.from_numpy(np.ascontiguousarray(a).view(np.int32)).to(DEV)


def _cells(records, shape):
    return _dev(records).reshape(*shape, 4)


def _u32(t):
    return t.cpu().numpy().view(np.uint32)


@pytest.mark.parametrize("R,S,n_seg", [(37, 7, 3), (5, 1, 4), (64, 128, 8), (3, 300, 2)])
def test_sampler_bit_exact(R, S, n_seg):
    nom = _nominal(n_seg, R, seed=R, scale=420.0)  # some nominals beyond the speed limit
    pl = VehiclePlanner(R, S, n_seg, 10, DEV, sigma=(120.0, 80.0, 3.0), seed=77, first=123456)
    pl.sample(nominal=_cells(nom, (n_seg, R)), seed=99)
    torch.cuda.synchronize()
    exp = streams.plan_commands_v2(nom, S, seed=99, first=123456, sigma=(120.0, 80.0, 3.0))
    np.testing.assert_array_equal(_u32(pl.candidates).reshape(n_seg, R * S, 4), exp.view(np.uint32).reshape(n_seg, R * S, 4))


def _mid_move_states(R, seed=4):
    """R robots after 300 ticks of stream commands from power-on (rk_vdt_rollout): moving, currents flowing."""
    inp = wl.plant_inputs(R, 300, seed=seed)
    vb = VehicleBatch(R, DEV)
    vb.rollout(300, sensor_mode=_cabi.RK_SENSOR_PLANT, cmd=_cells(inp["cmd"], (-1, R)), seg_len=inp["seg_len"],
               yaw=torch.from_numpy(inp["yaw"]).to(DEV), yaw_period=inp["yaw_period"])
    return vb


def _plan_rollout(vb, R, S, cand, n_seg, seg_len, ref, w, params=None):
    lib = rk.load()
    c = _cabi.PlanCost()
    ref_d = torch.from_numpy(np.ascontiguousarray(ref)).to(DEV)
    cand_d = _cells(cand, (n_seg, R * S))
    cost = torch.full((R * S,), float("nan"), dtype=torch.float32, device=DEV)
    c.d_ref, c.w_pos, c.w_goal, c.w_cur = ref_d.data_ptr(), *w
    p = params or rk.default_params()
    _cabi.check(lib.rk_plan_rollout(p, vb.state.data_ptr(), R, S, cand_d.data_ptr(), n_seg, seg_len, c, cost.data_ptr(),
                                    torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return cost.cpu().numpy()


def _params(kind):
    p = rk.default_params()
    if kind == "kd":
        p.kd = 0.0005
    elif kind == "transcription":
        p.raw_curr_lim = 8000  # outside the fast kernel's domain: the transcription kernel runs
    return p


@pytest.mark.parametrize("variant", ["default", "force_transcription", "scalar", "kd", "transcription"])
def test_rollout_costs_bit_exact_vs_port(variant):
    R, S, n_seg, seg_len = 24, 20, 4, 25
    vb = _mid_move_states(R)
    src = _u32(vb.state).copy()
    rng = np.random.default_rng(1)
    ref = rng.uniform(-0.5, 0.5, (n_seg, R, 2)).astype(np.float32)
    cand = streams.plan_commands_v2(_nominal(n_seg, R), S, seed=5)
    w = (1.0, 10.0, 1e-8)
    lib, p = rk.load(), _params(variant)
    try:
        if variant == "force_transcription":
            lib.rk_set_option(_cabi.RK_OPT_FORCE_TRANSCRIPTION, 1)
        if variant == "scalar":
            lib.rk_set_option(_cabi.RK_OPT_FAST_PACKED, 0)
        got = _plan_rollout(vb, R, S, cand, n_seg, seg_len, ref, w, params=p)
    finally:
        lib.rk_set_option(_cabi.RK_OPT_FORCE_TRANSCRIPTION, 0)
        lib.rk_set_option(_cabi.RK_OPT_FAST_PACKED, 1)
    assert np.array_equal(_u32(vb.state), src), "rk_plan_rollout wrote the source states"
    exp = pr.candidate_costs(src, R, S, cand, seg_len, ref, *w, params=p)
    assert np.isfinite(exp).all() and exp.min() > 0
    np.testing.assert_array_equal(got.view(np.uint32), exp.view(np.uint32))


def test_rollout_with_one_candidate_is_the_plain_rollout():
    R, n_seg, seg_len = 64, 3, 40
    vb = _mid_move_states(R, seed=8)
    cand = streams.plan_commands_v2(_nominal(n_seg, R, seed=2), 1, seed=3)
    ref = np.random.default_rng(2).uniform(-1, 1, (n_seg, R, 2)).astype(np.float32)
    got = _plan_rollout(vb, R, 1, cand, n_seg, seg_len, ref, (0.5, 4.0, 2e-8))
    plain = VehicleBatch(R, DEV)
    plain.state.copy_(vb.state)
    tr = torch.zeros((n_seg * seg_len, 16, R), dtype=torch.int32, device=DEV)
    plain.rollout(n_seg * seg_len, sensor_mode=_cabi.RK_SENSOR_PLANT, cmd=_cells(cand, (n_seg, R)), seg_len=seg_len, trace=tr)
    torch.cuda.synchronize()
    exp = pr.stage_cost(_u32(tr), ref, 1, seg_len, 0.5, 4.0, 2e-8)
    np.testing.assert_array_equal(got.view(np.uint32), exp.view(np.uint32))


def _select(cost, cand, R, S, n_seg, lam, shift):
    lib = rk.load()
    cost_d = torch.from_numpy(np.ascontiguousarray(cost)).to(DEV)
    cand_d = _cells(cand, (n_seg, R * S))
    nom = torch.full((n_seg, R, 4), -1, dtype=torch.int32, device=DEV)
    best = torch.full((R,), -1, dtype=torch.int32, device=DEV)
    bc = torch.zeros(R, dtype=torch.float32, device=DEV)
    _cabi.check(lib.rk_plan_select(cost_d.data_ptr(), cand_d.data_ptr(), R, S, n_seg, float(lam), shift, nom.data_ptr(), best.data_ptr(),
                                   bc.data_ptr(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return _u32(nom), best.cpu().numpy(), bc.cpu().numpy()


def _select_case(R, S, n_seg, seed):
    rng = np.random.default_rng(seed)
    cost = rng.integers(0, 50, (R, S)).astype(np.float32) * np.float32(0.125)  # many ties
    cost[rng.random((R, S)) < 0.2] = np.nan
    cost[0] = np.nan  # all NaN
    cost[1, :] = np.inf
    cost[2, 1::2] = np.nan
    cost = cost.reshape(-1)
    cand = streams.plan_commands_v2(_nominal(n_seg, R, seed=seed), S, seed=seed)
    return cost, cand


@pytest.mark.parametrize("R,S", [(40, 33), (9, 1), (17, 256)])
def test_select_argmin_exact(R, S):
    n_seg = 5
    cost, cand = _select_case(R, S, n_seg, seed=R + S)
    for shift in range(n_seg):
        nom, best, bc = _select(cost, cand, R, S, n_seg, 0.0, shift)
        enom, ebest, ebc = pr.select_argmin(cost, cand, R, S, shift)
        np.testing.assert_array_equal(best, ebest)
        np.testing.assert_array_equal(bc.view(np.uint32), ebc.view(np.uint32))
        np.testing.assert_array_equal(nom.reshape(n_seg, R, 4), enom.view(np.uint32).reshape(n_seg, R, 4))
    assert best[0] == 0 and np.isnan(bc[0])


@pytest.mark.parametrize("lam", [1e-3, 0.5, 20.0])
def test_select_mppi_vs_float64(lam):
    R, S, n_seg, shift = 33, 70, 4, 1
    cost, cand = _select_case(R, S, n_seg, seed=11)
    nom, best, _ = _select(cost, cand, R, S, n_seg, lam, shift)
    nom2, _, _ = _select(cost, cand, R, S, n_seg, lam, shift)
    assert np.array_equal(nom, nom2), "two calls differ"
    nom = nom.reshape(n_seg, R, 4)
    c = cost.reshape(R, S).astype(np.float64)
    fin = np.isfinite(np.nanmin(np.where(np.isnan(c), np.inf, c), axis=1))
    ss = np.minimum(np.arange(n_seg) + shift, n_seg - 1)
    cc = cand[ss].reshape(n_seg, R, S)
    for r in range(R):
        if not fin[r]:  # no finite minimum: candidate `best` as under lambda == 0
            np.testing.assert_array_equal(nom[:, r], np.ascontiguousarray(cc[:, r, best[r]]).view(np.uint32).reshape(n_seg, 4))
            continue
        w = np.exp(-(c[r] - np.nanmin(c[r])) / lam)
        w[np.isnan(w)] = 0.0
        for a, f in enumerate(("vx", "vy", "vth")):
            v = cc[f][:, r, :].astype(np.float64)
            ref = (w * v).sum(-1) / w.sum()
            scale = (w * np.abs(v)).sum(-1) / w.sum()
            got = nom[:, r, a].view(np.float32).astype(np.float64)
            assert (np.abs(got - ref) <= 1e-5 * scale + 1e-30).all(), (r, f, got, ref)
        assert (nom[:, r, 3] == _cabi.RK_CMD_MOVE).all()


def _gpu_plan_loop(lam, sc=pr.SCENARIO, check=None):
    R, S, n_seg, seg_len = sc["R"], sc["S"], sc["n_seg"], sc["seg_len"]
    g = pr.goals(R)
    ref = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(g, (n_seg, R, 2)))).to(DEV)
    vb = VehicleBatch(R, DEV)
    pl = VehiclePlanner(R, S, n_seg, seg_len, DEV, sigma=sc["sigma"], seed=sc["seed"])
    for it in range(sc["steps"]):
        pl.plan(vb, ref, sc["w_pos"], sc["w_goal"], sc["w_cur"], lam=lam, shift=1, seed=sc["seed"] + it)
        vb.rollout(seg_len, sensor_mode=_cabi.RK_SENSOR_PLANT, cmd=pl.first_command(), seg_len=seg_len)
        if check is not None:
            torch.cuda.synchronize()
            check(it, pl.cost.cpu().numpy(), pl.best.cpu().numpy(), _u32(vb.state))
    torch.cuda.synchronize()
    return _u32(vb.state), g


def test_closed_loop_planning_equals_the_host_restatement():
    exp, g = pr.plan_loop()

    def check(it, cost, best, state):
        ecost, ebest, estate = exp[it]
        np.testing.assert_array_equal(cost.view(np.uint32), ecost.view(np.uint32), err_msg=f"step {it}: costs")
        np.testing.assert_array_equal(best, ebest, err_msg=f"step {it}: best")
        np.testing.assert_array_equal(state, estate, err_msg=f"step {it}: executed states")

    state, g = _gpu_plan_loop(0.0, check=check)
    assert (pr.distances(state, pr.SCENARIO["R"], g) < PLAN_GOAL_TOLERANCE_M).all()


def test_mppi_planning_reaches_the_goals():
    state, g = _gpu_plan_loop(1e-3)
    d = pr.distances(state, pr.SCENARIO["R"], g)
    assert (d < PLAN_GOAL_TOLERANCE_M).all(), d
