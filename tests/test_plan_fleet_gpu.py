"""GPU: moving keep-out discs, candidate paths and fleet planning (rk_plan_rollout_moving, rk_plan_peer_discs,
VehiclePlanner.predict / peer_discs) against the host restatement tests/plan_fleet_ref.py -- bit for bit on every rollout
kernel, the equalities with rk_plan_rollout_obstacles and rk_plan_rollout, and the closed fleet loop under argmin and
CEM."""
import numpy as np
import pytest
import torch

import plan_cem_ref as pcr
import plan_fleet_ref as pfr
import plan_ref as pr
import roboken_fmskf_robot_controller_b200 as rk
from roboken_fmskf_robot_controller_b200 import _cabi
from roboken_fmskf_robot_controller_b200.planner import VehiclePlanner, fleet_peers
from roboken_fmskf_robot_controller_b200.vehicle import VehicleBatch
from test_plan_fleet_cpu import FLEET
from test_plan_gpu import _cells, _params, _plan_rollout, _u32
from test_plan_obst_gpu import N_SEG, R, S, SEG_LEN, W, _case, _discs, _obst_rollout

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _moving_discs(src, n_ck, m, seed):
    """A table float32 [n_ck, m, R, 4] of discs that move from checkpoint to checkpoint: test_plan_obst_gpu._discs (NaN
    discs included) whose centres walk up to 0.2 mm per checkpoint along each axis, so that the discs move but some
    candidates still miss every disc even at P = 1."""
    obs = np.repeat(_discs(src, m, seed)[None], n_ck, axis=0)
    obs[..., :2] += np.cumsum(np.random.default_rng(seed).uniform(-2e-4, 2e-4, (n_ck, m, R, 2)), axis=0).astype(np.float32)
    return obs


def _moving_rollout(vb, cand, ref, obs, P, w_obst, params=None, path=False):
    """rk_plan_rollout_moving: (cost float32 [R*S], path float32 [n_ck, R*S, 2] or None)."""
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
    _cabi.check(lib.rk_plan_rollout_moving(params or rk.default_params(), vb.state.data_ptr(), R, S, cand_d.data_ptr(), N_SEG, SEG_LEN, c, o,
                                           None if pth is None else pth.data_ptr(), cost.data_ptr(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return cost.cpu().numpy(), None if pth is None else pth.cpu().numpy()


@pytest.mark.parametrize("m", [1, 7])
@pytest.mark.parametrize("P", [1, 5, SEG_LEN])
@pytest.mark.parametrize("variant", ["default", "force_transcription", "scalar", "kd", "transcription"])
def test_moving_costs_and_paths_bit_exact_vs_port(variant, P, m):
    vb, src, ref, cand = _case()
    n_ck = N_SEG * SEG_LEN // P
    obs = _moving_discs(src, n_ck, m, seed=10 * m + P)  # the static discs of test_plan_obst_gpu, set moving
    w_obst = float("inf") if m == 7 else 3.0e3
    lib, p = rk.load(), _params(variant)
    try:
        if variant == "force_transcription":
            lib.rk_set_option(_cabi.RK_OPT_FORCE_TRANSCRIPTION, 1)
        if variant == "scalar":
            lib.rk_set_option(_cabi.RK_OPT_FAST_PACKED, 0)
        got, path = _moving_rollout(vb, cand, ref, obs, P, w_obst, params=p, path=True)
        bare, _ = _moving_rollout(vb, cand, ref, obs, P, w_obst, params=p)
    finally:
        lib.rk_set_option(_cabi.RK_OPT_FORCE_TRANSCRIPTION, 0)
        lib.rk_set_option(_cabi.RK_OPT_FAST_PACKED, 1)
    assert np.array_equal(_u32(vb.state), src), "rk_plan_rollout_moving wrote the source states"
    exp, O, exp_path = pfr.candidate_costs_moving(src, R, S, cand, SEG_LEN, ref, *W, obs, P, w_obst, params=p)
    assert (O == 0).any() and (O > 0).any(), "the discs must be entered by some candidates and missed by others"
    np.testing.assert_array_equal(got.view(np.uint32), exp.view(np.uint32))
    np.testing.assert_array_equal(bare.view(np.uint32), got.view(np.uint32), err_msg="d_path changed d_cost")
    np.testing.assert_array_equal(path.view(np.uint32), exp_path.view(np.uint32))


@pytest.mark.parametrize("variant", ["default", "scalar", "transcription"])
def test_equalities_with_the_static_and_plain_rollouts(variant):
    vb, src, ref, cand = _case(seed=6)
    P = 5
    n_ck = N_SEG * SEG_LEN // P
    obs = _discs(src, 3, seed=2)
    lib, p = rk.load(), _params(variant)
    try:
        if variant == "scalar":
            lib.rk_set_option(_cabi.RK_OPT_FAST_PACKED, 0)
        static = _obst_rollout(vb, cand, ref, obs, P, 3.0e3, params=p)
        plain = _plan_rollout(vb, R, S, cand, N_SEG, SEG_LEN, ref, W, params=p)
        rep = np.ascontiguousarray(np.broadcast_to(obs, (n_ck,) + obs.shape))
        for path in (False, True):
            got, _ = _moving_rollout(vb, cand, ref, rep, P, 3.0e3, params=p, path=path)
            np.testing.assert_array_equal(got.view(np.uint32), static.view(np.uint32), err_msg=f"repeated table, path={path}")
            got, _ = _moving_rollout(vb, cand, ref, rep[:, :0], P, 3.0e3, params=p, path=path)
            np.testing.assert_array_equal(got.view(np.uint32), plain.view(np.uint32), err_msg=f"m = 0, path={path}")
    finally:
        lib.rk_set_option(_cabi.RK_OPT_FAST_PACKED, 1)
    assert np.array_equal(_u32(vb.state), src)


def test_predict_matches_the_port():
    vb, src, ref, cand = _case(seed=8)
    pl = VehiclePlanner(R, S, N_SEG, SEG_LEN, DEV)
    nominal = cand.reshape(N_SEG, R, S)[:, :, 3].copy()  # any plan: candidate 3 of every robot
    pl.nominal.copy_(_cells(nominal, (N_SEG, R)))
    for P in (1, 5, SEG_LEN):
        got = pl.predict(vb, check_period=P)
        torch.cuda.synchronize()
        exp = pfr.predict(src, R, nominal, SEG_LEN, P)
        assert tuple(got.shape) == (N_SEG * SEG_LEN // P, R, 2)
        np.testing.assert_array_equal(_u32(got).reshape(exp.shape), exp.view(np.uint32))
    assert np.array_equal(_u32(vb.state), src)


def test_peer_discs_match_numpy():
    Rn, n_ck, M, k0 = 300, 7, 5, 2
    rng = np.random.default_rng(9)
    path = rng.uniform(-1, 1, (n_ck, Rn, 2)).astype(np.float32)
    peers = rng.integers(-3, Rn + 3, (2, Rn)).astype(np.int32)
    peers[0, :10] = np.arange(10)  # themselves
    peers[1, 10:20] = 1 << 30
    sentinel = np.full((n_ck, M, Rn, 4), 7.0, dtype=np.float32)
    pl = VehiclePlanner(Rn, 1, 1, 10, DEV)
    out = torch.from_numpy(sentinel.copy()).to(DEV)
    pl.peer_discs(torch.from_numpy(path).to(DEV), torch.from_numpy(peers).to(DEV), 0.33, out=out, k0=k0)
    torch.cuda.synchronize()
    exp = pfr.peer_discs(path, peers, np.float32(0.33), out=sentinel.copy(), k0=k0)
    np.testing.assert_array_equal(_u32(out).reshape(exp.shape), exp.view(np.uint32))
    fresh = pl.peer_discs(torch.from_numpy(path).to(DEV), fleet_peers(Rn, 4, DEV), 0.1)
    exp = pfr.peer_discs(path, pfr.fleet_peers(Rn, 4), np.float32(0.1))
    np.testing.assert_array_equal(_u32(fresh).reshape(exp.shape), exp.view(np.uint32))


@pytest.mark.parametrize("mode,steps", [("argmin", 12), ("cem", 6)])
def test_fleet_loop_equals_the_host_restatement(mode, steps):
    sc = FLEET
    cem = None if mode == "argmin" else dict(pcr.CEM, S=32)
    exp, g = pfr.fleet_loop(sc, avoid=True, cem=cem, steps=steps)
    n_grp, G, n_seg, seg_len, P = sc["groups"], sc["G"], sc["n_seg"], sc["seg_len"], sc["P"]
    Rf = n_grp * G
    start, _ = pfr.circle_swap(n_grp, G, sc["circle"], sc["spacing"])
    robots = VehicleBatch(Rf, DEV)
    robots.load_state_soa(pfr.start_states(start))
    pl = VehiclePlanner(Rf, sc["S"] if cem is None else cem["S"], n_seg, seg_len, DEV, sigma=sc["sigma"], seed=sc["seed"])
    ref = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(g, (n_seg, Rf, 2)))).to(DEV)
    peers = fleet_peers(Rf, G, DEV)
    w = (sc["w_pos"], sc["w_goal"], sc["w_cur"])
    for it in range(steps):
        path = pl.predict(robots, check_period=P)
        discs = pl.peer_discs(path, peers, radius=sc["disc"])
        if cem is None:
            pl.plan(robots, ref, *w, lam=0.0, shift=0, seed=sc["seed"] + it, obstacles=discs, w_obst=sc["w_obst"], check_period=P)
        else:
            pl.plan_cem(robots, ref, *w, cem["iters"], cem["elite"], cem["alpha"], cem["sigma_min"], shift=0, seed=sc["seed"] + it,
                        obstacles=discs, w_obst=sc["w_obst"], check_period=P)
        robots.rollout(seg_len, sensor_mode=_cabi.RK_SENSOR_PLANT, cmd=pl.first_command(), seg_len=seg_len)
        torch.cuda.synchronize()
        costs, ebest, estate, _ = exp[it]
        np.testing.assert_array_equal(_u32(pl.cost), costs[-1].view(np.uint32), err_msg=f"step {it}: costs")
        np.testing.assert_array_equal(pl.best.cpu().numpy(), ebest, err_msg=f"step {it}: best")
        np.testing.assert_array_equal(_u32(robots.state), estate, err_msg=f"step {it}: executed states")
    assert pr.distances(_u32(robots.state), Rf, g).max() < 2 * sc["circle"]
