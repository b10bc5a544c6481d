"""GPU: the cross-entropy planner (rk_plan_sample_commands_sigma / rk_plan_refit, VehiclePlanner.plan_cem) against its
definitions -- bit for bit against streams.plan_commands_v2(sigma_table=...) and tests/plan_cem_ref.py -- and the closed
CEM planning loop, with and without keep-out discs, against its host restatement on the port."""
import numpy as np
import pytest
import torch

import plan_cem_ref as cr
import plan_ref as pr
import roboken_fmskf_robot_controller_b200 as rk
from roboken_fmskf_robot_controller_b200 import _cabi, streams
from roboken_fmskf_robot_controller_b200.planner import VehiclePlanner
from roboken_fmskf_robot_controller_b200.vehicle import VehicleBatch
from test_plan_cpu import PLAN_GOAL_TOLERANCE_M, _nominal
from test_plan_gpu import _cells, _select, _select_case, _u32
from test_plan_obst_cpu import CHECK_PERIOD, obstacle_scenario

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
SIGMA = (120.0, 80.0, 3.0)


def _sigma_table(n_seg, R, seed):
    """A random scale per (segment, robot), with zero cells and zero axes; word 3 holds junk the sampler must ignore."""
    rng = np.random.default_rng(seed)
    tab = rng.uniform(0.0, 250.0, (n_seg, R, 4)).astype(np.float32)
    tab[..., 2] /= 50
    tab[rng.random((n_seg, R)) < 0.2] = 0.0
    tab[..., 1][rng.random((n_seg, R)) < 0.2] = 0.0
    tab[..., 3] = np.nan
    return tab


@pytest.mark.parametrize("R,S,n_seg", [(37, 7, 3), (5, 1, 4), (64, 128, 8), (3, 300, 2)])
def test_sigma_sampler_bit_exact(R, S, n_seg):
    nom = _nominal(n_seg, R, seed=R, scale=420.0)  # some nominals beyond the speed limit
    tab = _sigma_table(n_seg, R, seed=S)
    pl = VehiclePlanner(R, S, n_seg, 10, DEV, sigma=SIGMA, seed=77, first=123456)
    pl.sample(nominal=_cells(nom, (n_seg, R)), seed=99, sigma_table=torch.from_numpy(tab).to(DEV))
    torch.cuda.synchronize()
    exp = streams.plan_commands_v2(nom, S, seed=99, first=123456, sigma_table=tab)
    np.testing.assert_array_equal(_u32(pl.candidates).reshape(n_seg, R * S, 4), exp.view(np.uint32).reshape(n_seg, R * S, 4))
    # a table holding sigma in every cell: rk_plan_sample_commands' bits
    pl.sample(nominal=_cells(nom, (n_seg, R)), seed=99, sigma_table=torch.from_numpy(cr.sigma_cells(SIGMA, n_seg, R)).to(DEV))
    got = pl.candidates.clone()
    pl.sample(nominal=_cells(nom, (n_seg, R)), seed=99)
    assert torch.equal(got, pl.candidates)


def _refit(cost, cand, sig_in, R, S, n_seg, k, alpha, sigma_min, shift, in_place=False):
    lib = rk.load()
    cost_d = torch.from_numpy(np.ascontiguousarray(cost)).to(DEV)
    cand_d = _cells(cand, (n_seg, R * S))
    sin = torch.from_numpy(np.ascontiguousarray(sig_in)).to(DEV)
    sout = sin if in_place else torch.full((n_seg, R, 4), -1.0, dtype=torch.float32, device=DEV)
    nom = torch.full((n_seg, R, 4), -1, dtype=torch.int32, device=DEV)
    best = torch.full((R,), -1, dtype=torch.int32, device=DEV)
    bc = torch.zeros(R, dtype=torch.float32, device=DEV)
    rf = _cabi.PlanRefit()
    rf.elite, rf.alpha = k, alpha
    rf.sigma_min[:] = sigma_min
    _cabi.check(lib.rk_plan_refit(cost_d.data_ptr(), cand_d.data_ptr(), sin.data_ptr(), R, S, n_seg, rf, shift, nom.data_ptr(),
                                  sout.data_ptr(), best.data_ptr(), bc.data_ptr(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return _u32(nom), _u32(sout), best.cpu().numpy(), bc.cpu().numpy()


def _refit_case(R, S, n_seg, seed):
    """_select_case's costs (ties, NaN, an all-NaN robot, an all-+inf robot) with zeros of both signs and a -inf."""
    cost, cand = _select_case(R, S, n_seg, seed)
    c = cost.reshape(R, S)
    c[3, ::3], c[3, 1::3] = -0.0, 0.0
    c[4, S // 2] = -np.inf
    c[5, :] = c[5, 0]  # one cost throughout: the elites are the lowest j
    return c.reshape(-1), cand


K_CASES = [(S, k) for S in (1, 33, 256, 300) for k in sorted({1, 3, 32, 33, S}) if k <= S]


@pytest.mark.parametrize("S,k", K_CASES)
def test_refit_bit_exact(S, k):
    R, n_seg, sigma_min = 40, 5, (1.0, 0.0, 0.05)
    cost, cand = _refit_case(R, S, n_seg, seed=S + k)
    sig_in = _sigma_table(n_seg, R, seed=k)
    for alpha in (0.0, 0.3):
        for shift in range(n_seg):
            got = _refit(cost, cand, sig_in, R, S, n_seg, k, alpha, sigma_min, shift)
            enom, esig, ebest, ebc = cr.refit(cost, cand, sig_in, R, S, k, alpha, sigma_min, shift)
            what = f"alpha {alpha}, shift {shift}"
            np.testing.assert_array_equal(got[2], ebest, err_msg=what)
            np.testing.assert_array_equal(got[3].view(np.uint32), ebc.view(np.uint32), err_msg=what)
            np.testing.assert_array_equal(got[0].reshape(n_seg, R, 4), enom.view(np.uint32).reshape(n_seg, R, 4), err_msg=what)
            np.testing.assert_array_equal(got[1], esig.view(np.uint32), err_msg=what)
            again = _refit(cost, cand, sig_in, R, S, n_seg, k, alpha, sigma_min, shift)
            assert all(np.array_equal(x.view(np.uint32), y.view(np.uint32)) for x, y in zip(got, again)), f"{what}: two calls differ"
        inplace = _refit(cost, cand, sig_in, R, S, n_seg, k, alpha, sigma_min, 0, in_place=True)
        _, esig, _, _ = cr.refit(cost, cand, sig_in, R, S, k, alpha, sigma_min, 0)
        np.testing.assert_array_equal(inplace[1], esig.view(np.uint32), err_msg=f"alpha {alpha}: in place")
    assert (np.asarray([e.size for e in cr.elites(cost, R, S, k)]) == 0).sum() >= 2  # at least the all-NaN and the all-inf robot


@pytest.mark.parametrize("S", [33, 256])
def test_refit_with_one_elite_is_the_argmin_selection(S):
    R, n_seg = 40, 5
    cost, cand = _refit_case(R, S, n_seg, seed=S)
    cost[cost == -np.inf] = 0.5  # a -inf cost is rk_plan_select's argmin, but never an elite
    sig_in = _sigma_table(n_seg, R, seed=1)
    for shift in range(n_seg):
        nom, _, best, bc = _refit(cost, cand, sig_in, R, S, n_seg, 1, 0.0, (0.0, 0.0, 0.0), shift)
        snom, sbest, sbc = _select(cost, cand, R, S, n_seg, 0.0, shift)
        np.testing.assert_array_equal(nom, snom)
        np.testing.assert_array_equal(best, sbest)
        np.testing.assert_array_equal(bc.view(np.uint32), sbc.view(np.uint32))


def _cem_loop(cem, shift=1, obstacles=None, w_obst=0.0, check=None):
    sc = pr.SCENARIO
    R, n_seg, seg_len = sc["R"], sc["n_seg"], sc["seg_len"]
    g = pr.goals(R)
    ref = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(g, (n_seg, R, 2)))).to(DEV)
    vb = VehicleBatch(R, DEV)
    pl = VehiclePlanner(R, cem["S"], n_seg, seg_len, DEV, sigma=sc["sigma"], seed=sc["seed"])
    costs, refit = [], pl.refit

    def recording_refit(*a, **kw):  # every round's costs, as the refit sees them
        costs.append(pl.cost.clone())
        return refit(*a, **kw)

    pl.refit = recording_refit
    for it in range(sc["steps"]):
        src = vb.state.clone()
        costs.clear()
        pl.plan_cem(vb, ref, sc["w_pos"], sc["w_goal"], sc["w_cur"], cem["iters"], cem["elite"], alpha=cem["alpha"],
                    sigma_min=cem["sigma_min"], shift=shift, seed=sc["seed"] + it, obstacles=obstacles, w_obst=w_obst,
                    check_period=CHECK_PERIOD if obstacles is not None else None)
        torch.cuda.synchronize()
        assert torch.equal(vb.state, src), f"step {it}: plan_cem wrote the source states"
        vb.rollout(seg_len, sensor_mode=_cabi.RK_SENSOR_PLANT, cmd=pl.first_command(), seg_len=seg_len)
        torch.cuda.synchronize()
        if check is not None:
            check(it, [_u32(c) for c in costs], pl.best.cpu().numpy(), _u32(vb.state))
    return _u32(vb.state), g


def _checker(exp):
    def check(it, costs, best, state):
        ecosts, ebest, estate = exp[it]
        assert len(costs) == len(ecosts)
        for i, (c, e) in enumerate(zip(costs, ecosts)):
            np.testing.assert_array_equal(c, e.view(np.uint32), err_msg=f"step {it}, round {i}: costs")
        np.testing.assert_array_equal(best, ebest, err_msg=f"step {it}: best")
        np.testing.assert_array_equal(state, estate, err_msg=f"step {it}: executed states")

    return check


def test_closed_loop_cem_equals_the_host_restatement():
    exp, g = cr.plan_cem_loop()
    state, g = _cem_loop(cr.CEM, check=_checker(exp))
    d = pr.distances(state, pr.SCENARIO["R"], g)
    assert (d < PLAN_GOAL_TOLERANCE_M).all(), d


def test_closed_loop_cem_with_discs_equals_the_host_restatement():
    _, keep_out = obstacle_scenario()
    exp, g = cr.plan_cem_loop(shift=0, obs=keep_out, w_obst=np.inf, P=CHECK_PERIOD)
    assert any((c == np.inf).any() for step in exp for c in step[0]), "no candidate entered a disc: the case tests nothing"
    _cem_loop(cr.CEM, shift=0, obstacles=torch.from_numpy(keep_out).to(DEV), w_obst=float("inf"), check=_checker(exp))


def test_one_round_of_one_elite_is_the_argmin_plan():
    sc = pr.SCENARIO
    R, S, n_seg, seg_len = sc["R"], sc["S"], sc["n_seg"], sc["seg_len"]
    g = pr.goals(R)
    ref = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(g, (n_seg, R, 2)))).to(DEV)
    vb = VehicleBatch(R, DEV)
    a = VehiclePlanner(R, S, n_seg, seg_len, DEV, sigma=sc["sigma"], seed=sc["seed"])
    b = VehiclePlanner(R, S, n_seg, seg_len, DEV, sigma=sc["sigma"], seed=sc["seed"])
    for it in range(5):
        a.plan(vb, ref, sc["w_pos"], sc["w_goal"], sc["w_cur"], lam=0.0, shift=1, seed=sc["seed"] + it)
        b.plan_cem(vb, ref, sc["w_pos"], sc["w_goal"], sc["w_cur"], 1, 1, alpha=0.0, shift=1, seed=sc["seed"] + it)
        for name in ("candidates", "cost", "nominal", "best", "best_cost"):
            x, y = getattr(a, name), getattr(b, name)
            assert torch.equal(x.view(torch.int32), y.view(torch.int32)), f"step {it}: {name}"
        vb.rollout(seg_len, sensor_mode=_cabi.RK_SENSOR_PLANT, cmd=a.first_command(), seg_len=seg_len)
