"""GPU: rk_plan_rollout_field on every compiled kObstMoving instantiation -- each row of vdt_instances.MATRIX, costs and paths
bit for bit against tests/plan_field_ref.py with one and three fields (offset windows, +inf, NaN and negative cells, robots
with no field, end positions off the window), with and without a map, and the launched kernel confirmed under
torch.profiler -- and, without a field (field NULL or w_field = 0), rk_plan_rollout_map's bits and kernel.

These tests sit among test_vdt_instances_*_gpu.py for the profiler reason test_vdt_instances_map_gpu.py's docstring gives.
"""
import ctypes as C

import numpy as np
import pytest
import torch

import plan_field_ref as pf
import vdt_instances as vi
from roboken_fmskf_robot_controller_b200 import _cabi
from roboken_fmskf_robot_controller_b200.planner import CostToGo
from test_plan_gpu import _cells, _u32
from test_plan_map_gpu import DEV, W_OBST, _costmap, _host, _table, _world
from test_plan_obst_gpu import N_SEG, R, S, SEG_LEN, W, _case
from test_vdt_instances_gpu import options  # noqa: F401  (the fixture)
from test_vdt_instances_gpu import _params as _row_params
from test_vdt_instances_map_gpu import _launched

import plan_map_ref as pmr
import roboken_fmskf_robot_controller_b200 as rk

pytestmark = pytest.mark.gpu
_TRACE = {}


def _ctg(cm, n_fields, seed, outside=2.5):
    """A caller's field on the map's grid: float32 [n_fields, 36, 20] uniform in [-0.2, 1) with 5 % NaN and 3 % +inf,
    windows at offsets (2, 3) + f, and a field index per robot with two robots out of range."""
    rng = np.random.default_rng(seed)
    f = rng.uniform(-0.2, 1.0, (n_fields, 36, 20)).astype(np.float32)
    f[rng.random(f.shape) < 0.05] = np.nan
    f[rng.random(f.shape) < 0.03] = np.inf
    offs = np.array([[2 + k, 3 + k] for k in range(n_fields)], np.int32)
    field_of = rng.integers(0, n_fields, R).astype(np.int32)
    field_of[[0, 5]] = -1, n_fields
    return CostToGo(torch.from_numpy(f).to(DEV), cm, offsets=torch.from_numpy(offs).to(DEV), field_of=torch.from_numpy(field_of).to(DEV),
                    outside=outside)


def _hostfield(ctg, w_field):
    return pf.HostField(ctg.field.cpu().numpy(), ctg.offsets.cpu().numpy(), ctg.field_of.cpu().numpy(), np.float32(ctg.costmap.x0),
                        np.float32(ctg.costmap.y0), np.float32(ctg.costmap.inv_res), np.float32(ctg.outside), np.float32(w_field))


def _field_rollout(vb, cand, ref, obs, P, cm, w_map, ctg, w_field, params=None, path=True):
    """rk_plan_rollout_field: (cost float32 [R*S], path float32 [n_ck, R*S, 2] or None)."""
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
    o.d_obs, o.m, o.check_period, o.w_obst = obs_d.data_ptr(), obs.shape[1], P, W_OBST
    mp = None if cm is None else cm.struct(w_map)
    fd = None if ctg is None else ctg.struct(w_field)
    _cabi.check(lib.rk_plan_rollout_field(params or rk.default_params(), vb.state.data_ptr(), R, S, cand_d.data_ptr(), N_SEG, SEG_LEN, c, o,
                                          None if mp is None else C.byref(mp), None if fd is None else C.byref(fd),
                                          None if pth is None else pth.data_ptr(), cost.data_ptr(), torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return cost.cpu().numpy(), None if pth is None else pth.cpu().numpy()


@pytest.mark.parametrize("row", vi.MATRIX, ids=vi.row_id)
def test_field_costs_and_paths_bit_exact_on_every_row(row, options):  # noqa: F811
    p = _row_params(row)
    options(row)
    vb, src, ref, cand = _case()
    key = (row["kd"], row["ff_limit"])
    if key not in _TRACE:
        _TRACE[key] = pmr.port_trace(src, R, S, cand, SEG_LEN, params=p)
    trace = _TRACE[key]
    exp_kernel = vi.expected_kernel("moving", **row)
    cm = _costmap(_world(src, 1, np.inf, seed=1))
    fields = {1: _ctg(cm, 1, seed=11), 3: _ctg(cm, 3, seed=13, outside=np.inf)}  # finite and +inf off the window
    cases = [(P, m, nf, with_map) for P in (5, SEG_LEN) for m in (0, 3) for nf in fields for with_map in (False, True)]

    def launch_all():
        out = {}
        for P, m, nf, with_map in cases:
            obs = _table(src, N_SEG * SEG_LEN // P, m, seed=10 * m + P)
            out[(P, m, nf, with_map)] = (obs,) + _field_rollout(vb, cand, ref, obs, P, cm if with_map else None, 40.0, fields[nf], 7.5, params=p)
        return out

    got_all, ran = _launched(launch_all)
    priced_inf = priced_finite = False
    assert ran == {exp_kernel}, f"{vi.row_id(row)}: launched {sorted(ran)}, expected {exp_kernel}"
    for (P, m, nf, with_map), (obs, got, path) in got_all.items():
        what = f"{vi.row_id(row)} P={P} m={m} fields={nf} map={with_map}"
        hf = _hostfield(fields[nf], 7.5)
        exp, O, exp_path = pf.candidate_costs_field(src, R, S, cand, SEG_LEN, ref, *W, obs, P, W_OBST, _host(cm, 40.0) if with_map else None, hf,
                                                    trace=trace)
        assert (O > 0).any(), f"{what}: the field must price some candidates"
        priced_inf |= bool(np.isinf(O).any())
        priced_finite |= bool(((O > 0) & np.isfinite(O)).any())
        np.testing.assert_array_equal(got.view(np.uint32), exp.view(np.uint32), err_msg=what)
        np.testing.assert_array_equal(path.view(np.uint32), exp_path.view(np.uint32), err_msg=f"{what}: path")
    assert priced_inf and priced_finite, "some candidates must end on +inf (a +inf cell, or off a window with outside = +inf), some on finite cells"
    assert np.array_equal(_u32(vb.state), src), "rk_plan_rollout_field wrote the source states"


@pytest.mark.parametrize("m", [0, 3])
def test_without_a_field_it_is_the_map_rollout(m):
    from test_plan_map_gpu import _map_rollout

    vb, src, ref, cand = _case(seed=7)
    P = 5
    obs = _table(src, N_SEG * SEG_LEN // P, m, seed=4)
    cm = _costmap(_world(src, 1, np.inf, seed=2))
    ctg = _ctg(cm, 1, seed=3)
    for cmap, w_map in ((cm, 30.0), (None, 0.0)):
        (exp, exp_path), ran_map = _launched(lambda: _map_rollout(vb, cand, ref, obs, P, W_OBST, cmap, w_map))
        for what, (fd, w_field) in {"field NULL": (None, 1.0), "w_field 0": (ctg, 0.0)}.items():
            (got, got_path), ran = _launched(lambda: _field_rollout(vb, cand, ref, obs, P, cmap, w_map, fd, w_field))
            np.testing.assert_array_equal(got.view(np.uint32), exp.view(np.uint32), err_msg=f"{what}, map={cmap is not None}")
            np.testing.assert_array_equal(got_path.view(np.uint32), exp_path.view(np.uint32), err_msg=what)
            assert ran == ran_map == {vi.expected_kernel("moving")}, f"{what}: launched {sorted(ran)}"
