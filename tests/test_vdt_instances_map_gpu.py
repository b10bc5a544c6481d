"""GPU: rk_plan_rollout_map on every compiled kObstMoving instantiation -- each row of vdt_instances.MATRIX, costs and
paths bit for bit against tests/plan_map_ref.py with one and three maps, +inf cells and `outside` under finite and
infinite w_map, and the launched kernel confirmed under torch.profiler -- and, without a map (map NULL or w_map = 0),
rk_plan_rollout_moving's bits and kernel.

These tests sit next to test_vdt_instances_gpu.py so that the suite starts torch.profiler no earlier than it did: when a
profiler session runs before the GPU tests of test_plan_obst_gpu.py .. test_vdt_task_gpu.py, the sessions after them
record no kernels (observed with torch 2.11 on a B200), and test_vdt_instances_gpu.py's checks would fail for it.
"""
import numpy as np
import pytest
import torch
from torch.profiler import ProfilerActivity, profile

import plan_map_ref as pmr
import vdt_instances as vi
from test_plan_fleet_gpu import _moving_rollout
from test_plan_map_gpu import W_OBST, _costmap, _host, _map_rollout, _table, _world
from test_plan_obst_gpu import N_SEG, R, S, SEG_LEN, W, _case
from test_plan_gpu import _u32
from test_vdt_instances_gpu import options  # noqa: F401  (the fixture)
from test_vdt_instances_gpu import _params as _row_params

pytestmark = pytest.mark.gpu
_TRACE = {}


def _launched(fn):
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        out = fn()
        torch.cuda.synchronize()
    return out, {t for t in (vi.parse(e.name) for e in prof.events()) if t is not None}


@pytest.mark.parametrize("row", vi.MATRIX, ids=vi.row_id)
def test_map_costs_and_paths_bit_exact_on_every_row(row, options):  # noqa: F811
    p = _row_params(row)
    options(row)
    vb, src, ref, cand = _case()
    key = (row["kd"], row["ff_limit"])
    if key not in _TRACE:
        _TRACE[key] = pmr.port_trace(src, R, S, cand, SEG_LEN, params=p)
    trace = _TRACE[key]
    exp_kernel = vi.expected_kernel("moving", **row)
    worlds = {1: (_world(src, 1, np.inf, seed=1), 40.0), 3: (_world(src, 3, 0.5, seed=3), np.inf)}  # (world, w_map)
    cases = [(P, m, n_maps) for P in (1, 5, SEG_LEN) for m in (0, 3) for n_maps in worlds]

    def launch_all():
        out = {}
        for P, m, n_maps in cases:
            world, w_map = worlds[n_maps]
            obs = _table(src, N_SEG * SEG_LEN // P, m, seed=10 * m + P)
            cm = _costmap(world)
            out[(P, m, n_maps)] = (obs, cm, w_map) + _map_rollout(vb, cand, ref, obs, P, W_OBST, cm, w_map, params=p)
        return out

    # one profiler session for the row's 12 launches: every one of them must be the row's instantiation (a launch that
    # ran nothing leaves NaN costs, which the comparison below rejects)
    got_all, ran = _launched(launch_all)
    assert ran == {exp_kernel}, f"{vi.row_id(row)}: launched {sorted(ran)}, expected {exp_kernel}"
    for (P, m, n_maps), (obs, cm, w_map, got, path) in got_all.items():
        what = f"{vi.row_id(row)} P={P} m={m} maps={n_maps} w_map={w_map}"
        exp, O, exp_path = pmr.candidate_costs_map(src, R, S, cand, SEG_LEN, ref, *W, obs, P, W_OBST, _host(cm, w_map), trace=trace)
        assert np.isinf(O).any() and np.isfinite(O).any() and (O > 0).any(), f"{what}: the map must price some candidates, not all"
        np.testing.assert_array_equal(got.view(np.uint32), exp.view(np.uint32), err_msg=what)
        np.testing.assert_array_equal(path.view(np.uint32), exp_path.view(np.uint32), err_msg=f"{what}: path")
    assert np.array_equal(_u32(vb.state), src), "rk_plan_rollout_map wrote the source states"


@pytest.mark.parametrize("m", [0, 3])
def test_without_a_map_it_is_the_moving_rollout(m):
    vb, src, ref, cand = _case(seed=6)
    P = 5
    obs = _table(src, N_SEG * SEG_LEN // P, m, seed=4)
    cm = _costmap(_world(src, 1, np.inf, seed=2))
    for path in (False, True):
        exp, exp_path = _moving_rollout(vb, cand, ref, obs, P, W_OBST, path=path)
        for what, (mp, w_map) in {"map NULL": (None, 1.0), "w_map 0": (cm, 0.0)}.items():
            (got, got_path), ran = _launched(lambda: _map_rollout(vb, cand, ref, obs, P, W_OBST, mp, w_map, path=path))
            np.testing.assert_array_equal(got.view(np.uint32), exp.view(np.uint32), err_msg=f"{what}, path={path}")
            entry = "moving" if (m or path) else "plan"  # no discs, no path, no map: rk_plan_rollout's kernel
            assert ran == {vi.expected_kernel(entry)}, f"{what}, path={path}: launched {sorted(ran)}"
            if path:
                np.testing.assert_array_equal(got_path.view(np.uint32), exp_path.view(np.uint32), err_msg=what)
        if path:  # the path does not depend on the map
            _, with_map = _map_rollout(vb, cand, ref, obs, P, W_OBST, cm, np.inf, path=True)
            np.testing.assert_array_equal(with_map.view(np.uint32), exp_path.view(np.uint32))
