"""CPU: keep-out discs in the planner's candidate cost (rk_plan_rollout_obstacles) -- the C-ABI struct and argument
checks, the obstacle-cost definition on hand-made trace rows, and the lambda = 0 planning loop on the port with discs
(tests/plan_obst_ref.py), which must keep every robot out of its disc and still reach the goal."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import plan_obst_ref as por
import plan_ref as pr
import roboken_fmskf_robot_controller_b200 as rk
from roboken_fmskf_robot_controller_b200 import _cabi, build
from test_plan_cpu import PLAN_GOAL_TOLERANCE_M

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_obstacle_struct_matches_the_header(tmp_path):
    cls = _cabi.PlanObstacles
    lines = ["#include <stdio.h>", "#include <stddef.h>", '#include "robotick.h"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(rk_plan_obstacles_t));']
    for fname, _ in cls._fields_:
        lines.append(f'  printf("{fname} %zu\\n", offsetof(rk_plan_obstacles_t, {fname}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "abi.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "abi"
    subprocess.run(["gcc", "-I" + os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    seen = 0
    for line in out.splitlines():
        fname, val = line.split()
        got = C.sizeof(cls) if fname == "size" else getattr(cls, fname).offset
        assert got == int(val), f"rk_plan_obstacles_t.{fname}: header {val}, ctypes {got}"
        seen += 1
    assert seen == len(cls._fields_) + 1 and C.sizeof(cls) == 24


@pytest.fixture(scope="module")
def lib():
    build.build()
    return rk.load()


def _buf(nbytes):
    b = (C.c_uint8 * (nbytes + 16))()
    return b, C.c_void_p((C.addressof(b) + 15) & ~15)


def _obst(d_obs, m, P, w):
    o = _cabi.PlanObstacles()
    o.d_obs, o.m, o.check_period, o.w_obst = d_obs, m, P, w
    return o


def test_obstacle_argument_errors(lib):
    p = rk.default_params()
    c = _cabi.PlanCost()
    keep, a = _buf(4096)
    c.d_ref = a.value
    roll = lib.rk_plan_rollout_obstacles
    bad = {
        "m < 0": _obst(a.value, -1, 10, 1.0),
        "m > 0, d_obs NULL": _obst(None, 2, 10, 1.0),
        "m > 0, d_obs not 16-byte aligned": _obst(a.value + 8, 2, 10, 1.0),
        "P < 1": _obst(a.value, 2, 0, 1.0),
        "seg_len % P != 0": _obst(a.value, 2, 3, 1.0),
        "w_obst < 0": _obst(a.value, 2, 5, -1.0),
        "w_obst NaN": _obst(a.value, 2, 5, float("nan")),
    }
    for what, o in bad.items():
        assert roll(C.byref(p), a, 1, 4, a, 2, 10, C.byref(c), C.byref(o), a, None) == 1, f"{what}: {lib.rk_last_error()}"
        assert b"rk_plan_rollout_obstacles" in lib.rk_last_error(), f"{what}: no message"
    ok = _obst(a.value, 2, 5, float("inf"))
    # rk_plan_rollout's own checks
    assert roll(C.byref(p), a, 1, 4, a, 2, 0, C.byref(c), C.byref(ok), a, None) == 1  # seg_len < 1
    assert roll(C.byref(p), a, -1, 4, a, 2, 10, C.byref(c), C.byref(ok), a, None) == 1
    assert roll(C.byref(p), C.c_void_p(a.value + 4), 1, 4, a, 2, 10, C.byref(c), C.byref(ok), a, None) == 1
    assert roll(C.byref(p), a, 1, 1 << 30, a, 4, 10, C.byref(c), C.byref(ok), a, None) == 1
    assert roll(None, a, 1, 4, a, 2, 10, C.byref(c), C.byref(ok), a, None) == 1
    # R == 0 is a no-op
    assert roll(C.byref(p), None, 0, 4, None, 2, 10, C.byref(c), C.byref(ok), None, None) == 0
    assert roll(C.byref(p), None, 0, 4, None, 2, 10, C.byref(c), None, None, None) == 0


def test_obstacle_rollout_fails_without_a_device(lib):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    p = rk.default_params()
    c = _cabi.PlanCost()
    keep, a = _buf(1 << 16)
    c.d_ref = a.value
    b = C.c_void_p(a.value + 32768)
    for o in (_obst(a.value, 3, 5, 2.0), _obst(None, 0, 5, 2.0), None):
        assert lib.rk_plan_rollout_obstacles(C.byref(p), a, 1, 4, b, 2, 10, C.byref(c), None if o is None else C.byref(o), a, None) == 2
        assert b"no CPU fallback" in lib.rk_last_error()


def _trace(xy_rows):
    """Trace rows [K, 16, n] with the position words of xy_rows float32 [K, n, 2]."""
    xy = np.asarray(xy_rows, dtype=np.float32)
    tr = np.zeros((xy.shape[0], 16, xy.shape[1]), dtype=np.uint32)
    tr[:, 0], tr[:, 1] = xy[:, :, 0].view(np.uint32), xy[:, :, 1].view(np.uint32)
    return tr


def test_obstacle_cost_definition():
    f32 = np.float32
    K, P = 6, 2  # checkpoints are rows 1, 3, 5
    xy = np.full((K, 2, 2), 5.0, dtype=np.float32)  # robot 0, candidates 0 and 1: far away ...
    xy[3, 0] = (0.1, 0.0)  # ... except candidate 0 at checkpoint 2 (row 3)
    xy[2, 1] = (0.0, 0.0)  # candidate 1 sits on the centre between two checkpoints: not seen
    obs = np.array([[[0.0, 0.0, 0.5, 0.0]]], dtype=np.float32)
    O = por.obstacle_cost(_trace(xy), obs, 2, P, 3.0)
    assert O[0] == f32(3.0) * (f32(0.25) - f32(0.1) * f32(0.1)) and O[1] == 0.0

    # exactly on the boundary: pen = 0 adds nothing; one ulp inside adds
    xy = np.full((2, 1, 2), 0.0, dtype=np.float32)
    xy[1, 0] = (0.75, 0.0)
    on = np.array([[[0.0, 0.0, 0.75, 0.0]]], dtype=np.float32)
    assert por.obstacle_cost(_trace(xy), on, 1, 2, 1.0)[0] == 0.0
    inside = on.copy()
    inside[0, 0, 2] = np.nextafter(f32(0.75), f32(1))
    assert por.obstacle_cost(_trace(xy), inside, 1, 2, 1.0)[0] > 0.0

    # NaN radius or centre: nothing; w = inf: +inf once inside, never NaN
    nan_r = np.array([[[0.75, 0.0, np.nan, 0.0]], [[np.nan, 0.0, 1.0, 0.0]]], dtype=np.float32)
    assert por.obstacle_cost(_trace(xy), nan_r, 1, 1, 1.0)[0] == 0.0
    assert por.obstacle_cost(_trace(xy), inside, 1, 2, np.inf)[0] == np.inf
    assert por.obstacle_cost(_trace(xy), on, 1, 2, np.inf)[0] == 0.0

    # the disc order is part of the definition: pens 1, 2^-24, 2^-24 sum to 1 in this order (1 + 2^-24 is a tie to
    # even) and to 1 + 2^-23 in the reverse order
    xy = np.zeros((1, 1, 2), dtype=np.float32)
    obs = np.zeros((3, 1, 4), dtype=np.float32)
    obs[:, 0, 2] = (1.0, 2.0 ** -12, 2.0 ** -12)
    assert por.obstacle_cost(_trace(xy), obs, 1, 1, 1.0)[0] == f32(1.0)
    assert por.obstacle_cost(_trace(xy), obs[::-1].copy(), 1, 1, 1.0)[0] == f32(1.0 + 2.0 ** -23)


# The planning loop of test_plan_cpu.py with one disc per robot halfway to the goal, 15 mm to the left of the straight
# path, radius 40 mm: the straight path cuts 25 mm into it.  The cost keeps candidates 2 mm further out than the disc
# (P = 5 ticks at no more than 400 mm/s between two checkpoints: 2 mm) with w_obst = +inf, and the robots execute the
# segment the cost checked (shift = 0).  Observed on the port: with the discs every robot keeps 2.0 - 21.8 mm of
# clearance from its disc and ends 3.0 - 30.1 mm from its goal; without them all 8 robots pass 10 - 38 mm deep inside.
DISC_RADIUS_M, DISC_OFFSET_M, CHECK_PERIOD = 0.04, 0.015, 5
KEEP_OUT_M = DISC_RADIUS_M + CHECK_PERIOD * 0.4e-3


def obstacle_scenario():
    """(the discs, the keep-out discs the cost uses), float32 [1, R, 4] each."""
    g = pr.goals(pr.SCENARIO["R"])
    return por.discs_near_the_path(g, DISC_RADIUS_M, DISC_OFFSET_M), por.discs_near_the_path(g, KEEP_OUT_M, DISC_OFFSET_M)


def test_cpu_planning_loop_avoids_the_discs():
    disc, keep_out = obstacle_scenario()
    out, g = por.plan_loop_obst(keep_out, np.inf, CHECK_PERIOD)
    clear = por.min_clearance(out, disc)
    d = pr.distances(out[-1][2], pr.SCENARIO["R"], g)
    assert (clear > 0).all(), f"an executed tick inside a disc: clearance {clear}"
    assert (d < PLAN_GOAL_TOLERANCE_M).all(), f"distances to the goals after planning: {d}"
    free, _ = por.plan_loop_obst(keep_out, 0.0, CHECK_PERIOD)
    assert (por.min_clearance(free, disc) < 0).any(), "without the discs' cost no robot enters a disc: the scenario tests nothing"
