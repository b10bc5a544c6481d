"""CPU: the sampling planner's definitions (streams.plan_commands_v2, the stage cost, argmin selection), its C-ABI
structs and argument checks, and the whole planning loop restated on the port (tests/plan_ref.py) -- which must plan."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import plan_ref as pr
import roboken_fmskf_robot_controller_b200 as rk
from roboken_fmskf_robot_controller_b200 import _cabi, build, streams

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _nominal(n_seg, R, seed=3, scale=150.0):
    rng = np.random.default_rng(seed)
    nom = np.zeros((n_seg, R), dtype=pr.CMD_DT)
    nom["vx"] = rng.uniform(-scale, scale, (n_seg, R)).astype(np.float32)
    nom["vy"] = rng.uniform(-scale, scale, (n_seg, R)).astype(np.float32)
    nom["vth"] = rng.uniform(-1.0, 1.0, (n_seg, R)).astype(np.float32)
    nom["kind"] = rng.integers(0, 3, (n_seg, R))
    return nom


def test_sample_zero_is_the_nominal():
    nom = _nominal(5, 7)
    c = streams.plan_commands_v2(nom, 16, seed=11).reshape(5, 7, 16)
    for f in ("vx", "vy", "vth"):
        assert np.array_equal(c[f][:, :, 0].view(np.uint32), nom[f].view(np.uint32)), f
    assert (c["kind"] == _cabi.RK_CMD_MOVE).all()
    assert not np.array_equal(c["vx"][:, :, 1], nom["vx"])


def test_samples_within_both_limits():
    p = rk.default_params()
    nom = _nominal(4, 6, scale=380.0)
    c = streams.plan_commands_v2(nom, 64, seed=2, sigma=(400.0, 400.0, 30.0))
    ln = np.sqrt(c["vx"] * c["vx"] + c["vy"] * c["vy"], dtype=np.float32)
    L, rl = np.float32(p.limit_speed_mmps), np.float32(p.limit_rot_radps)
    assert (ln <= L * np.float32(1.000001)).all() and (np.abs(c["vth"]) <= rl).all()
    assert (ln > L * np.float32(0.999)).any() and (np.abs(c["vth"]) == rl).any()  # both limiters acted


def test_noise_depends_only_on_seed_and_global_index():
    nom = _nominal(3, 10)
    full = streams.plan_commands_v2(nom, 8, seed=7, first=1000)
    a = streams.plan_commands_v2(nom[:, :4], 8, seed=7, first=1000)
    b = streams.plan_commands_v2(np.ascontiguousarray(nom[:, 4:]), 8, seed=7, first=1004)
    assert np.array_equal(full.view(np.uint32), np.concatenate([a, b], axis=1).view(np.uint32))
    other = streams.plan_commands_v2(nom, 8, seed=8, first=1000)
    assert not np.array_equal(full["vx"], other["vx"])


def test_noise_is_about_unit_normal():
    h = streams.h32(0x5EED, 40, np.arange(200_000, dtype=np.uint64), 3)
    xi = streams.plan_xi_v2(h).astype(np.float64)
    assert np.abs(xi.mean(axis=0)).max() < 0.01
    assert np.abs(xi.var(axis=0) - 1.0).max() < 0.01
    assert np.abs(xi).max() <= 2.0 * 1.7320508 + 1e-6  # Irwin-Hall: bounded


def test_plan_structs_match_the_header(tmp_path):
    structs = {"rk_plan_sample_t": _cabi.PlanSample, "rk_plan_cost_t": _cabi.PlanCost}
    lines = ["#include <stdio.h>", "#include <stddef.h>", '#include "robotick.h"', "int main(void) {"]
    for cname, cls in structs.items():
        lines.append(f'  printf("{cname} size %zu\\n", sizeof({cname}));')
        for fname, _ in cls._fields_:
            lines.append(f'  printf("{cname} {fname} %zu\\n", offsetof({cname}, {fname}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "abi.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "abi"
    subprocess.run(["gcc", "-I" + os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout
    seen = 0
    for line in out.splitlines():
        cname, fname, val = line.split()
        cls = structs[cname]
        got = C.sizeof(cls) if fname == "size" else getattr(cls, fname).offset
        assert got == int(val), f"{cname}.{fname}: header {val}, ctypes {got}"
        seen += 1
    assert seen == sum(len(c._fields_) + 1 for c in structs.values())
    assert C.sizeof(_cabi.PlanSample) == 32 and C.sizeof(_cabi.PlanCost) == 24


@pytest.fixture(scope="module")
def lib():
    build.build()
    return rk.load()


def _buf(nbytes):
    b = (C.c_uint8 * (nbytes + 16))()
    return b, C.c_void_p((C.addressof(b) + 15) & ~15)


def test_plan_argument_errors(lib):
    p = rk.default_params()
    s, c = _cabi.PlanSample(), _cabi.PlanCost()
    keep, a = _buf(4096)
    c.d_ref = a.value
    sample, roll, sel = lib.rk_plan_sample_commands, lib.rk_plan_rollout, lib.rk_plan_select
    bad = [
        lambda: sample(C.byref(p), C.byref(s), a, -1, 4, 2, a, None),
        lambda: sample(C.byref(p), C.byref(s), a, 1, 0, 2, a, None),
        lambda: sample(C.byref(p), C.byref(s), a, 1, 1 << 30, 4, a, None),  # n_seg * S >= 2^32
        lambda: sample(C.byref(p), C.byref(s), C.c_void_p(a.value + 8), 1, 4, 2, C.c_void_p(a.value + 2048), None),
        lambda: sample(C.byref(p), C.byref(s), a, 2, 4, 2, C.c_void_p(a.value + 32), None),  # overlaps the nominal
        lambda: roll(C.byref(p), a, 1, 4, a, 2, 0, C.byref(c), a, None),  # seg_len < 1
        lambda: roll(C.byref(p), a, -1, 4, a, 2, 10, C.byref(c), a, None),
        lambda: roll(C.byref(p), C.c_void_p(a.value + 4), 1, 4, a, 2, 10, C.byref(c), a, None),
        lambda: roll(C.byref(p), a, 1, 1 << 30, a, 4, 10, C.byref(c), a, None),
        lambda: sel(a, a, 1, 4, 2, 0.0, 2, C.c_void_p(a.value + 2048), None, None, None),  # shift >= n_seg
        lambda: sel(a, a, 1, 4, 2, 0.0, -1, C.c_void_p(a.value + 2048), None, None, None),
        lambda: sel(a, a, 1, 4, 2, -1.0, 0, C.c_void_p(a.value + 2048), None, None, None),
        lambda: sel(a, a, 1, 4, 2, float("inf"), 0, C.c_void_p(a.value + 2048), None, None, None),
        lambda: sel(a, a, 1, 4, 2, float("nan"), 0, C.c_void_p(a.value + 2048), None, None, None),
        lambda: sel(a, a, 1, 4, 2, 0.0, 0, C.c_void_p(a.value + 64), None, None, None),  # aliases d_cmd
        lambda: sel(a, a, 1, 0, 2, 0.0, 0, C.c_void_p(a.value + 2048), None, None, None),
    ]
    for k, call in enumerate(bad):
        assert call() == 1, f"case {k}: {lib.rk_last_error()}"
        assert lib.rk_last_error(), f"case {k}: no message"
    # R == 0 is a no-op
    assert sample(C.byref(p), C.byref(s), None, 0, 4, 2, None, None) == 0
    assert roll(C.byref(p), None, 0, 4, None, 2, 10, C.byref(c), None, None) == 0
    assert sel(None, None, 0, 4, 2, 0.0, 0, None, None, None, None) == 0


def test_plan_entries_fail_without_a_device(lib):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    p = rk.default_params()
    s, c = _cabi.PlanSample(), _cabi.PlanCost()
    keep, a = _buf(1 << 16)
    c.d_ref = a.value
    b = C.c_void_p(a.value + 32768)
    assert lib.rk_plan_sample_commands(C.byref(p), C.byref(s), a, 1, 4, 2, b, None) == 2
    assert b"no CPU fallback" in lib.rk_last_error()
    assert lib.rk_plan_rollout(C.byref(p), a, 1, 4, b, 2, 10, C.byref(c), a, None) == 2
    assert lib.rk_plan_select(a, a, 1, 4, 2, 0.5, 1, b, None, None, None) == 2


def test_stage_cost_and_argmin_definitions():
    # two segments, two robots x two candidates, hand-made trace rows
    R, S, seg_len = 2, 2, 3
    tr = np.zeros((2 * seg_len, 16, R * S), dtype=np.uint32)
    pos = np.array([[0.5, 0.25], [1.0, -1.0], [0.0, 0.0], [2.0, 2.0]], dtype=np.float32)
    tr[seg_len - 1, 0], tr[seg_len - 1, 1] = pos[:, 0].view(np.uint32), pos[:, 1].view(np.uint32)
    tr[2 * seg_len - 1, 0], tr[2 * seg_len - 1, 1] = pos[:, 0].view(np.uint32), pos[:, 1].view(np.uint32)
    tr[2 * seg_len - 1, 9] = np.array([-3, 0, 1, 2], dtype=np.int32).view(np.uint32)
    ref = np.zeros((2, R, 2), dtype=np.float32)
    J = pr.stage_cost(tr, ref, S, seg_len, 1.0, 10.0, 0.5)
    e = (pos ** 2).sum(axis=1)
    np.testing.assert_array_equal(J, (e + 10.0 * e + 0.5 * np.array([9, 0, 1, 4])).astype(np.float32))
    cand = np.zeros((3, R * S), dtype=pr.CMD_DT)
    cand["vx"] = np.arange(3 * R * S, dtype=np.float32).reshape(3, R * S)
    cost = np.array([np.nan, np.nan, 1.0, 1.0], dtype=np.float32)
    nom, best, bc = pr.select_argmin(cost, cand, R, S, shift=1)
    assert list(best) == [0, 0] and np.isnan(bc[0]) and bc[1] == 1.0
    assert list(nom["vx"][:, 1]) == [6.0, 10.0, 10.0]  # segments 1, 2, 2 of candidate 2


# The planning loop on the port, from power-on: the final distance of every robot to its goal stays below this bound
# (the robots start 205 - 281 mm from their goals; this run ends 10.5 - 44.7 mm from them after 1.5 s).
PLAN_GOAL_TOLERANCE_M = 0.06


def test_cpu_planning_loop_reaches_the_goals():
    out, g = pr.plan_loop()
    d0 = np.hypot(g[:, 0], g[:, 1])
    d = pr.distances(out[-1][2], pr.SCENARIO["R"], g)
    assert (d < PLAN_GOAL_TOLERANCE_M).all(), f"distances to the goals after planning: {d} (from {d0})"
    costs = np.array([c.reshape(pr.SCENARIO["R"], -1).min(axis=1) for c, _, _ in out])
    assert (costs[-1] < costs[0]).all()
