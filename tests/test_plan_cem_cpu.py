"""CPU: the cross-entropy planner's definitions -- the per-robot sigma table in streams.plan_commands_v2, the refit
restated in tests/plan_cem_ref.py on hand-made cases -- its C-ABI struct and argument checks, and the whole CEM planning
loop on the port, which must plan."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import plan_cem_ref as cr
import plan_ref as pr
import roboken_fmskf_robot_controller_b200 as rk
from roboken_fmskf_robot_controller_b200 import _cabi, streams
from test_plan_cpu import PLAN_GOAL_TOLERANCE_M, _buf, _nominal, lib  # noqa: F401  (lib: the module's fixture)

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
f32 = np.float32


def test_refit_struct_matches_the_header(tmp_path):
    lines = ["#include <stdio.h>", "#include <stddef.h>", '#include "robotick.h"', "int main(void) {",
             '  printf("size %zu\\n", sizeof(rk_plan_refit_t));']
    for fname, _ in _cabi.PlanRefit._fields_:
        lines.append(f'  printf("{fname} %zu\\n", offsetof(rk_plan_refit_t, {fname}));')
    lines += ["  return 0;", "}"]
    src = tmp_path / "abi.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "abi"
    subprocess.run(["gcc", "-I" + os.path.join(ROOT, "include"), str(src), "-o", str(exe)], check=True)
    out = subprocess.run([str(exe)], check=True, capture_output=True, text=True).stdout.split()
    got = dict(zip(out[0::2], map(int, out[1::2])))
    assert got.pop("size") == C.sizeof(_cabi.PlanRefit) == 24
    assert got == {f: getattr(_cabi.PlanRefit, f).offset for f, _ in _cabi.PlanRefit._fields_}


def test_sigma_table_sampler_definition():
    n_seg, R, S = 3, 5, 16
    nom = _nominal(n_seg, R)
    sigma = (120.0, 80.0, 0.5)
    plain = streams.plan_commands_v2(nom, S, seed=9, first=40, sigma=sigma)
    same = streams.plan_commands_v2(nom, S, seed=9, first=40, sigma=(1.0, 2.0, 3.0), sigma_table=cr.sigma_cells(sigma, n_seg, R))
    assert np.array_equal(plain.view(np.uint32), same.view(np.uint32)), "a broadcast table must give the plain sampler's bits"
    tab = np.random.default_rng(1).uniform(0.0, 200.0, (n_seg, R, 4)).astype(np.float32)
    tab[1, 2, :3] = 0.0  # no noise at all: every candidate of robot 2, segment 1 is its nominal
    got = streams.plan_commands_v2(nom, S, seed=9, first=40, sigma_table=tab).reshape(n_seg, R, S)
    for f in ("vx", "vy", "vth"):
        assert (got[f][1, 2].view(np.uint32) == got[f][1, 2, 0].view(np.uint32)).all(), f
    # the scale of cell [s, r] is that segment's and robot's alone
    tab2 = tab.copy()
    tab2[0, 4, 0] *= 2
    got2 = streams.plan_commands_v2(nom, S, seed=9, first=40, sigma_table=tab2).reshape(n_seg, R, S)
    diff = got2["vx"] != got["vx"]
    assert diff[0, 4, 1:].any() and not diff[0, :4].any() and not diff[1:].any()


def _cand(vals):
    """One robot's candidates in every one of 2 segments, vx = vals, vy = 2 * vals (segment 1: + 1000), vth = -vals / 100."""
    S = len(vals)
    c = np.zeros((2, S), dtype=pr.CMD_DT)
    v = np.asarray(vals, dtype=np.float32)
    for s in range(2):
        c["vx"][s], c["vy"][s], c["vth"][s] = v + f32(1000 * s), f32(2) * v, -v / f32(100)
    c["kind"] = _cabi.RK_CMD_MOVE
    return c


def _mean_sd(x):
    """The header's statistics of one axis over members x (ascending j), float32 step by step."""
    acc = f32(x[0])
    for v in x[1:]:
        acc = f32(acc + f32(v))
    m = f32(acc / f32(len(x)))
    q = f32(0)
    for v in x:
        d = f32(f32(v) - m)
        q = f32(q + f32(d * d))
    return m, f32(np.sqrt(f32(q / f32(len(x)))))


def test_elite_order_ties_zeros_and_nonfinite():
    c = np.array([2, 1, 2, 2, 0, 3], dtype=np.float32)
    assert list(cr.elites(c, 1, 6, 3)[0]) == [0, 1, 4]  # the tie at the threshold goes to the lowest j
    assert list(cr.elites(c, 1, 6, 4)[0]) == [0, 1, 2, 4]
    z = np.array([1.0, -0.0, 0.0, -0.0], dtype=np.float32)
    assert list(cr.elites(z, 1, 4, 1)[0]) == [1] and list(cr.elites(z, 1, 4, 2)[0]) == [1, 2]  # -0 equals +0
    assert list(cr.elites(np.array([0.0, -0.0], np.float32), 1, 2, 1)[0]) == [0]
    odd = np.array([np.nan, np.inf, -np.inf, 5, 4, np.nan], dtype=np.float32)
    assert list(cr.elites(odd, 1, 6, 6)[0]) == [3, 4]  # fewer finite costs than k: all of them
    assert cr.elites(np.array([np.nan, np.inf, -np.inf], np.float32), 1, 3, 2)[0].size == 0
    assert list(cr.elites(np.array([3, -1, 7, -5], np.float32), 1, 4, 4)[0]) == [0, 1, 2, 3]


@pytest.mark.parametrize("shift", [0, 1])
def test_refit_statistics_by_hand(shift):
    vals = [3.0, -7.5, 0.1, 12.0, 4.25, -0.3]
    cost = np.array([5, 1, np.nan, 1, 0, np.inf], dtype=np.float32)  # elites of k = 3: j = 1, 3, 4
    cand = _cand(vals)
    sig_in = np.array([[[10, 20, 0.3, 7]], [[11, 21, 0.4, 8]]], dtype=np.float32)
    nom, sig, best, bc = cr.refit(cost, cand, sig_in, 1, 6, 3, sigma_min=(0.0, 3.0, 0.0), shift=shift)
    assert best[0] == 4 and bc[0] == 0
    ss = min(shift, 1)
    for a, f in enumerate(("vx", "vy", "vth")):
        m, sd = _mean_sd(cand[f][ss, [1, 3, 4]])
        assert nom[f][0, 0].view(np.uint32) == m.view(np.uint32), f
        assert sig[0, 0, a].view(np.uint32) == np.fmax(sd, f32((0.0, 3.0, 0.0)[a])).view(np.uint32), f
    assert nom["kind"][0, 0] == _cabi.RK_CMD_MOVE and sig[0, 0, 3] == 0
    # smoothing toward candidate 0 and the incoming sigma of the source segment
    nom2, sig2, _, _ = cr.refit(cost, cand, sig_in, 1, 6, 3, alpha=0.25, shift=shift)
    m, sd = _mean_sd(cand["vy"][ss, [1, 3, 4]])
    a, b = f32(0.25), f32(1) - f32(0.25)
    assert nom2["vy"][0, 0] == f32(f32(a * cand["vy"][ss, 0]) + f32(b * m))
    assert sig2[0, 0, 1] == f32(f32(a * sig_in[ss, 0, 1]) + f32(b * sd))


def test_refit_one_elite_is_the_argmin_and_all_elites_the_mean():
    vals = np.random.default_rng(2).uniform(-300, 300, 9).astype(np.float32)
    cost = np.random.default_rng(3).uniform(0, 1, 9).astype(np.float32)
    cand = _cand(vals)
    sig_in = cr.sigma_cells((1, 1, 1), 2, 1)
    nom, sig, best, _ = cr.refit(cost, cand, sig_in, 1, 9, 1, sigma_min=(0.5, 0.0, 0.25))
    sel, sbest, _ = pr.select_argmin(cost, cand, 1, 9, 1)
    assert best[0] == sbest[0] == np.argmin(cost)
    assert np.array_equal(nom.view(np.uint32), sel.view(np.uint32))
    assert np.array_equal(sig[..., :3], np.broadcast_to(np.array([0.5, 0.0, 0.25], np.float32), (2, 1, 3)))
    nom, _, _, _ = cr.refit(cost, cand, sig_in, 1, 9, 9, shift=0)
    for s in range(2):
        assert nom["vx"][s, 0] == _mean_sd(cand["vx"][s])[0]


def test_refit_without_a_finite_cost_copies_best_and_sigma():
    cand = _cand([1.0, 2.0, 3.0, 4.0])
    sig_in = np.random.default_rng(4).uniform(1, 9, (2, 1, 4)).astype(np.float32)
    for cost, b in (([np.nan, np.nan, np.nan, np.nan], 0), ([np.nan, np.inf, -np.inf, np.inf], 2)):
        nom, sig, best, _ = cr.refit(np.array(cost, np.float32), cand, sig_in, 1, 4, 2, shift=1)
        assert best[0] == b
        assert np.array_equal(nom.view(np.uint32), cand[[1, 1]][:, [b]].view(np.uint32))
        assert np.array_equal(sig.view(np.uint32), sig_in[[1, 1]].view(np.uint32))  # bit for bit, word 3 included


def _refit_args(a, **kw):
    """A valid rk_plan_refit call on the aligned buffer at a (R = 1, S = 4, n_seg = 2), overridden by kw."""
    rf = _cabi.PlanRefit()
    rf.elite, rf.alpha = kw.pop("elite", 2), kw.pop("alpha", 0.0)
    rf.sigma_min[:] = kw.pop("sigma_min", (0.0, 0.0, 0.0))
    p = lambda off: C.c_void_p(a.value + off)  # noqa: E731
    args = dict(cost=p(0), cmd=p(256), sig_in=p(1024), R=1, S=4, n_seg=2, rf=C.byref(rf), shift=0, nom=p(2048), sig_out=p(3072))
    args.update(kw)
    return (args["cost"], args["cmd"], args["sig_in"], args["R"], args["S"], args["n_seg"], args["rf"], args["shift"], args["nom"],
            args["sig_out"], None, None, None), rf


def test_cem_argument_errors(lib):  # noqa: F811
    p, s = rk.default_params(), _cabi.PlanSample()
    keep, a = _buf(4096)
    at = lambda off: C.c_void_p(a.value + off)  # noqa: E731
    refit, sample = lib.rk_plan_refit, lib.rk_plan_sample_commands_sigma
    bad = [
        dict(R=-1), dict(S=0), dict(S=1 << 30, n_seg=4, elite=1), dict(shift=2), dict(shift=-1),
        dict(cost=None), dict(cost=at(2)), dict(cmd=at(264)), dict(nom=None), dict(nom=at(272)),  # nom overlaps cmd
        dict(rf=None), dict(elite=0), dict(elite=5), dict(alpha=float("nan")), dict(alpha=-0.1), dict(alpha=1.5),
        dict(sigma_min=(0.0, -1.0, 0.0)), dict(sigma_min=(0.0, 0.0, float("nan"))), dict(sigma_min=(float("inf"), 0.0, 0.0)),
        dict(sig_in=None), dict(sig_in=at(1032)), dict(sig_out=None), dict(sig_out=at(3080)),
        dict(sig_out=at(1040)),  # overlaps sigma_in
        dict(sig_out=at(1024), shift=1),  # in place, but with a shift
    ]
    for k, kw in enumerate(bad):
        args, rf = _refit_args(a, **kw)
        assert refit(*args) == 1, f"refit case {k} {kw}: {lib.rk_last_error()}"
        assert lib.rk_last_error(), f"refit case {k}: no message"
    bad_sample = [
        lambda: sample(C.byref(p), C.byref(s), a, None, 1, 4, 2, at(2048), None),
        lambda: sample(C.byref(p), C.byref(s), a, at(1032), 1, 4, 2, at(2048), None),
        lambda: sample(C.byref(p), C.byref(s), a, at(2064), 1, 4, 2, at(2048), None),  # inside d_cmd
        lambda: sample(C.byref(p), C.byref(s), a, at(1024), 1, 0, 2, at(2048), None),
        lambda: sample(C.byref(p), C.byref(s), a, at(1024), 2, 4, 2, at(32), None),  # d_cmd overlaps the nominal
        lambda: sample(None, C.byref(s), a, at(1024), 1, 4, 2, at(2048), None),
    ]
    for k, call in enumerate(bad_sample):
        assert call() == 1, f"sample case {k}: {lib.rk_last_error()}"
        assert lib.rk_last_error(), f"sample case {k}: no message"
    # R == 0 is a no-op
    args, rf = _refit_args(a, R=0, cost=None, cmd=None, sig_in=None, nom=None, sig_out=None)
    assert refit(*args) == 0
    assert sample(C.byref(p), C.byref(s), None, None, 0, 4, 2, None, None) == 0


def test_cem_entries_fail_without_a_device(lib):  # noqa: F811
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    p, s = rk.default_params(), _cabi.PlanSample()
    keep, a = _buf(4096)
    assert lib.rk_plan_sample_commands_sigma(C.byref(p), C.byref(s), a, C.c_void_p(a.value + 1024), 1, 4, 2, C.c_void_p(a.value + 2048),
                                             None) == 2
    assert b"no CPU fallback" in lib.rk_last_error()
    for kw in (dict(), dict(sig_out=C.c_void_p(a.value + 1024)), dict(alpha=1.0, elite=4)):  # in place with shift 0 is allowed
        args, rf = _refit_args(a, **kw)
        assert lib.rk_plan_refit(*args) == 2, kw
        assert b"no CPU fallback" in lib.rk_last_error()


def test_cpu_cem_planning_loop_reaches_the_goals():
    out, g = cr.plan_cem_loop()
    R = pr.SCENARIO["R"]
    d = pr.distances(out[-1][2], R, g)
    assert (d < PLAN_GOAL_TOLERANCE_M).all(), f"distances to the goals after CEM planning: {d} (from {np.hypot(g[:, 0], g[:, 1])})"
    costs = np.array([c[-1].reshape(R, -1).min(axis=1) for c, _, _ in out])
    assert (costs[-1] < costs[0]).all()
