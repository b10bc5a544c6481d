"""CPU: pin the RobotManager guard of the plain-C oracle (orc_rmt_guard, orc_atan2f) against the compiled
reference -- src/RobotManager/RM_task_main.cpp and src/Utility/util_mymath.cpp, both unmodified, behind
micro-ROS / FreeRTOS stubs (oracle/ref_harness_rm.cpp) -- and the generated arctangent tables against the
reference's own arrays (SURVEY 8f-2)."""
import os
import re

import numpy as np
import pytest

import oracle_lib as ol
from roboken_fmskf_robot_controller_b200 import _cabi, layout, streams

needs_ref = pytest.mark.skipif(not ol.have_ref("libref_rm.so"), reason="oracle/_ref/libref_rm.so not available")
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(os.path.dirname(__file__), "golden", "rmt_golden.npz")


def generated_tables():
    text = open(os.path.join(ROOT, "oracle", "atan_table.inc")).read()
    assert text == open(os.path.join(ROOT, "roboken-fmskf-robot-controller_b200", "csrc", "atan_table.inc")).read()
    out = []
    for name in ("RK_ATAN_TABLE_BITS", "RK_ATAN_DELIMIT_BITS", "RK_ATAN_WIDTH_BITS"):
        body = text.split("#define " + name)[1].split("#define")[0]
        body = re.sub(r"/\*.*?\*/", "", body, flags=re.S)
        out.append(np.array([int(v, 16) for v in re.findall(r"0x([0-9A-Fa-f]{8})u", body)], dtype=np.uint32).view(np.float32))
    out[0] = out[0][:625]  # the pad word after the table
    return out


def special_values():
    v = [0.0, -0.0, 1e-30, 0.009, 0.01, 0.25819889, 0.2581989, 1.0, 1.0000001, 3.872983346, 572957.7951, 572957.8125, 572958.0, 1e9,
         np.inf, np.nan]
    v = np.array(v + [-x for x in v], dtype=np.float32)
    return v


def reference_tables(kind):
    """The arctangent tables of util_mymath.cpp as the compiled reference holds them; the port's are the generated ones."""
    if kind == "port":
        return generated_tables()
    rt, rd, rw = np.zeros(700, dtype=np.float32), np.zeros(27, dtype=np.float32), np.zeros(26, dtype=np.float32)
    nt = ol.ref("libref_rm.so").ref_rm_atan_tables(rt.ctypes.data, rd.ctypes.data, rw.ctypes.data)
    return [rt[:nt], rd, rw]


def test_generated_atan_tables_equal_the_reference_arrays():
    t, d, w = generated_tables()
    rt, rd, rw = ol.reference_result("rm_atan_tables", reference_tables, "libref_rm.so")
    assert len(rt) == 625 and len(t) == 625 and len(d) == 27 and len(w) == 26
    np.testing.assert_array_equal(t.view(np.uint32), rt.view(np.uint32))
    np.testing.assert_array_equal(d.view(np.uint32), rd.view(np.uint32))
    np.testing.assert_array_equal(w.view(np.uint32), rw.view(np.uint32))


def test_atan_port_equals_ref():
    p = ol.port()
    rng = np.random.default_rng(4)
    xs = np.concatenate([special_values(), generated_tables()[1], np.nextafter(generated_tables()[1], np.float32(np.inf)),
                         (rng.standard_normal(4000) * 3).astype(np.float32), np.exp(rng.uniform(-20, 20, 4000)).astype(np.float32)])
    ys = rng.permutation(xs)

    def values(kind):
        atanf, atan2f = (p.orc_atanf, p.orc_atan2f) if kind == "port" else (ol.ref("libref_rm.so").ref_rm_atanf, ol.ref("libref_rm.so").ref_rm_atan2f)
        return np.float32([atanf(float(x)) for x in xs]), np.float32([atan2f(float(y), float(x)) for y, x in zip(ys, xs)])

    for a, b in zip(values("port"), ol.reference_result("rm_atan", values, "libref_rm.so")):
        np.testing.assert_array_equal(a.view(np.uint32), b.view(np.uint32))
    assert np.float32(p.orc_atan2f(1, 1)) == np.float32(0.785398185)  # SURVEY Appendix D probes
    assert np.float32(p.orc_atanf(0.5)) == np.float32(0.463646978)
    assert np.float32(p.orc_atan2f(-1, -2)) == np.float32(-2.67794585)


@pytest.mark.parametrize("n,K,seed", [(96, 700, 1), (257, 320, 2)])
def test_guard_port_equals_ref(n, K, seed):
    inp = streams.rm_inputs(n, K, seed=seed)
    p = _cabi.RmtParams(17, 333, 55)
    inp2 = streams.rm_inputs(n, 120, seed=seed + 10)

    def run(kind):
        st = np.zeros(layout.RS_WORDS * n, dtype=np.uint32)
        c1, a1 = ol.rm_guard(kind, st, n, inp)
        s1 = st.copy()
        c2, a2 = ol.rm_guard(kind, st, n, inp2, params=p)  # continue from that state, other parameters
        return c1, a1, s1, c2, a2, st

    got = run("port")
    for x, y in zip(got, ol.reference_result(f"rm_guard_{seed}", run, "libref_rm.so")):
        np.testing.assert_array_equal(x, y)
    seen = np.bitwise_or.reduce(got[1].reshape(-1))
    assert seen == 0x10F0F  # every abort bit the block can raise was raised


def record(kind=0, a=0, b=0, c=0, x=0.0, y=0.0, z=0.0, floor=(1,) * 8):
    """One RK_RI_* record; floor = (rForward, lForward, rBack, lBack, right, left, forward, back)."""
    w = np.zeros(12, dtype=np.uint32)
    w[0:4] = kind, a, b, c
    w[4:10] = np.array([x, y, z], dtype=np.float64).view(np.uint32)
    w[10] = sum(int(f) << (8 * k) for k, f in enumerate(floor[:4]))
    w[11] = sum(int(f) << (8 * k) for k, f in enumerate(floor[4:]))
    return w


def run_records(kind, recs, state=None, params=None):
    K = len(recs)
    inp = np.ascontiguousarray(np.stack(recs).reshape(K, 1, 3, 4).transpose(0, 2, 1, 3))
    st = np.zeros(layout.RS_WORDS, dtype=np.uint32) if state is None else state
    cmd, ab = ol.rm_guard(kind, st, 1, inp, params=params)
    return cmd[:, 0], ab[:, 0], st


def _known_answers(kind):
    MOVE_DIR, CONT = _cabi.RK_CMD_MSG_MOVE_DIR, _cabi.RK_CMD_MSG_MOVE_CONT_DIR
    no_fwd = (1, 1, 1, 1, 1, 1, 0, 1)
    wall_fwd = (1, 1, 1, 1, 1, 1, 2, 1)
    # GO_FORWARD over a missing floor -> MOVE_STOP for 1 ms, fllr_abort_vdt_x_p
    cmd, ab, _ = run_records(kind, [record(1, _cabi.RK_DIR_GO_FORWARD, 800, 300, floor=no_fwd)])
    assert list(cmd[0]) == [0, 0, 0, MOVE_DIR | (1 << 8)] and ab[0] == layout.RM_ABORT_FLOOR_XP
    # the same command sideways passes untouched
    cmd, ab, _ = run_records(kind, [record(1, _cabi.RK_DIR_GO_LEFT, 800, 300, floor=no_fwd)])
    assert list(cmd[0]) == [_cabi.RK_DIR_GO_LEFT, 300, 0, MOVE_DIR | (800 << 8)] and ab[0] == 0
    # five sensors without floor: the veto is ignored
    cmd, ab, _ = run_records(kind, [record(1, _cabi.RK_DIR_GO_FORWARD, 800, 300, floor=(0, 0, 0, 0, 1, 1, 0, 1))])
    assert list(cmd[0]) == [_cabi.RK_DIR_GO_FORWARD, 300, 0, MOVE_DIR | (800 << 8)]
    # continuous order heading forward (atan2 = 0) over a missing floor: translation zeroed, rotation kept
    cmd, ab, _ = run_records(kind, [record(2, 700, x=200.0, y=0.0, z=1.5, floor=no_fwd)])
    assert list(cmd[0]) == [0, 0, np.float32(1.5).view(np.uint32), CONT | (700 << 8)] and ab[0] == layout.RM_ABORT_CONT_TRANS
    # heading left (atan2 = pi/2) is outside the forward sector
    cmd, ab, _ = run_records(kind, [record(2, 700, x=0.0, y=200.0, z=1.5, floor=no_fwd)])
    assert cmd[0, 1] == np.float32(200.0).view(np.uint32) and ab[0] == 0
    # cmd_vel: metres per second scaled in double, 500 ms
    cmd, ab, _ = run_records(kind, [record(3, x=0.1, y=-0.2, z=0.3)])
    assert list(cmd[0]) == [np.float32(0.1 * 1000.0).view(np.uint32), np.float32(-0.2 * 1000.0).view(np.uint32),
                            np.float32(0.3).view(np.uint32), CONT | (500 << 8)]
    # Command MOVE_START stops the vehicle; with a wall ahead every later cycle backs off 200 ms at 100 mm/s
    cmd, ab, st = run_records(kind, [record(4, 2), record(0, floor=wall_fwd), record(0)])
    assert list(cmd[0]) == [0, 0, 0, MOVE_DIR | (1 << 8)] and st[layout.RS_CMD_STATUS] == 2
    assert list(cmd[1]) == [_cabi.RK_DIR_GO_BACK, 100, 0, MOVE_DIR | (200 << 8)] and ab[1] == layout.RM_ABORT_WALL_XP
    assert list(cmd[2]) == [0, 0, 0, 0] and ab[2] == layout.RM_ABORT_WALL_XP  # nothing sent; the flag stays until the next command
    # watchdog: the 201st silent cycle sends MOVE_STOP and restarts the count
    cmd, ab, st = run_records(kind, [record(0)] * 403)
    sent = np.nonzero(cmd[:, 3])[0]
    assert list(sent) == [200, 401] and list(cmd[200]) == [0, 0, 0, MOVE_DIR | (1 << 8)] and st[layout.RS_NO_CMD_CNT] == 1
    # SWITCH_FLOOR_SENSOR toggles the ignore flag; QUIT_PG becomes UNKNOWN_CMD
    _, _, st = run_records(kind, [record(4, 10)])
    assert st[layout.RS_IGNORE_FLOOR] == 1 and st[layout.RS_CMD_STATUS] == 10
    _, _, st = run_records(kind, [record(4, 3)], state=st)
    assert st[layout.RS_IGNORE_FLOOR] == 1 and st[layout.RS_CMD_STATUS] == 0xFF
    cmd, ab, _ = run_records(kind, [record(1, _cabi.RK_DIR_GO_FORWARD, 800, 300, floor=no_fwd)], state=st)
    assert list(cmd[0]) == [_cabi.RK_DIR_GO_FORWARD, 300, 0, MOVE_DIR | (800 << 8)]  # floor detection ignored


def test_guard_known_answers_port():
    _known_answers("port")


@needs_ref
def test_guard_known_answers_ref():
    _known_answers("ref")


def test_golden_rmt():
    g = np.load(GOLD)
    n, K = 40, 460
    inp = streams.rm_inputs(n, K, seed=0x5EED)
    st = np.zeros(layout.RS_WORDS * n, dtype=np.uint32)
    cmd, ab = ol.rm_guard("port", st, n, inp)
    np.testing.assert_array_equal(cmd, g["cmd"])
    np.testing.assert_array_equal(ab, g["abort"])
    np.testing.assert_array_equal(st, g["state"])
    y, x = g["atan_y"], g["atan_x"]
    got = np.array([ol.port().orc_atan2f(float(a), float(b)) for a, b in zip(y, x)], dtype=np.float32)
    np.testing.assert_array_equal(got.view(np.uint32), g["atan_out"].view(np.uint32))
