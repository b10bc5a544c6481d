"""CPU tests that PIN the arm part of the plain-C oracle (oracle/robotick_oracle.c, orc_adt_batch)
against oracle/_ref/libref_arm.so -- the reference's own ArmDrive sources compiled unmodified
(ADTModePositioningSeq + JointIcsServo / JointMgServo / JointMyBldcServo / JointDfGear*) --
state word for state word and trace word for trace word, and against tests/golden/arm_golden.npz
(the reference's own POS_CMD_SEQ_DEBUG_0/1/2 run through the compiled reference)."""
import os

import numpy as np
import pytest

import oracle_lib as ol
from roboken_fmskf_robot_controller_b200 import _cabi, layout, streams

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def fresh(n):
    return np.zeros(layout.AS_WORDS * n, dtype=np.uint32), np.zeros(layout.ACMD_WORDS * n, dtype=np.uint32)


def run_script(kind, n, script, state=None, tab=None):
    """script: list of ("init",) | ("push", img_aos[n,260], valid|None) | ("update", K) | ("status", ids)."""
    st, tb = fresh(n)
    if state is not None:
        st[:] = state
    if tab is not None:
        tb[:] = tab
    outs = []
    for step in script:
        if step[0] == "init":
            ol.arm_batch(kind, "init", st, tb, n)
        elif step[0] == "push":
            ol.arm_batch(kind, "push", st, tb, n, seq=layout.aos_to_soa(step[1]), valid=step[2])
        elif step[0] == "update":
            tr, _ = ol.arm_batch(kind, "update", st, tb, n, K=step[1], trace=True)
            outs.append(tr)
        elif step[0] == "status":
            _, s = ol.arm_batch(kind, "status", st, tb, n, ids=np.asarray(step[1], dtype=np.uint32))
            outs.append(s)
        outs.append(st.copy())
    return st, tb, outs


def assert_same(a, b):
    assert len(a[2]) == len(b[2])
    for x, y in zip(a[2], b[2]):
        np.testing.assert_array_equal(x, y)
    np.testing.assert_array_equal(a[0], b[0])
    np.testing.assert_array_equal(a[1], b[1])


def random_arm_states(n, seed, mg_any_branch=False):
    """Random but valid arm states: offsets, targets, flags, ring indices, mid-move FSM.  The MG joint
    is kept in its position-control branch (torque on + initialised) unless mg_any_branch, which also
    randomises its PI_D state so that every branch of JointMgServo::update runs."""
    rng = np.random.default_rng(seed)
    a = np.zeros((n, layout.AS_WORDS), dtype=np.uint32)
    f = lambda lo, hi, shape: (rng.integers(int(lo * 64), int(hi * 64) + 1, shape).astype(np.float32) / np.float32(64)).view(np.uint32)
    for k in range(7):
        a[:, layout.AS_JOINT0 + 4 * k + layout.AJ_OFS] = f(-30, 30, n)
        a[:, layout.AS_JOINT0 + 4 * k + layout.AJ_RAW_TGT] = f(-150, 150, n)
        a[:, layout.AS_JOINT0 + 4 * k + layout.AJ_CURLIM] = f(0, 3, n)
        a[:, layout.AS_JOINT0 + 4 * k + layout.AJ_RAW_NOW] = f(-150, 150, n)
    a[:, layout.AS_DFV_P] = f(-300, 300, n)
    a[:, layout.AS_DFV_R] = f(-300, 300, n)
    fl = rng.integers(0, 16, (n, 7)).astype(np.uint32)
    if not mg_any_branch:
        fl[:, layout.AJ_P1] = (fl[:, layout.AJ_P1] & 8) | 7
    else:
        a[:, layout.AS_MG_CTRL : layout.AS_MG_CTRL + 7] = f(-2, 2, (n, 7))
        a[:, layout.AS_MG_CTRL + 7] = rng.integers(0, 2, n)
    fl[:, [layout.AJ_Y0, layout.AJ_P2, layout.AJ_R0]] &= 7
    a[:, layout.AS_JFLAGS] = sum(fl[:, k] << np.uint32(4 * k) for k in range(7))
    a[:, layout.AS_MG_PRE_TGT] = f(-150, 150, n)
    a[:, layout.AS_ICS_SERVO] = rng.integers(-4000, 4001, n).astype(np.int32).view(np.uint32)
    a[:, layout.AS_ICS_POS] = np.uint32(0xFFFFFFFF)
    ex, hd = rng.integers(0, 4, n), rng.integers(0, 4, n)
    a[:, layout.AS_SEQ_IDX] = (ex | (hd << 16)).astype(np.uint32)
    st = rng.integers(0, 3, n)
    a[:, layout.AS_FSM] = (st | (rng.integers(0, 2, n) << 8) | (rng.integers(0, 2, n) << 9)).astype(np.uint32)
    a[:, layout.AS_CMD_IDX] = rng.integers(0, 34, n)
    cnt = rng.integers(1, 50, n)
    a[:, layout.AS_MOVE_CNT] = cnt
    a[:, layout.AS_CYCLE] = rng.integers(0, 52, n)
    a[:, layout.AS_TOTAL_MS] = rng.integers(0, 3000, n)
    a[:, layout.AS_NOW_DT] = rng.integers(0, 3000, n)
    a[:, layout.AS_NOW_TGT : layout.AS_NOW_TGT + 5] = f(-150, 150, (n, 5))
    a[:, layout.AS_MOVE_DEG : layout.AS_MOVE_DEG + 5] = f(-3, 3, (n, 5))
    return layout.aos_to_soa(a)


def test_debug_sequences_port_equals_ref():
    """POS_CMD_SEQ_DEBUG_0/1/2 (AD_mode_positioning_seq_debug_data.cpp:5-64): bring-up, push all
    three, run 600 ticks (the three sequences take 110 + 100 + 300 cycles + transitions)."""
    imgs = [img.copy() for img in np.load(os.path.join(GOLD, "arm_golden.npz"))["seq_a"][:3]]  # DEBUG_0/1/2 as the reference defines them
    if ol.have_ref("libref_arm.so"):
        r = ol.ref("libref_arm.so")
        for w in range(3):
            q = _cabi.AdtPosCmdSeq()
            assert r.ref_adt_debug_seq(w, q) == (1 if w == 2 else 0)  # get_poscmdseq_debug() returns DEBUG_2
            img = ol.seq_struct_to_image(q)
            img[0] = 1
            np.testing.assert_array_equal(img, imgs[w])
    for w in range(3):
        imgs[w][0] = 10 + w
    script = [("init",)] + [("push", im[None, :], None) for im in imgs] + [("status", [10]), ("update", 150), ("status", [10]),
                                                                             ("status", [11]), ("update", 450), ("status", [12])]
    a, b = ol.reference_result("arm_debug_sequences", lambda kind: run_script(kind, 1, script), "libref_arm.so"), run_script("port", 1, script)
    assert_same(a, b)
    tr = a[2][-4]  # the 450-tick trace
    assert tr[-1, 11, 0] == layout.ASTATE_STANDBY
    # the arm ends on the last waypoint of DEBUG_2
    np.testing.assert_array_equal(tr[-1, 0:5, 0].view(np.float32), np.float32([0, 120, -60, 0, 45]))


@pytest.mark.parametrize("seed", [1, 2])
def test_random_sequences_port_equals_ref(seed):
    n = 96
    s1 = streams.arm_sequences(n, seed=seed, seq_id=1, max_len=8)
    s2 = streams.arm_sequences(n, seed=seed + 50, seq_id=2, max_len=6)
    valid = (np.arange(n) % 3 != 0).astype(np.uint8)
    script = [("init",), ("push", s1, None), ("update", 37), ("push", s2, valid), ("status", np.full(n, 1)),
              ("update", 500), ("status", np.full(n, 2)), ("status", np.full(n, 7))]
    assert_same(ol.reference_result(f"arm_random_sequences_{seed}", lambda kind: run_script(kind, n, script), "libref_arm.so"), run_script("port", n, script))


def test_ring_overflow_and_id0_port_equals_ref():
    """Five pushes into the 4-slot ring (the 4th/5th are dropped while the first is executing),
    id 0 before the first move (isModeFirstCall), status for ids in every ring position."""
    n = 8
    seqs = [streams.arm_sequences(n, seed=10 + k, seq_id=k, max_len=3) for k in range(6)]
    script = [("init",), ("status", np.zeros(n)), ("push", seqs[0], None), ("status", np.zeros(n)), ("update", 1),
              ("status", np.zeros(n))]
    for k in range(1, 6):
        script += [("push", seqs[k], None)] + [("status", np.full(n, j)) for j in range(6)]
    script += [("update", 900)] + [("status", np.full(n, j)) for j in range(6)]
    script += [("push", seqs[5], None), ("update", 5)] + [("status", np.full(n, j)) for j in range(6)]
    assert_same(ol.reference_result("arm_ring_overflow", lambda kind: run_script(kind, n, script), "libref_arm.so"), run_script("port", n, script))


def test_random_states_port_equals_ref():
    n = 400
    st0 = random_arm_states(n, seed=4)
    tab = np.zeros(layout.ACMD_WORDS * n, dtype=np.uint32)
    taos = np.zeros((n, layout.ACMD_WORDS), dtype=np.uint32)
    for s in range(4):
        taos[:, s * 260 : (s + 1) * 260] = streams.arm_sequences(n, seed=20 + s, seq_id=s + 1, max_len=5)
    tab[:] = layout.aos_to_soa(taos)
    script = [("update", 3), ("status", np.full(n, 2)), ("update", 120)]
    assert_same(ol.reference_result("arm_random_states", lambda kind: run_script(kind, n, script, st0, tab), "libref_arm.so"),
                run_script("port", n, script, st0, tab))


def test_mg_torque_control_branches_port_equals_ref():
    """JointMgServo::update, all four branches (AD_joint_mg_servo.cpp:50-73): torque on->off edge
    (PI_D reset), not initialised + torque on (torque control), position control, torque off
    (InitGain + torque control incl. the gravity feed-forward through the CMSIS sine and the
    double-precision current -> raw map)."""
    n = 512
    st0 = random_arm_states(n, seed=6, mg_any_branch=True)
    taos = np.zeros((n, layout.ACMD_WORDS), dtype=np.uint32)
    for s in range(4):
        taos[:, s * 260 : (s + 1) * 260] = streams.arm_sequences(n, seed=30 + s, seq_id=s + 1, max_len=4)
    tab = layout.aos_to_soa(taos)
    script = [("update", 1), ("update", 2), ("update", 60)]
    a, b = ol.reference_result("arm_mg_branches", lambda kind: run_script(kind, n, script, st0, tab), "libref_arm.so"), run_script("port", n, script, st0, tab)
    assert_same(a, b)
    fl = (layout.soa_to_aos(st0, n, layout.AS_WORDS)[:, layout.AS_JFLAGS] >> 4) & 0xF
    assert len(np.unique(fl)) == 16  # every flag combination of the MG joint occurred
    tr = a[2][0]
    assert set(np.unique(tr[0, 5, :] * 0 + (layout.soa_to_aos(a[2][1], n, layout.AS_WORDS)[:, layout.AS_MG_TX] & 0xFF))) >= {0xA1, 0xA4}


def test_extreme_waypoints_port_equals_ref():
    """dt going backwards (u32 wrap -> huge count), dt == previous (count clamps to 1), angles past
    the ICS range (+-180 deg: degPos100 rejects; > +-135 deg: setPos rejects) and a len-0 sequence."""
    wp = [(0, (170, 10, 10, 10, 10)), (50, (-190, 20, -20, 5, 5)), (50, (140, 0, 0, 0, 0)), (40, (0, 0, 0, 0, 0)),
          (45, (100, -100, 100, -100, 100))]
    img = np.stack([streams.arm_seq_image(3, wp), streams.arm_seq_image(4, []), streams.arm_seq_image(5, wp[:2])])
    script = [("init",), ("push", img, None), ("update", 40), ("status", [3, 4, 5]), ("update", 40)]
    assert_same(ol.reference_result("arm_extreme_waypoints", lambda kind: run_script(kind, 3, script), "libref_arm.so"), run_script("port", 3, script))


def test_port_matches_golden():
    g = np.load(os.path.join(GOLD, "arm_golden.npz"))
    n = int(g["n"])
    script = [("init",), ("push", g["seq_a"], None), ("push", g["seq_b"], g["valid_b"]), ("update", int(g["K"]))]
    st, tb, outs = run_script("port", n, script)
    np.testing.assert_array_equal(outs[-2], g["trace"])
    np.testing.assert_array_equal(st, g["state"])
    np.testing.assert_array_equal(tb, g["cmdtab"])
    _, s = ol.arm_batch("port", "status", st, tb, n, ids=g["ids"])
    np.testing.assert_array_equal(s, g["status"])


def test_default_params_and_struct_sizes():
    import ctypes as C

    assert C.sizeof(_cabi.AdtPosCmdSeq) == 776 and C.sizeof(_cabi.AdtPosCmd) == 24  # SURVEY 8a: a11
    p = _cabi.default_arm_params()
    assert np.float32(p.gear_ratio[4]) == np.float32(24.0) / np.float32(7.0)
