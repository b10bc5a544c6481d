"""CPU: the ADTModePositioning part of the oracle port (orc_adp_batch) pinned against the compiled
reference (AD_mode_positioning.cpp + the joint classes, unmodified), word for word."""
import numpy as np
import pytest

import oracle_lib as ol
from roboken_fmskf_robot_controller_b200 import layout
from test_arm_cpu import random_arm_states



def pos_cmds(n, seed, cid):
    """One ADTModePositioning::PosCmd per arm as two planes [2, n, 4]: dt ~ U{0..1500} ms (1 in 6 is 0),
    angles ~ U[-150, 150] deg in 1/64 deg."""
    rng = np.random.default_rng(seed)
    c = np.zeros((2, n, 4), dtype=np.uint32)
    c[0, :, 0] = cid
    dt = rng.integers(0, 1501, n)
    dt[rng.integers(0, 6, n) == 0] = 0
    c[0, :, 1] = dt
    ang = (rng.integers(-150 * 64, 150 * 64 + 1, (n, 5)).astype(np.float32) / np.float32(64)).view(np.uint32)
    c[0, :, 2:4] = ang[:, 0:2]
    c[1, :, 0:3] = ang[:, 2:5]
    return c


def run_pos_script(kind, n, script, astate, runner=None):
    st = astate.copy()
    ps = np.zeros(layout.PS_WORDS * n, dtype=np.uint32)
    outs = []
    for step in script:
        if step[0] == "init":
            ol.armpos_batch(kind, "init", st, ps, n)
        elif step[0] == "push":
            ol.armpos_batch(kind, "push", st, ps, n, cmd=step[1], valid=step[2])
        elif step[0] == "update":
            tr, _ = ol.armpos_batch(kind, "update", st, ps, n, K=step[1], trace=True)
            outs.append(tr)
        elif step[0] == "status":
            _, s = ol.armpos_batch(kind, "status", st, ps, n, ids=np.asarray(step[1], dtype=np.uint32))
            outs.append(s)
        outs += [st.copy(), ps.copy()]
    return st, ps, outs


def pos_script(n, seed):
    valid = (np.arange(n) % 4 != 2).astype(np.uint8)
    sc = [("init",), ("status", np.full(n, 1)), ("push", pos_cmds(n, seed, 1), None), ("status", np.full(n, 1)), ("update", 3),
          ("status", np.full(n, 1))]
    # six pushes in a row: the FIFO keeps the newest four (the oldest is dropped, not the new one)
    for k in range(2, 8):
        sc.append(("push", pos_cmds(n, seed + k, k), valid if k == 4 else None))
    sc += [("status", np.full(n, j)) for j in range(1, 8)]
    sc += [("update", 400)] + [("status", np.full(n, j)) for j in range(1, 8)] + [("update", 300)]
    sc += [("status", np.full(n, j)) for j in range(1, 8)]
    return sc


def bringup_state(n, seed):
    """Random joint states with the MG joint in its position-control branch, then the arm bring-up."""
    st = random_arm_states(n, seed)
    tab = np.zeros(layout.ACMD_WORDS * n, dtype=np.uint32)
    ol.arm_batch("port", "init", st, tab, n)
    return st


@pytest.mark.parametrize("seed", [1, 2])
def test_positioning_mode_port_equals_ref(seed):
    n = 64
    st0 = bringup_state(n, seed)
    sc = pos_script(n, seed)
    a = ol.reference_result(f"armpos_{seed}", lambda kind: run_pos_script(kind, n, sc, st0), "libref_arm.so")
    b = run_pos_script("port", n, sc, st0)
    assert len(a[2]) == len(b[2])
    for x, y in zip(a[2], b[2]):
        np.testing.assert_array_equal(x, y)


def test_positioning_mode_known_answer():
    """One arm, zero offsets / measured angles: a 100 ms command is ten cycles from the present angle
    (0) to the target; while it runs its id is in neither the queue nor the history -> NO_DATA (0x63),
    afterwards DONE -- the reference's behaviour (AD_mode_positioning.cpp:134-148)."""
    n = 1
    st = np.zeros(layout.AS_WORDS, dtype=np.uint32)
    tab = np.zeros(layout.ACMD_WORDS, dtype=np.uint32)
    ol.arm_batch("port", "init", st, tab, n)
    ps = np.zeros(layout.PS_WORDS, dtype=np.uint32)
    c = np.zeros((2, 1, 4), dtype=np.uint32)
    c[0, 0, 0], c[0, 0, 1] = 7, 100
    c[0, 0, 2:4] = np.float32([10, 20]).view(np.uint32)
    c[1, 0, 0:3] = np.float32([-30, 40, 50]).view(np.uint32)
    ol.armpos_batch("port", "init", st, ps, n)
    ol.armpos_batch("port", "push", st, ps, n, cmd=c)
    assert ol.armpos_batch("port", "status", st, ps, n, ids=np.uint32([7]))[1][0] == 0
    tr, _ = ol.armpos_batch("port", "update", st, ps, n, K=13, trace=True)
    assert ol.armpos_batch("port", "status", st, ps, n, ids=np.uint32([7]))[1][0] == 1
    f = tr.view(np.float32)
    np.testing.assert_array_equal(f[0, 0:5, 0], np.float32([0, 0, 0, 0, 0]))       # tick 0: exec_standby only
    np.testing.assert_array_equal(f[1, 0:5, 0], np.float32([0, 0, 0, 0, 0]))       # tick 1: remaining = 10 cycles
    np.testing.assert_allclose(f[6, 0:5, 0], np.float32([5, 10, -15, 20, 25]), rtol=1e-6)
    np.testing.assert_array_equal(f[11, 0:5, 0], np.float32([10, 20, -30, 40, 50]))
    assert list(tr[:, 11, 0]) == [1] * 11 + [0, 0]
