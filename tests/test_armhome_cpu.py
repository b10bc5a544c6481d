"""CPU: pin the homing modes of the plain-C oracle (orc_adh_batch: ADTModeInitialize, ADTModeInitPosMove) against the
compiled reference modes (src/ArmDrive/AD_mode_initialize.cpp, AD_mode_initpos_move.cpp, unmodified, on the unmodified
joint classes) -- SURVEY 8f-4."""
import os

import numpy as np
import pytest

import oracle_lib as ol
from roboken_fmskf_robot_controller_b200 import _cabi, layout

GOLD = os.path.join(os.path.dirname(__file__), "golden", "armhome_golden.npz")
PREV_JOINTS = (layout.AJ_P1, layout.AJ_DFL, layout.AJ_DFR, layout.AJ_P3)


def start_states(n, seed, zero=False):
    """Arms as a running robot could leave them: random offsets / targets / measured angles, random joint flags (the
    torque_on_prev bit only on the joints that have one), the ICS servo anywhere in its range."""
    rng = np.random.default_rng(seed)
    a = np.zeros((n, layout.AS_WORDS), dtype=np.uint32)
    a[:, layout.AS_ICS_POS] = 0xFFFFFFFF
    if not zero:
        for k in range(7):
            for f, lo, hi in ((layout.AJ_RAW_NOW, -100, 100), (layout.AJ_OFS, -20, 20), (layout.AJ_RAW_TGT, -100, 100), (layout.AJ_CURLIM, 0, 2)):
                a[:, layout.AS_JOINT0 + 4 * k + f] = rng.uniform(lo, hi, n).astype(np.float32).view(np.uint32)
        a[:, layout.AS_ICS_SERVO] = rng.integers(-3000, 3000, n).astype(np.int32).view(np.uint32)
        fl = np.zeros(n, dtype=np.uint32)
        for k in range(7):
            bits = rng.integers(0, 8, n).astype(np.uint32)
            if k in PREV_JOINTS:
                bits |= rng.integers(0, 2, n).astype(np.uint32) << 3
            fl |= bits << (4 * k)
        a[:, layout.AS_JFLAGS] = fl
        a[:, layout.AS_MG_PRE_TGT] = rng.uniform(-100, 100, n).astype(np.float32).view(np.uint32)
    return layout.aos_to_soa(a)


def feedback(n, K, seed):
    """Servo angles drifting as a random walk (degrees): float32 [K, 4, n] for P1, DF_Left, DF_Right, P3."""
    rng = np.random.default_rng(seed)
    return np.ascontiguousarray((rng.standard_normal((K, 4, n)).cumsum(axis=0) * 0.5 + rng.uniform(-100, 100, (1, 4, n))).astype(np.float32))


def run(kind, mode, s0, n, K, now, chunks=None):
    st, hs = s0.copy(), np.zeros(layout.HS_WORDS * n, dtype=np.uint32)
    ol.arm_homing(kind, "init", st, hs, n, mode=mode)
    if chunks is None:
        tr = ol.arm_homing(kind, "update", st, hs, n, K=K, now=now, trace=True)
    else:
        parts, k0 = [], 0
        for k1 in chunks:
            parts.append(ol.arm_homing(kind, "update", st, hs, n, K=k1 - k0, now=None if now is None else np.ascontiguousarray(now[k0:k1]), trace=True))
            k0 = k1
        tr = np.concatenate(parts)
    return st, hs, tr


@pytest.mark.parametrize("mode", [_cabi.RK_ADH_MODE_INIT, _cabi.RK_ADH_MODE_INIT_POS_MOVE])
@pytest.mark.parametrize("fb", [False, True])
def test_homing_port_equals_ref(mode, fb):
    n, K = 48, 1500
    s0 = start_states(n, seed=10 * mode + fb)
    now = feedback(n, K, seed=3) if fb else None
    a, b = run("port", mode, s0, n, K, now), ol.reference_result(f"armhome_{mode}_{int(fb)}", lambda kind: run(kind, mode, s0, n, K, now), "libref_arm.so")
    for x, y, nm in zip(a, b, ("state", "mode block", "trace")):
        np.testing.assert_array_equal(x, y, err_msg=nm)
    final = layout.soa_to_aos(a[1], n, layout.HS_WORDS)[:, layout.HS_STATE]
    done = 5 if mode == _cabi.RK_ADH_MODE_INIT else 3
    assert ((final & 0xFF) == done).all() and (final & layout.AS_FSM_IS_COMP).all()  # every arm reached COMPLETED


def test_homing_from_power_on_known_sequence():
    """All-zero arm through INIT: 1 + 101 + 501 + 1 cycles of the fixed phases, then the ramp to the init pose
    (slowest axis J2: 0 -> -90 deg at 30 deg/s = 300 cycles; J1 sits at its mechanical end, 150 deg, after the reset and
    needs 17), COMPLETED afterwards; MG in torque control until MOVE_INIT_POS."""
    n, K = 2, 1200
    s0 = start_states(n, 0, zero=True)
    for st, hs, tr in (run("port", _cabi.RK_ADH_MODE_INIT, s0, n, K, None),
                       ol.reference_result("armhome_power_on", lambda kind: run(kind, _cabi.RK_ADH_MODE_INIT, s0, n, K, None), "libref_arm.so")):
        states = tr[:, 11, 0]
        first = {s: int(np.argmax(states == s)) for s in (1, 2, 3, 4, 5)}
        assert first[1] == 0 and first[2] == 101 and first[3] == 101 + 501 and first[4] == 101 + 501 + 1
        assert first[5] == first[4] + 300
        a = layout.soa_to_aos(st, n, layout.AS_WORDS)[0]
        f = lambda k, w: a[layout.AS_JOINT0 + 4 * k + w : layout.AS_JOINT0 + 4 * k + w + 1].view(np.float32)[0]
        assert f(layout.AJ_P1, layout.AJ_OFS) == -150.0  # raw_now 0 - mechend 150
        assert abs((f(layout.AJ_P1, layout.AJ_RAW_TGT) - f(layout.AJ_P1, layout.AJ_OFS)) - 145.0) < 1e-4
        assert f(layout.AJ_P1, layout.AJ_CURLIM) == np.float32(0.7) and f(layout.AJ_DFL, layout.AJ_CURLIM) == 1.0
        assert (a[layout.AS_MG_TX] & 0xFF) == 0xA4  # position control at the end


def test_homing_port_chunked_equals_one_pass():
    n, K = 32, 1300
    for mode in (_cabi.RK_ADH_MODE_INIT, _cabi.RK_ADH_MODE_INIT_POS_MOVE):
        s0 = start_states(n, seed=77 + mode)
        now = feedback(n, K, seed=5)
        a = run("port", mode, s0, n, K, now)
        b = run("port", mode, s0, n, K, now, chunks=(1, 2, 103, 104, 610, 1300))
        for x, y in zip(a, b):
            np.testing.assert_array_equal(x, y)


def test_golden_armhome():
    g = np.load(GOLD)
    n, K = 24, 1300
    for mode, tag in ((_cabi.RK_ADH_MODE_INIT, "init"), (_cabi.RK_ADH_MODE_INIT_POS_MOVE, "ipm")):
        st, hs, tr = run("port", mode, start_states(n, seed=0x5EED + mode), n, K, feedback(n, K, seed=0x5EED))
        np.testing.assert_array_equal(st, g[tag + "_state"])
        np.testing.assert_array_equal(hs, g[tag + "_hstate"])
        np.testing.assert_array_equal(tr[::13], g[tag + "_trace"])
