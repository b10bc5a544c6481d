"""SURVEY 8f-3, arm side: the servo feedback decoders -- the port against the reference's own rx callbacks
(JointMyBldcServo::rx_callback AD_joint_mybldc_servo.cpp:45-70, JointMgServo::rx_callback AD_joint_mg_servo.cpp:75-92)
compiled for x86, bit for bit, plus known answers that hold without the compiled reference."""
import numpy as np
import pytest

import oracle_lib as ol
from roboken_fmskf_robot_controller_b200 import layout



def rx_cases(n, seed, mg_upper_zero=True):
    """Random joint blocks (torque on / off per joint) and random frames for all four receivers."""
    rng = np.random.default_rng(seed)
    aos = np.zeros((n, layout.AS_WORDS), dtype=np.uint32)
    aos[:, layout.AS_JOINT0:layout.AS_JOINT0 + 28] = rng.uniform(-200, 200, (n, 28)).astype(np.float32).view(np.uint32)
    # joint flags as the reference can hold them: connected | torque_on | initialized for all seven, torque_on_prev only
    # for the four CAN servos (P1, DF_Left, DF_Right, P3); no ICS position word sent yet
    aos[:, layout.AS_JFLAGS] = rng.integers(0, 1 << 28, n, dtype=np.uint32) & np.uint32(0xF77FFF7)
    aos[:, layout.AS_JFLAGS + 2] = 0xFFFFFFFF
    frames = []
    for which in range(3):
        f = rng.integers(0, 256, (n, 8), dtype=np.uint8)
        f[: n // 8, 2:4] = np.array([[0x00, 0x80], [0xFF, 0x7F], [0, 0], [0xFF, 0xFF]], dtype=np.uint8)[rng.integers(0, 4, n // 8)]
        f[: n // 8, 4] = np.array([0x80, 0x7F, 0, 0xFF], dtype=np.uint8)[rng.integers(0, 4, n // 8)]
        frames.append(np.ascontiguousarray(f).view(np.uint64).reshape(n))
    f = rng.integers(0, 256, (n, 8), dtype=np.uint8)
    f[:, 0] = np.array([0x92, 0x9C, 0xA1, 0x92, 0x9C, 0x31, 0xA4], dtype=np.uint8)[rng.integers(0, 7, n)]
    if mg_upper_zero:
        f[f[:, 0] == 0x92, 5:8] = 0  # where the x86 build and the Cortex-M7 agree on the undefined shift (see the port)
    f[: n // 8, 2:4] = np.array([[0x00, 0x80], [0xFF, 0x7F], [0, 0], [0xFF, 0xFF]], dtype=np.uint8)[rng.integers(0, 4, n // 8)]
    frames.append(np.ascontiguousarray(f).view(np.uint64).reshape(n))
    cmdid = np.where(rng.integers(0, 4, n) == 0, rng.integers(0, 0x10000, n), 0x1000).astype(np.uint32)
    return layout.aos_to_soa(aos), frames, cmdid


def run(kind, state, n, frames, cmdid):
    st = state.copy()
    curs = []
    for which in range(4):
        cur = np.full(n, 123.25, dtype=np.float32)
        ol.arm_rx(kind, which, st, n, frames[which], cmdid if which < 3 else None, cur)
        curs.append(cur)
    return st, curs


@pytest.mark.parametrize("seed", [1, 2, 3])
def test_port_equals_reference_rx(seed):
    n = 4000
    state, frames, cmdid = rx_cases(n, seed)
    pst, pcur = run("port", state, n, frames, cmdid)
    rst, rcur = ol.reference_result(f"armrx_{seed}", lambda kind: run(kind, state, n, frames, cmdid), "libref_arm.so")
    np.testing.assert_array_equal(pst, rst)
    for a, b in zip(pcur, rcur):
        np.testing.assert_array_equal(a.view(np.uint32), b.view(np.uint32))
    assert not np.array_equal(pst, state)


def test_rx_known_answers():
    """Firmware constants (AD_task_main.cpp:38-107): P3 gear 48/19 dir -1; DF_Left gear 1 dir +1."""
    n = 4
    aos = np.zeros((n, layout.AS_WORDS), dtype=np.uint32)
    aos[:, layout.AS_JFLAGS] = [0x2222222, 0, 0x2222222, 0]  # torque on everywhere / off everywhere
    state = layout.aos_to_soa(aos)

    def frame(b):
        return np.frombuffer(bytes(b), dtype=np.uint64)[0]

    # MyBldc summary: angle 0x0190 = 400 -> 25 deg at the output; current 0x10 -> 1 A (Q4)
    fr = np.array([frame([0x10, 0, 0x90, 0x01, 0x10, 0, 0, 0])] * n, dtype=np.uint64)
    cur = np.zeros(n, dtype=np.float32)
    st = state.copy()
    ol.arm_rx("port", 0, st, n, fr, None, cur)  # DF_Left
    a = layout.soa_to_aos(st, n, layout.AS_WORDS)
    j = layout.AS_JOINT0 + 4 * 2
    assert a[0, j + 3].view(np.float32) == np.float32(25.0) and cur[0] == np.float32(1.0)
    assert a[0, j + 1] == 0 and a[1, j + 1].view(np.float32) == np.float32(25.0)  # the target follows only while torque is off
    st = state.copy()
    ol.arm_rx("port", 2, st, n, fr, np.array([0x1000, 0x1000, 0x1001, 0x1001], dtype=np.uint32), cur)  # P3, ids 2-3 ignored
    a = layout.soa_to_aos(st, n, layout.AS_WORDS)
    j = layout.AS_JOINT0 + 4 * 6
    want = np.float32(np.float32(np.float32(400.0) / np.float32(16.0)) / np.float32(np.float32(48.0) / np.float32(19.0))) * np.float32(-1.0)
    assert a[0, j + 3].view(np.float32) == want and cur[0] == np.float32(-1.0) and a[2, j + 3] == 0
    # MG: 0x92 with angle 12345 * 0.01 deg at the motor = -12345 / 1000 deg at the output (1:10, direction -1)
    ang = 12345
    fr = np.array([frame([0x92] + list(int(ang).to_bytes(7, "little", signed=True)))] * n, dtype=np.uint64)
    st = state.copy()
    ol.arm_rx("port", 3, st, n, fr, None, cur)
    a = layout.soa_to_aos(st, n, layout.AS_WORDS)
    j = layout.AS_JOINT0 + 4 * 1
    db = np.float64(np.float32(np.float32(np.float32(-1.0) / np.float32(100.0)) / np.float32(10.0)) / np.float32(256.0))
    assert a[0, j + 3].view(np.float32) == np.float32(np.float64(ang * 256) * db) and abs(float(a[0, j + 3].view(np.float32)) + 12.345) < 1e-5
    # MG: 0x9C with iq = +-1000 -> -+(C_A * 1e6 + C_B * 1e3) A
    for iq in (1000, -1000):
        fr = np.array([frame([0x9C, 30] + list(int(iq).to_bytes(2, "little", signed=True)) + [0, 0, 0, 0])] * n, dtype=np.uint64)
        cur[:] = 0
        st2 = state.copy()
        ol.arm_rx("port", 3, st2, n, fr, None, cur)
        mag = 0.0000057204 * 1000.0 * 1000.0 + (-0.0000485371) * 1000.0
        assert cur[0] == np.float32(-1.0) * np.float32(mag if iq > 0 else -mag)
        np.testing.assert_array_equal(st2, state)  # a current frame leaves the joint block alone
