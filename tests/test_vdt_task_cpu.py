"""CPU: the VDT::main command layer of the oracle port (messages, speed limiters, move-time auto-stop)
pinned against the reference's WHOLE vehicle task -- VD_task_main.cpp compiled unmodified with its 100 Hz
loop, its ISR and its CAN tx routine (oracle/ref_harness_vdt_task.cpp) -- trace word for trace word."""
import numpy as np
import pytest

import oracle_lib as ol
from roboken_fmskf_robot_controller_b200 import _cabi, layout, streams



def task_inputs(n, steps, seed, seg_len=50, yaw_period=10):
    n_seg, n_yaw = (steps + seg_len - 1) // seg_len, (steps + yaw_period - 1) // yaw_period
    yaw_deg = streams.vehicle_yaw(n, n_yaw, seed, degrees=True)
    return dict(n=n, steps=steps, cmd=streams.vehicle_messages(n, n_seg, seed), seg_len=seg_len,
                yaw=(yaw_deg * streams.DEG2RAD).astype(np.float32), yaw_deg=yaw_deg, yaw_period=yaw_period)


def run(kind, inp, trace=True):
    n = inp["n"]
    st = np.zeros(layout.VS_WORDS * n, dtype=np.uint32)
    ro = ol.HostRollout(n, inp["steps"], _cabi.RK_SENSOR_PLANT, inp["cmd"], inp["seg_len"], inp["yaw"], inp["yaw_period"],
                        trace=trace, task_period=10)
    if kind == "port":
        ol.run_port(st, n, ro)
    else:
        ol.run_task_ref(st, n, ro, inp["yaw_deg"])
    return st, ro.trace


@pytest.mark.parametrize("seed,seg_len", [(1, 50), (2, 30), (3, 200)])
def test_port_equals_reference_task(seed, seg_len):
    inp = task_inputs(40, 1200, seed, seg_len=seg_len)
    s_ref, t_ref = ol.reference_result(f"vdt_task_{seed}", lambda kind: run(kind, inp), "libref_vdt_task.so")
    s_port, t_port = run("port", inp)
    np.testing.assert_array_equal(t_port, t_ref)
    np.testing.assert_array_equal(s_port, s_ref)


def test_every_direction_and_limiter():
    """All REQ_MOVE_DIR codes (0..10 + two undefined) x speeds {default, in range, over the limit}, time 300 ms:
    after the countdown fires every vehicle is commanded to stop."""
    codes = list(range(13))
    speeds = [0, 150, 400, 401, 65, 70000]
    n = len(codes) * len(speeds)
    cmd = np.zeros((1, n), dtype=streams.vehicle_messages(1, 1).dtype)
    k = 0
    for c in codes:
        for s in speeds:
            cmd["vx"][0, k] = np.uint32(c).view(np.float32)
            cmd["vy"][0, k] = np.uint32(s).view(np.float32)
            cmd["kind"][0, k] = _cabi.RK_CMD_MSG_MOVE_DIR | (300 << 8)
            k += 1
    yaw_deg = np.zeros((1, n), dtype=np.float32)
    inp = dict(n=n, steps=700, cmd=cmd, seg_len=1000, yaw=yaw_deg.copy(), yaw_deg=yaw_deg, yaw_period=1000)
    s_ref, t_ref = ol.reference_result("vdt_task_directions", lambda kind: run(kind, inp), "libref_vdt_task.so")
    s_port, t_port = run("port", inp)
    np.testing.assert_array_equal(t_port, t_ref)
    np.testing.assert_array_equal(s_port, s_ref)
    cnt = t_ref[:, 13, :]
    assert cnt[0, 0] == 300 * 100 // 1000 + 1 - 1 and (cnt[-1] == 0).all()  # decremented once in the iteration that set it
    tgt = t_ref.view(np.float32)[:, 6:9, :]
    fwd = 1 * len(speeds)  # GO_FORWARD, default speed: target reaches 200 mm/s, then the auto-stop brings it back to 0
    assert 150.0 < tgt[:, 0, fwd].max() <= np.float32(200.0) and tgt[-1, 0, fwd] == 0.0
    over = 1 * len(speeds) + 5  # speed 70000 -> limited to 400
    assert tgt[:, 0, over].max() <= np.float32(400.0)


def test_port_known_answers_without_reference():
    """REQ_MOVE_CONT_DIR limiter: (300, 400) has length 500 -> scaled to (240, 320); vth 25 -> 6*pi."""
    cmd = np.zeros((1, 1), dtype=streams.vehicle_messages(1, 1).dtype)
    cmd["vx"], cmd["vy"], cmd["vth"] = 300.0, 400.0, 25.0
    cmd["kind"] = _cabi.RK_CMD_MSG_MOVE_CONT_DIR | (100000 << 8)
    z = np.zeros((1, 1), dtype=np.float32)
    st, tr = run("port", dict(n=1, steps=3000, cmd=cmd, seg_len=5000, yaw=z, yaw_deg=z, yaw_period=5000))
    tgt = tr.view(np.float32)[-1, 6:9, 0]
    assert tgt[0] == np.float32(240.0) and tgt[1] == np.float32(320.0)
    assert tgt[2] == np.float32(6.0 * np.pi)
