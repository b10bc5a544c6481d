"""CPU: the WT901C Yaw-register form of the rollout's yaw input (rk_vdt_rollout_t::d_yaw_reg) is pinned three ways: the
port and the compiled vehicle reference agree on it, both agree with the float stream computed on the host, and that
float stream IS what the compiled IMU reference (IMU_IF_WT901C::updateData -> getYawDate) reports for the register."""
import numpy as np

import oracle_lib as ol
import workloads as wl
from roboken_fmskf_robot_controller_b200 import _cabi, layout, streams



def rollout(kind, n, steps, inp, yaw):
    st = np.zeros(layout.VS_WORDS * n, dtype=np.uint32)
    ro = ol.HostRollout(n, steps, _cabi.RK_SENSOR_PLANT, inp["cmd"], inp["seg_len"], yaw, 10, trace=True)
    (ol.run_port if kind == "port" else ol.run_ref)(st, n, ro)
    return st, ro.trace


def test_yaw_register_stream_three_ways():
    n, steps = 48, 700
    inp = wl.plant_inputs(n, steps, seed=3)
    reg = streams.vehicle_yaw_reg(n, steps // 10, seed=3)
    assert reg.dtype == np.int16 and reg.min() < -30000 and reg.max() > 30000  # wraps through +-180 degrees
    # the IMU reference's own yaw for these register values
    regs = np.zeros((steps // 10 + 1, 16, n), dtype=np.int16)
    regs[0, 12] = 32767
    regs[1:, 11] = reg
    regs[1:, 12] = 32767
    out = ol.reference_result("yaw_reg_imu", lambda kind: (ol.imu_port if kind == "port" else ol.imu_ref)(
        np.zeros(layout.IS_WORDS * n, dtype=np.uint32), n, regs, None, want_out=True, do_init=True), "libref_imu.so")
    yaw_deg = out.view(np.float32)[1:, 2, :, 3]  # Data word 11 = angle[2] = getYawDate()
    rad = (yaw_deg * streams.DEG2RAD).astype(np.float32)  # the ISR's mymath::deg2rad
    np.testing.assert_array_equal(rad.view(np.uint32), streams.yaw_reg_to_rad(reg).view(np.uint32))
    base = ol.reference_result("yaw_reg_float", lambda kind: rollout(kind, n, steps, inp, np.ascontiguousarray(rad)), "libref_vdt.so")
    for got in (rollout("port", n, steps, inp, reg),
                ol.reference_result("yaw_reg_register", lambda kind: rollout(kind, n, steps, inp, reg), "libref_vdt.so")):
        np.testing.assert_array_equal(got[1], base[1])
        np.testing.assert_array_equal(got[0], base[0])


def test_yaw_register_port_matches_float_stream():
    n, steps = 32, 300
    inp = wl.plant_inputs(n, steps, seed=5)
    reg = streams.vehicle_yaw_reg(n, steps // 10, seed=5)
    a, b = rollout("port", n, steps, inp, reg), rollout("port", n, steps, inp, streams.yaw_reg_to_rad(reg))
    np.testing.assert_array_equal(a[1], b[1])
    np.testing.assert_array_equal(a[0], b[0])
