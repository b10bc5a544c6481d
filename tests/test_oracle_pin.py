"""CPU tests that PIN the plain-C oracle (oracle/robotick_oracle.c):
  * against oracle/_ref -- the reference's own sources compiled unmodified -- bit for bit;
  * against the probe values recorded in SURVEY.md Appendix D;
  * against the committed golden fixtures (tests/golden/*.npz, generated from oracle/_ref).
"""
import ctypes as C
import os

import numpy as np
import pytest

import oracle_lib as ol
import workloads as wl
from roboken_fmskf_robot_controller_b200 import _cabi, layout

GOLD = os.path.join(os.path.dirname(__file__), "golden")
needs_ref = pytest.mark.skipif(not ol.have_ref(), reason="oracle/_ref not built and no /root/reference")


def _run(kind, inp, sensor=_cabi.RK_SENSOR_PLANT, state=None, trace=True, lib="libref_vdt.so", frames=None):
    n = inp["n"]
    st = np.zeros(layout.VS_WORDS * n, dtype=np.uint32) if state is None else state.copy()
    ro = ol.HostRollout(n, inp["steps"], sensor, inp.get("cmd"), inp.get("seg_len", 0), inp.get("yaw"),
                        inp.get("yaw_period", 0), frames=frames, trace=trace)
    if kind == "port":
        ol.run_port(st, n, ro)
    else:
        ol.run_ref(st, n, ro, name=lib)
    return st, ro.trace


def _check_appendix_d(trace, pos_libm):
    f = trace.view(np.float32)
    for step, (tgt, vel, cur) in wl.APPENDIX_D.items():
        np.testing.assert_allclose(f[step, 6:9, 0], np.float32(tgt), rtol=2e-7, atol=0)
        np.testing.assert_allclose(f[step, 3:6, 0], np.float32(vel), rtol=2e-7, atol=0)
        assert tuple(trace[step, 9:13, 0].view(np.int32)) == cur
    if pos_libm:
        np.testing.assert_allclose(f[9999, 0:2, 0], np.float32(wl.APPENDIX_D_POS_LIBM), rtol=2e-7)


@needs_ref
def test_ref_reproduces_survey_appendix_d():
    _, tr = _run("ref", wl.c1_inputs(), lib="libref_vdt_libm.so")
    _check_appendix_d(tr, pos_libm=True)


def test_port_reproduces_survey_appendix_d():
    # every column except pos is independent of the sin/cos shim
    _, tr = _run("port", wl.c1_inputs())
    _check_appendix_d(tr, pos_libm=False)


def test_port_equals_ref_c1_trace():
    s_ref, t_ref = ol.reference_result("vdt_c1", lambda kind: _run(kind, wl.c1_inputs()), "libref_vdt.so")
    s_port, t_port = _run("port", wl.c1_inputs())
    np.testing.assert_array_equal(t_port, t_ref)
    np.testing.assert_array_equal(s_port, s_ref)


@pytest.mark.parametrize("seed", [0x5EED, 7])
def test_port_equals_ref_plant_rollout(seed):
    inp = wl.plant_inputs(48, 2000, seed=seed)
    s_ref, t_ref = ol.reference_result(f"vdt_plant_{seed}", lambda kind: _run(kind, inp), "libref_vdt.so")
    s_port, t_port = _run("port", inp)
    np.testing.assert_array_equal(t_port, t_ref)
    np.testing.assert_array_equal(s_port, s_ref)


def test_port_equals_ref_stream_rollout():
    from roboken_fmskf_robot_controller_b200 import streams

    inp = wl.plant_inputs(32, 600, seed=11)
    fr = streams.vehicle_frames(32, 600, seed=11)
    s_ref, t_ref = ol.reference_result("vdt_stream", lambda kind: _run(kind, inp, sensor=_cabi.RK_SENSOR_STREAM, frames=fr),
                                       "libref_vdt.so")
    s_port, t_port = _run("port", inp, sensor=_cabi.RK_SENSOR_STREAM, frames=fr)
    np.testing.assert_array_equal(t_port, t_ref)
    np.testing.assert_array_equal(s_port, s_ref)


def test_port_equals_ref_from_random_states():
    n = 512
    st0 = layout.aos_to_soa(wl.random_states(n, seed=3))
    inp = wl.plant_inputs(n, 40, seed=5, seg_len=8, yaw_period=4)
    s_ref, t_ref = ol.reference_result("vdt_random_states", lambda kind: _run(kind, inp, state=st0), "libref_vdt.so")
    s_port, t_port = _run("port", inp, state=st0)
    np.testing.assert_array_equal(t_port, t_ref)
    np.testing.assert_array_equal(s_port, s_ref)
    # hold mode (no frames) as well
    s_ref, t_ref = ol.reference_result("vdt_random_states_hold", lambda kind: _run(kind, inp, sensor=_cabi.RK_SENSOR_HOLD, state=st0),
                                       "libref_vdt.so")
    s_port, t_port = _run("port", inp, sensor=_cabi.RK_SENSOR_HOLD, state=st0)
    np.testing.assert_array_equal(t_port, t_ref)
    np.testing.assert_array_equal(s_port, s_ref)


def test_mymath_known_answers():
    xs = np.concatenate([np.linspace(-50, 50, 4001), [0.0, 6.2831855, 6.283185, -6.2831855, 360.0, -360.0, 720.5]]).astype(np.float32)

    def values(kind):
        lib, pre = (ol.ref(), "ref_") if kind == "ref" else (ol.port(), "orc_")
        fn = {nm: getattr(lib, pre + nm) for nm in ("atan2f", "atanf", "normalize_rad_0to2pi", "normalize_deg_0to360")}
        sin, cos = (lib.ref_sinf, lib.ref_cosf) if kind == "ref" else (lib.orc_sin, lib.orc_cos)
        known = [fn["atan2f"](1, 1), fn["atanf"](0.5), fn["atan2f"](-1, -2), fn["normalize_rad_0to2pi"](-0.5),
                 fn["normalize_rad_0to2pi"](7), fn["normalize_deg_0to360"](-190)]
        return [np.float32(known)] + [np.float32([f(x) for x in xs]) for f in (fn["normalize_rad_0to2pi"], fn["normalize_deg_0to360"], sin, cos)]

    r = ol.reference_result("mymath", values, "libref_vdt.so")
    # SURVEY.md Appendix D
    np.testing.assert_array_equal(r[0], np.float32([0.785398185, 0.463646978, -2.67794585, 5.78318548, 0.716814518, 170]))
    for got, exp in zip(values("port"), r):
        np.testing.assert_array_equal(got.view(np.uint32), exp.view(np.uint32))


def test_sin_table_accuracy():
    """The restated CMSIS table-lerp is a sine to ~2e-5 (its documented accuracy)."""
    p = ol.port()
    xs = np.linspace(0, 2 * np.pi, 5000, endpoint=False).astype(np.float32)
    s = np.array([p.orc_sin(x) for x in xs])
    c = np.array([p.orc_cos(x) for x in xs])
    assert np.max(np.abs(s - np.sin(xs.astype(np.float64)))) < 3e-5
    assert np.max(np.abs(c - np.cos(xs.astype(np.float64)))) < 3e-5
