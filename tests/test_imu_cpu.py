"""CPU: pin the IMU part of the plain-C oracle against the compiled reference (lib/wt901c
frame parser + IMU_IF_WT901C driven through serial frames) and SURVEY.md Appendix D."""
import os

import numpy as np
import pytest

import oracle_lib as ol
from roboken_fmskf_robot_controller_b200 import layout, streams

needs_ref = pytest.mark.skipif(not ol.have_ref("libref_imu.so"), reason="oracle/_ref/libref_imu.so not available")
GOLD = os.path.join(os.path.dirname(__file__), "golden", "imu_golden.npz")

APPX_D_INIT = np.array([0] * 12 + [32767, 0, 0, 0], dtype=np.int16)
APPX_D_REGS = np.array([2048, -1024, 512, 164, -328, 16384, 11, -22, 33, -16384, 8192, -24576, 23170, 100, -200, 23170], dtype=np.int16)
APPX_D_OUT = np.array([1, 0.5, -0.25, 10.0097656, 20.0195312, -1000, 11, 22, -33, 90, 45, -135,
                       0.00305166468, -0.00610332936, 0.707070708, 0.707070708], dtype=np.float32)


def _appendix_d(fn):
    regs = np.stack([APPX_D_INIT, APPX_D_REGS, APPX_D_REGS]).reshape(3, 16, 1).copy()
    have = np.array([[1], [1], [0]], dtype=np.uint8)
    st = np.zeros(layout.IS_WORDS, dtype=np.uint32)
    out = fn(st, 1, regs, have, want_out=True, do_init=True)
    f = out.view(np.float32).reshape(3, 16)
    np.testing.assert_allclose(f[1], APPX_D_OUT, rtol=2e-7)
    np.testing.assert_array_equal(f[2], f[1])  # no quaternion frame: data retained ...
    assert st[layout.IS_FLAGS] & 1  # ... and isError() set
    assert f[1, layout.IS_D_ANGLE + 2] == -135.0  # getYawDate()


def test_port_appendix_d():
    _appendix_d(ol.imu_port)


@needs_ref
def test_ref_appendix_d():
    _appendix_d(ol.imu_ref)


def test_port_equals_ref_random_streams():
    n, K = 96, 40
    regs, have = streams.imu_samples(n, K, seed=5, drop_every=7)
    have[0] = 1
    regs2, have2 = streams.imu_samples(n, K, seed=6, drop_every=5)

    def run(kind):
        fn = ol.imu_port if kind == "port" else ol.imu_ref
        st = np.zeros(layout.IS_WORDS * n, dtype=np.uint32)
        o1 = fn(st, n, regs, have, want_out=True, do_init=True)
        s1 = st.copy()
        o2 = fn(st, n, regs2, have2, want_out=True)  # continue from that state without init
        return o1, s1, o2, st

    for x, y in zip(run("port"), ol.reference_result("imu_random_streams", run, "libref_imu.so")):
        np.testing.assert_array_equal(x, y)


def test_golden_imu():
    g = np.load(GOLD)
    n, K = 64, 32
    regs, have = streams.imu_samples(n, K, seed=0x5EED, drop_every=8)
    st = np.zeros(layout.IS_WORDS * n, dtype=np.uint32)
    out = ol.imu_port(st, n, regs, have, want_out=True, do_init=True)
    np.testing.assert_array_equal(out, g["out"])
    np.testing.assert_array_equal(st, g["state"])
