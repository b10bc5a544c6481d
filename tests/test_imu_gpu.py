"""GPU parity: rk_imt_update / rk_imt_update_yaw (C-ABI) vs the oracle / golden fixture, bit-exact."""
import os

import numpy as np
import pytest
import torch

import oracle_lib as ol
from roboken_fmskf_robot_controller_b200 import _cabi, layout, streams
from roboken_fmskf_robot_controller_b200.imu import Imu, ImuBatch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def gpu_imu(n, regs, have, state=None, do_init=False, want_out=True):
    ib = ImuBatch(n, DEV)
    if state is not None:
        ib.load_state_soa(state)
    K = regs.shape[0]
    out = torch.zeros((K, 4, n, 4), dtype=torch.float32, device=DEV) if want_out else None
    ib.update(torch.from_numpy(streams.imu_cells(regs)).to(DEV), None if have is None else torch.from_numpy(have).to(DEV), out, do_init)
    torch.cuda.synchronize()
    return ib.state.cpu().numpy().view(np.uint32), (out.cpu().numpy().view(np.uint32) if want_out else None)


def test_imu_golden_and_port():
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "imu_golden.npz"))
    n, K = 64, 32
    regs, have = streams.imu_samples(n, K, seed=0x5EED, drop_every=8)
    st, out = gpu_imu(n, regs, have, do_init=True)
    np.testing.assert_array_equal(out, g["out"])
    np.testing.assert_array_equal(st, g["state"])


@pytest.mark.parametrize("n,K,seed", [(1, 5, 1), (1000, 64, 2), (4099, 16, 3)])
def test_imu_vs_port(n, K, seed):
    regs, have = streams.imu_samples(n, K, seed=seed, drop_every=5)
    a = np.zeros(layout.IS_WORDS * n, dtype=np.uint32)
    oa = ol.imu_port(a, n, regs, have, want_out=True, do_init=True)
    st, out = gpu_imu(n, regs, have, do_init=True)
    np.testing.assert_array_equal(out, oa)
    np.testing.assert_array_equal(st, a)
    regs2, have2 = streams.imu_samples(n, K, seed=seed + 100, drop_every=3)
    oa = ol.imu_port(a, n, regs2, have2, want_out=True)
    st2, out2 = gpu_imu(n, regs2, have2, state=st)
    np.testing.assert_array_equal(out2, oa)
    np.testing.assert_array_equal(st2, a)


@pytest.mark.parametrize("do_init", [True, False])
@pytest.mark.parametrize("with_have", [True, False])
@pytest.mark.parametrize("with_out", [True, False])
def test_imu_yaw_entry_vs_port(with_out, with_have, do_init):
    """rk_imt_update_yaw, with the output page and with the yaw alone: every update's yaw is the port's Data.angle[2]
    times DEG2RAD in float32, and the page and the state block are the port's, bit for bit."""
    n, K = 1000, 9
    seed = 20 + 4 * with_out + 2 * with_have + do_init
    regs, have = streams.imu_samples(n, K, seed=seed, drop_every=3)
    have = have if with_have else None
    st0 = np.zeros(layout.IS_WORDS * n, dtype=np.uint32)
    ol.imu_port(st0, n, streams.imu_samples(n, 1, seed=seed + 100)[0], None, do_init=True)  # a booted block
    exp = st0.copy()
    oe = ol.imu_port(exp, n, regs, have, want_out=True, do_init=do_init)
    yaw_exp = (np.ascontiguousarray(oe[:, 2, :, 3]).view(np.float32) * streams.DEG2RAD).astype(np.float32)  # Data.angle[2]
    ib = ImuBatch(n, DEV)
    ib.load_state_soa(st0)
    regs_d = torch.from_numpy(streams.imu_cells(regs)).to(DEV)
    have_d = None if have is None else torch.from_numpy(have).to(DEV)
    out = torch.zeros((K, 4, n, 4), dtype=torch.float32, device=DEV) if with_out else None
    yaw = torch.zeros((K, n), dtype=torch.float32, device=DEV)
    _cabi.check(ib.lib.rk_imt_update_yaw(ib.state.data_ptr(), n, K, regs_d.data_ptr(), None if have_d is None else have_d.data_ptr(),
                                         None if out is None else out.data_ptr(), yaw.data_ptr(), int(do_init), None))
    torch.cuda.synchronize()
    np.testing.assert_array_equal(yaw.cpu().numpy().view(np.uint32), yaw_exp.view(np.uint32))
    if with_out:
        np.testing.assert_array_equal(out.cpu().numpy().view(np.uint32), oe)
    np.testing.assert_array_equal(ib.state.cpu().numpy().view(np.uint32), exp)


def test_imu_extreme_registers():
    """Every register at its int16 extremes (roll wrap at +-180 deg, -32768 quaternion words)."""
    vals = np.array([-32768, -32767, -1, 0, 1, 16384, -16384, 32767], dtype=np.int16)
    n = len(vals) ** 2
    regs = np.zeros((2, 16, n), dtype=np.int16)
    a, b = np.meshgrid(vals, vals)
    for r in range(16):
        regs[:, r, :] = (a if r % 2 == 0 else b).reshape(-1)
    regs[0, 12:16] = np.roll(regs[1, 12:16], 3, axis=-1)
    exp = np.zeros(layout.IS_WORDS * n, dtype=np.uint32)
    oe = ol.imu_port(exp, n, regs, None, want_out=True, do_init=True)
    st, out = gpu_imu(n, regs, None, do_init=True)
    np.testing.assert_array_equal(out, oe)
    np.testing.assert_array_equal(st, exp)


def test_imu_full_size_c3():
    """BASELINE.json configs[2]: 2^20 batched updates; sampled parity + a checksum of the
    integer-valued outputs (mag is an exact copy of the registers with Y/Z negated)."""
    n, K = 1 << 20, 1
    regs, have = streams.imu_samples(n, K + 1, seed=9, drop_every=64)
    have[0] = 1
    st, out = gpu_imu(n, regs, have, do_init=True)
    idx = np.unique(np.random.default_rng(0).integers(0, n, 300))
    exp = np.zeros(layout.IS_WORDS * len(idx), dtype=np.uint32)
    ol.imu_port(exp, len(idx), np.ascontiguousarray(regs[:, :, idx]), np.ascontiguousarray(have[:, idx]), do_init=True)
    got = layout.soa_to_aos(st, n, layout.IS_WORDS)[idx]
    np.testing.assert_array_equal(got, layout.soa_to_aos(exp, len(idx), layout.IS_WORDS))
    f = out.view(np.float32)[1]  # [4, n, 4] planes of the second sample
    ok = have[1] != 0
    mag_x = f[1, :, 2]  # word 6
    np.testing.assert_array_equal(mag_x[ok], regs[1, 6, ok].astype(np.float32))


def test_imu_single_instance_handle_appendix_d():
    imu = Imu()
    imu.init([0] * 12 + [32767, 0, 0, 0])
    imu.update([2048, -1024, 512, 164, -328, 16384, 11, -22, 33, -16384, 8192, -24576, 23170, 100, -200, 23170])
    d, err = imu.getDataLatest()
    exp = np.array([1, 0.5, -0.25, 10.0097656, 20.0195312, -1000, 11, 22, -33, 90, 45, -135,
                    0.00305166468, -0.00610332936, 0.707070708, 0.707070708], dtype=np.float32)
    np.testing.assert_allclose(d, exp, rtol=2e-7)
    assert not err and imu.getYawDate() == -135.0
    imu.update([7] * 16, have_quat=False)
    d2, err2 = imu.getDataLatest()
    assert err2 and np.array_equal(d2, d)
    imu.close()
