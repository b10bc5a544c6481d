"""A launch of rk_imt_update without per-update output (no output page, no yaw: the full tick's IMU, the boot init)
forms the end state from the last sample with a quaternion frame instead of running every update.  Its state words are
compared bit for bit with the port running every update, over flag patterns where that sample is the last, an earlier
one or none, and through rk_tick_rollout with the register table and with the samples drawn from the descriptor."""
import numpy as np
import pytest
import torch

import oracle_lib as ol
from roboken_fmskf_robot_controller_b200 import layout, streams
from roboken_fmskf_robot_controller_b200.devstreams import DeviceStreams
from roboken_fmskf_robot_controller_b200.imu import ImuBatch
from roboken_fmskf_robot_controller_b200.robot import RobotBatch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PATTERNS = ("all", "none", "only_first", "only_last_missing", "last_1_missing", "last_5_missing", "last_99_missing",
            "drop_1_in_3", "drop_1_in_64")
PER_PATTERN = 37  # robots per pattern; the patterns are interleaved so that the lanes of a warp scan different lengths


def flag_patterns(K, rng):
    """uint8 [K, n]: robot i follows PATTERNS[i % len(PATTERNS)]."""
    n = PER_PATTERN * len(PATTERNS)
    have = np.ones((K, n), dtype=np.uint8)
    for p, name in enumerate(PATTERNS):
        col = have[:, p :: len(PATTERNS)]
        if name == "none":
            col[:] = 0
        elif name == "only_first":
            col[1:] = 0
        elif name == "only_last_missing":
            col[K - 1] = 0
        elif name.startswith("last_"):
            col[max(0, K - int(name.split("_")[1])) :] = 0
        elif name.startswith("drop_1_in_"):
            col[:] = rng.integers(0, int(name.split("_")[-1]), col.shape) != 0
    return have


def start_state(n, seed):
    """A booted block (q_init latched from a random sample) with the error bit set on every other IMU."""
    regs, _ = streams.imu_samples(n, 1, seed=seed)
    st = np.zeros(layout.IS_WORDS * n, dtype=np.uint32)
    ol.imu_port(st, n, regs, None, do_init=True)
    aos = layout.soa_to_aos(st, n, layout.IS_WORDS)
    aos[1::2, layout.IS_FLAGS] |= layout.IS_FLAG_ERROR
    return layout.aos_to_soa(aos)


def gpu_state(state, regs, have, do_init):
    n = regs.shape[2]
    ib = ImuBatch(n, DEV)
    ib.load_state_soa(state)
    ib.update(torch.from_numpy(streams.imu_cells(regs)).to(DEV), None if have is None else torch.from_numpy(have).to(DEV), None, do_init)
    torch.cuda.synchronize()
    return ib.state.cpu().numpy().view(np.uint32)


def port_state(state, regs, have, do_init):
    st = state.copy()
    ol.imu_port(st, regs.shape[2], regs, have, do_init=do_init)
    return st


@pytest.mark.parametrize("K,do_init", [(1, False), (2, False), (100, False), (1, True), (2, True), (3, True), (100, True)])
@pytest.mark.parametrize("with_flags", [True, False])
def test_state_equals_every_update(K, do_init, with_flags):
    rng = np.random.default_rng(K * 10 + do_init)
    have = flag_patterns(K, rng)
    n = have.shape[1]
    regs, _ = streams.imu_samples(n, K, seed=1000 + K)
    have = have if with_flags else None
    st0 = start_state(n, 7)
    np.testing.assert_array_equal(gpu_state(st0, regs, have, do_init), port_state(st0, regs, have, do_init))


@pytest.mark.parametrize("K,do_init", [(2, False), (100, False), (3, True), (100, True)])
def test_other_samples_are_not_observable(K, do_init):
    """Every sample except the one the end state is formed from (and the init sample) is overwritten with random
    registers after the port ran on the original table: the GPU state still equals the port's.  The update loop passes
    this too (its end state depends on the same sample); what it guards is the choice of that sample -- a kernel that
    forms the page from any other sample (one too early or too late, the wrong side of the init) reads noise here."""
    rng = np.random.default_rng(K)
    have = flag_patterns(K, rng)
    n = have.shape[1]
    regs, _ = streams.imu_samples(n, K, seed=2000 + K)
    st0 = start_state(n, 8)
    exp = port_state(st0, regs, have, do_init)
    u0 = 1 if do_init else 0
    keep = np.zeros((K, n), dtype=bool)
    keep[:u0] = True
    for i in range(n):
        hit = np.nonzero(have[u0:, i])[0]
        if len(hit):
            keep[u0 + hit[-1], i] = True
    noise = rng.integers(-32768, 32768, regs.shape, dtype=np.int16)
    regs2 = np.where(keep[:, None, :], regs, noise)
    assert (regs2 != regs).any()
    np.testing.assert_array_equal(gpu_state(st0, regs2, have, do_init), exp)


@pytest.mark.parametrize("first_update", [0, 5])
@pytest.mark.parametrize("drop_every", [0, 3, 64])
def test_tick_imu_state_table_and_descriptor_equal_port(first_update, drop_every):
    """rk_tick_rollout's IMU, reading the register table and drawing the samples from the same descriptor in registers,
    ends in the state of the port's full_tick (which runs every update)."""
    n, steps, slow, seg_len, seed, first = 1500, 300, 10, 125, 77, 4096
    n_seg, n_slow = (steps + seg_len - 1) // seg_len, (steps + slow - 1) // slow
    ds = DeviceStreams(DEV, seed=seed, first=first, first_update=first_update, drop_every=drop_every)
    cmd = ds.vehicle_commands(torch.empty((n_seg, n, 4), dtype=torch.int32, device=DEV))
    yawc = torch.empty((n_slow, n), dtype=torch.int16, device=DEV)
    regs, have = ds.imu_samples(torch.empty((n_slow, 2, n, 8), dtype=torch.int16, device=DEV),
                                torch.empty((n_slow, n), dtype=torch.uint8, device=DEV), yaw_reg=yawc)
    boot = DeviceStreams(DEV, seed=seed + 1, first=first).imu_samples(torch.empty((1, 2, n, 8), dtype=torch.int16, device=DEV), None)[0]
    got = {}
    for name, kw in (("table", dict(regs=regs)), ("descriptor", dict(regs=None, imu_desc=ds))):
        rb = RobotBatch(n, DEV)
        rb.reset()
        rb.imu.update(boot, None, None, do_init=True)
        rb.rollout(steps, slow, cmd=cmd, seg_len=seg_len, have_quat=have, yaw_reg=yawc, yaw=torch.zeros(n, dtype=torch.float32, device=DEV), **kw)
        torch.cuda.synchronize()
        got[name] = (rb.imu.state.cpu().numpy().view(np.uint32).copy(), rb.vehicle.state.cpu().numpy().view(np.uint32).copy())
    gidx = np.arange(n, dtype=np.uint64) + np.uint64(first)
    regs_h, have_h = streams.imu_samples_v2(0, n_slow, seed, drop_every=drop_every, inst=gidx, first_update=first_update)
    np.testing.assert_array_equal(have_h, have.cpu().numpy())
    if drop_every == 3:
        assert 0.2 < 1.0 - have_h[-1].mean() < 0.45  # the last sample misses its frame for about a third of the robots
    boot_h, _ = streams.imu_samples_v2(0, 1, seed + 1, inst=gidx)
    v, i, a, t = (np.zeros(w * n, dtype=np.uint32) for w in (layout.VS_WORDS, layout.IS_WORDS, layout.AS_WORDS, layout.ACMD_WORDS))
    ol.imu_port(i, n, boot_h, None, do_init=True)
    ol.arm_batch("port", "init", a, t, n)
    cmd_h = streams.vehicle_commands_v2(0, n_seg, seed, inst=gidx)
    ol.full_tick("port", n, steps, slow, cmd_h, seg_len, regs_h, have_h, v, i, a, t, nthreads=8)
    for name, (gi, gv) in got.items():
        np.testing.assert_array_equal(gi, i, err_msg=f"{name}: IMU state")
        np.testing.assert_array_equal(gv, v, err_msg=f"{name}: vehicle state")
