"""GPU parity of the full controller tick (rk_tick_rollout: vehicle + IMU + arm coupled through the
IMU yaw) against the per-module oracles composed on the host, bit for bit."""
import numpy as np
import pytest
import torch

import oracle_lib as ol
from roboken_fmskf_robot_controller_b200 import _cabi, layout, streams
from roboken_fmskf_robot_controller_b200.robot import RobotBatch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def make_inputs(n, steps, slow, seed, seg_len=125):
    n_seg = (steps + seg_len - 1) // seg_len
    n_slow = (steps + slow - 1) // slow
    cmd = streams.vehicle_commands(n, n_seg, seed)
    regs, have = streams.imu_samples(n, n_slow + 1, seed=seed, drop_every=16)
    seq = streams.arm_sequences(n, seed=seed, seq_id=3, max_len=12)
    return cmd, regs, have, seq


def gpu_full(n, steps, slow, cmd, regs, have, seq, trace=True, goal=None):
    rb = RobotBatch(n, DEV)
    rb.reset()
    # IMU boot: IMU_IF_WT901C::init() consumes the first sample; arm: one sequence pushed
    rb.imu.update(torch.from_numpy(streams.imu_cells(regs[:1])).to(DEV), None, None, do_init=True)
    rb.arm.push_cmdseq(torch.from_numpy(layout.aos_to_soa(seq).view(np.int32)).to(DEV))
    n_slow = (steps + slow - 1) // slow
    cmd_d = torch.from_numpy(cmd.view(np.int32).reshape(cmd.shape[0], n, 4)).to(DEV)
    regs_d = torch.from_numpy(streams.imu_cells(regs[1 : 1 + n_slow])).to(DEV)
    have_d = torch.from_numpy(np.ascontiguousarray(have[1 : 1 + n_slow])).to(DEV)
    yaw_d = torch.zeros((n_slow, n), dtype=torch.float32, device=DEV)
    vtr = torch.zeros((steps, 16, n), dtype=torch.int32, device=DEV) if trace else None
    atr = torch.zeros((n_slow, 16, n), dtype=torch.int32, device=DEV) if trace else None
    goal_d = cost_d = None
    if goal is not None:
        goal_d, cost_d = torch.from_numpy(goal).to(DEV), torch.zeros(n, dtype=torch.float32, device=DEV)
    rb.rollout(steps, slow, cmd=cmd_d, seg_len=125, regs=regs_d, have_quat=have_d, yaw=yaw_d, vdt_trace=vtr, adt_trace=atr,
               goal=goal_d, cost=cost_d)
    torch.cuda.synchronize()
    u = lambda t: None if t is None else t.cpu().numpy().view(np.uint32)
    return dict(v=u(rb.vehicle.state), i=u(rb.imu.state), a=u(rb.arm.state), vtr=u(vtr), atr=u(atr), yaw=yaw_d.cpu().numpy(),
                cost=None if cost_d is None else cost_d.cpu().numpy())


def oracle_full(kind, n, steps, slow, cmd, regs, have, seq, trace=True, goal=None):
    v = np.zeros(layout.VS_WORDS * n, dtype=np.uint32)
    i = np.zeros(layout.IS_WORDS * n, dtype=np.uint32)
    a = np.zeros(layout.AS_WORDS * n, dtype=np.uint32)
    t = np.zeros(layout.ACMD_WORDS * n, dtype=np.uint32)
    (ol.imu_port if kind == "port" else ol.imu_ref)(i, n, regs[:1], None, do_init=True)
    ol.arm_batch(kind, "init", a, t, n)
    ol.arm_batch(kind, "push", a, t, n, seq=layout.aos_to_soa(seq))
    n_slow = (steps + slow - 1) // slow
    vtr, atr, yaw, cost = ol.full_tick(kind, n, steps, slow, cmd, 125, np.ascontiguousarray(regs[1 : 1 + n_slow]),
                                       np.ascontiguousarray(have[1 : 1 + n_slow]), v, i, a, t, trace=trace, goal=goal, nthreads=8)
    return dict(v=v, i=i, a=a, vtr=vtr, atr=atr, yaw=yaw, cost=cost)


def compare(g, o):
    # the yaw the vehicle took before every tick is word 2 of its trace (pos.th), so the coupling is compared tick by tick
    for k in ("vtr", "atr", "v", "i", "a"):
        if g[k] is not None:
            np.testing.assert_array_equal(g[k], o[k], err_msg=k)


@pytest.mark.parametrize("n,steps,seed", [(300, 1000, 41), (1, 95, 42), (2050, 250, 43)])
def test_full_tick_vs_port(n, steps, seed):
    inp = make_inputs(n, steps, 10, seed)
    compare(gpu_full(n, steps, 10, *inp), oracle_full("port", n, steps, 10, *inp))


def test_full_tick_vs_compiled_reference():
    n, steps = 64, 600
    inp = make_inputs(n, steps, 10, 44)
    exp = ol.reference_result("full_tick_gpu", lambda kind: oracle_full(kind, n, steps, 10, *inp), "libref_vdt.so", "libref_imu.so", "libref_arm.so")
    compare(gpu_full(n, steps, 10, *inp), exp)


def test_full_tick_cost_and_slice_invariance():
    """The G-GPU result equals the 1-GPU result slice by slice (SURVEY 8e): a rollout of the second
    half of the instances alone gives the second half of the full rollout's costs and states."""
    n, steps = 512, 400
    cmd, regs, have, seq = make_inputs(n, steps, 10, 45)
    goal = np.zeros((n, 2), dtype=np.float32)
    full = gpu_full(n, steps, 10, cmd, regs, have, seq, trace=False, goal=goal)
    h = n // 2
    half = gpu_full(h, steps, 10, np.ascontiguousarray(cmd[:, h:]), np.ascontiguousarray(regs[:, :, h:]),
                    np.ascontiguousarray(have[:, h:]), seq[h:], trace=False, goal=goal[h:])
    np.testing.assert_array_equal(full["cost"][h:].view(np.uint32), half["cost"].view(np.uint32))
    np.testing.assert_array_equal(layout.soa_to_aos(full["v"], n, layout.VS_WORDS)[h:], layout.soa_to_aos(half["v"], h, layout.VS_WORDS))
    np.testing.assert_array_equal(layout.soa_to_aos(full["a"], n, layout.AS_WORDS)[h:], layout.soa_to_aos(half["a"], h, layout.AS_WORDS))
    o = oracle_full("port", n, steps, 10, cmd, regs, have, seq, trace=False, goal=goal)
    np.testing.assert_array_equal(full["cost"].view(np.uint32), o["cost"].view(np.uint32))


# ---- BASELINE configs[4] at full size ------------------------------------------------------------------------
def _device_chunk(dev, n, first, steps, slow, seed, seg_len=125, side_ctas=None):
    """One chunk of the bench's full-tick launch on `dev`: tables expanded on the device from the descriptor, IMU boot,
    arm bring-up + sequence push, rk_tick_rollout.  Returns the RobotBatch and the cost vector."""
    from roboken_fmskf_robot_controller_b200.devstreams import DeviceStreams

    n_seg, n_slow = (steps + seg_len - 1) // seg_len, (steps + slow - 1) // slow
    with torch.cuda.device(dev):
        rb = RobotBatch(n, dev)
        if side_ctas is not None:
            rb.lib.rk_set_option(_cabi.RK_OPT_TICK_SIDE_CTAS, side_ctas)
        rb.reset()
        boot = DeviceStreams(dev, seed=seed, first=first, first_update=0).imu_samples(torch.empty((1, 2, n, 8), dtype=torch.int16, device=dev), None)[0]
        rb.imu.update(boot, None, None, do_init=True)
        ds = DeviceStreams(dev, seed=seed, first=first, first_update=1, arm_seq_id=1)
        cmd = ds.vehicle_commands(torch.empty((n_seg, n, 4), dtype=torch.int32, device=dev))
        regs, have = ds.imu_samples(torch.empty((n_slow, 2, n, 8), dtype=torch.int16, device=dev), torch.empty((n_slow, n), dtype=torch.uint8, device=dev))
        seq = ds.arm_sequences(torch.empty(layout.ACMD_SLOT_WORDS * n, dtype=torch.int32, device=dev))
        rb.arm.push_cmdseq(seq)
        cost = torch.zeros(n, dtype=torch.float32, device=dev)
        rb.rollout(steps, slow, cmd=cmd, seg_len=seg_len, regs=regs, have_quat=have, yaw=torch.zeros(n, dtype=torch.float32, device=dev),
                   goal=torch.zeros((n, 2), dtype=torch.float32, device=dev), cost=cost)
        torch.cuda.synchronize(dev)
    return rb, cost


def _oracle_sample(kind, gidx, steps, slow, seed, seg_len=125):
    """The same robots (global indices gidx) through the per-module oracles on host-generated copies of their streams."""
    m = len(gidx)
    n_seg, n_slow = (steps + seg_len - 1) // seg_len, (steps + slow - 1) // slow
    cmd = streams.vehicle_commands_v2(0, n_seg, seed, inst=gidx)
    regs, have = streams.imu_samples_v2(0, n_slow + 1, seed, inst=gidx)
    seq = streams.arm_sequences_v2(0, seed, inst=gidx, seq_id=1)
    v, i, a, t = (np.zeros(w * m, dtype=np.uint32) for w in (layout.VS_WORDS, layout.IS_WORDS, layout.AS_WORDS, layout.ACMD_WORDS))
    (ol.imu_port if kind == "port" else ol.imu_ref)(i, m, regs[:1], None, do_init=True)
    ol.arm_batch(kind, "init", a, t, m)
    ol.arm_batch(kind, "push", a, t, m, seq=layout.aos_to_soa(seq))
    _, _, _, cost = ol.full_tick(kind, m, steps, slow, cmd, seg_len, np.ascontiguousarray(regs[1:]), np.ascontiguousarray(have[1:]), v, i, a, t,
                                 goal=np.zeros((m, 2), dtype=np.float32), nthreads=8)
    return v, i, a, np.asarray(cost, dtype=np.float32)


def _assert_sample_equal(rb, cost, idx, exp, what):
    n, m = rb.n, len(idx)
    v, i, a, c = exp
    for got, e, words, name in ((rb.vehicle.state, v, layout.VS_WORDS, "vehicle"), (rb.imu.state, i, layout.IS_WORDS, "imu"),
                                (rb.arm.state, a, layout.AS_WORDS, "arm")):
        g = layout.soa_to_aos(got.cpu().numpy().view(np.uint32), n, words)[idx]
        np.testing.assert_array_equal(g, layout.soa_to_aos(e, m, words), err_msg=f"{what}: {name} state")
    np.testing.assert_array_equal(cost.cpu().numpy()[idx].view(np.uint32), c.view(np.uint32), err_msg=f"{what}: cost")


def test_full_size_c5_sampled_parity_vs_reference():
    """BASELINE configs[4] at its full size -- 2^24 robots x 1000 ticks in 16 chunks of 2^20, exactly the bench's launches
    (device-generated streams, rk_tick_rollout with the IMU / arm kernels in the vehicle rollout's shadow) -- with 24
    robots sampled from every chunk (384 in all) compared bit for bit, all three state blocks and the rollout cost,
    against the reference's own sources compiled for x86 (the port if oracle/_ref is absent)."""
    kind = "ref" if (ol.have_ref("libref_arm.so") and ol.have_ref("libref_imu.so") and ol.have_ref("libref_vdt.so")) else "port"
    n, steps, slow, seed = 1 << 20, 1000, 10, 0x5EED
    total = 0
    for c in range(16):
        first = c * n
        rb, cost = _device_chunk(DEV, n, first, steps, slow, seed)
        idx = np.unique(np.concatenate([[0, n - 1], np.random.default_rng(c).integers(0, n, 22)]))
        _assert_sample_equal(rb, cost, idx, _oracle_sample(kind, idx.astype(np.uint64) + np.uint64(first), steps, slow, seed), f"chunk {c}")
        total += len(idx)
        del rb, cost
        torch.cuda.empty_cache()
    assert total >= 256


def test_side_kernel_cap_does_not_change_results():
    """RK_OPT_TICK_SIDE_CTAS only schedules: full grids, one and two CTAs per SM give the same bits."""
    n, steps = 40000, 300
    ref = None
    try:
        for cap in (0, 1, 2):
            rb, cost = _device_chunk(DEV, n, 777, steps, 10, 5, side_ctas=cap)
            got = [t.cpu().numpy().copy() for t in (rb.vehicle.state, rb.imu.state, rb.arm.state, cost)]
            if ref is None:
                ref = got
            for x, y in zip(got, ref):
                np.testing.assert_array_equal(x.view(np.uint32), y.view(np.uint32))
    finally:
        RobotBatch(1, DEV).lib.rk_set_option(_cabi.RK_OPT_TICK_SIDE_CTAS, 1)


def test_yaw_column_equals_register_cells():
    """rk_tick_rollout_t::d_yaw_reg: the vehicle reading the Yaw register from the 2-byte column the generator writes beside
    the register cells gives the same blocks and costs as reading it from the cells -- with every third quaternion frame
    missing, so that the hold semantics (and the yaw the IMU block held at launch) are exercised in both forms."""
    from roboken_fmskf_robot_controller_b200.devstreams import DeviceStreams

    n, steps, slow, seg_len = 3000, 400, 10, 125
    n_seg, n_slow = (steps + seg_len - 1) // seg_len, (steps + slow - 1) // slow
    ds = DeviceStreams(DEV, seed=91, first=7, first_update=1, arm_seq_id=1, drop_every=3)
    cmd = ds.vehicle_commands(torch.empty((n_seg, n, 4), dtype=torch.int32, device=DEV))
    yawc = torch.empty((n_slow, n), dtype=torch.int16, device=DEV)
    regs, have = ds.imu_samples(torch.empty((n_slow, 2, n, 8), dtype=torch.int16, device=DEV), torch.empty((n_slow, n), dtype=torch.uint8, device=DEV),
                                yaw_reg=yawc)
    seq = ds.arm_sequences(torch.empty(layout.ACMD_SLOT_WORDS * n, dtype=torch.int32, device=DEV))
    torch.cuda.synchronize()
    np.testing.assert_array_equal(yawc.cpu().numpy(), regs.cpu().numpy()[:, 1, :, 3])  # register 11 = Yaw
    assert 0.2 < 1.0 - have.float().mean().item() < 0.45
    out = []
    for col in (None, yawc):
        rb = RobotBatch(n, DEV)
        rb.reset()
        boot = DeviceStreams(DEV, seed=91, first=7, first_update=0).imu_samples(torch.empty((1, 2, n, 8), dtype=torch.int16, device=DEV), None)[0]
        rb.imu.update(boot, None, None, do_init=True)
        rb.arm.push_cmdseq(seq)
        cost = torch.zeros(n, dtype=torch.float32, device=DEV)
        for _ in range(2):  # the second launch starts from an IMU block that holds a yaw
            rb.rollout(steps, slow, cmd=cmd, seg_len=seg_len, regs=regs, have_quat=have, yaw_reg=col, yaw=torch.zeros(n, dtype=torch.float32, device=DEV),
                       goal=torch.zeros((n, 2), dtype=torch.float32, device=DEV), cost=cost)
        torch.cuda.synchronize()
        out.append([rb.vehicle.state.cpu().numpy().copy(), rb.imu.state.cpu().numpy().copy(), rb.arm.state.cpu().numpy().copy(), cost.cpu().numpy().view(np.uint32).copy()])
    for x, y in zip(*out):
        np.testing.assert_array_equal(x, y)
    # ... and with the IMU update drawing the samples from the descriptor in registers (d_imu_desc): no register table at all
    yc2, hv2 = ds.imu_columns(torch.empty((n_slow, n), dtype=torch.int16, device=DEV), torch.empty((n_slow, n), dtype=torch.uint8, device=DEV))
    torch.cuda.synchronize()
    np.testing.assert_array_equal(yc2.cpu().numpy(), yawc.cpu().numpy())
    np.testing.assert_array_equal(hv2.cpu().numpy(), have.cpu().numpy())
    rb = RobotBatch(n, DEV)
    rb.reset()
    boot = DeviceStreams(DEV, seed=91, first=7, first_update=0).imu_samples(torch.empty((1, 2, n, 8), dtype=torch.int16, device=DEV), None)[0]
    rb.imu.update(boot, None, None, do_init=True)
    rb.arm.push_cmdseq(seq)
    cost = torch.zeros(n, dtype=torch.float32, device=DEV)
    for _ in range(2):
        rb.rollout(steps, slow, cmd=cmd, seg_len=seg_len, regs=None, imu_desc=ds, have_quat=hv2, yaw_reg=yc2, yaw=torch.zeros(n, dtype=torch.float32, device=DEV),
                   goal=torch.zeros((n, 2), dtype=torch.float32, device=DEV), cost=cost)
    torch.cuda.synchronize()
    for x, y in zip(out[0], [rb.vehicle.state.cpu().numpy(), rb.imu.state.cpu().numpy(), rb.arm.state.cpu().numpy(), cost.cpu().numpy().view(np.uint32)]):
        np.testing.assert_array_equal(x, y)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
def test_two_gpu_slices_equal_one_gpu_run():
    """SURVEY 8e on real devices: the two halves of a batch run on cuda:0 and cuda:1 (contiguous slices of the global
    index space, as bench.py shards them) equal the one-GPU run of the whole batch, bit for bit."""
    n, steps, slow, seed = 6000, 500, 10, 77
    whole, cost = _device_chunk("cuda:0", n, 1000, steps, slow, seed)
    lo = _device_chunk("cuda:0", n // 2, 1000, steps, slow, seed)
    hi = _device_chunk("cuda:1", n - n // 2, 1000 + n // 2, steps, slow, seed)
    for words, name in ((layout.VS_WORDS, "vehicle"), (layout.IS_WORDS, "imu"), (layout.AS_WORDS, "arm")):
        w = layout.soa_to_aos(getattr(whole, name).state.cpu().numpy().view(np.uint32), n, words)
        a = layout.soa_to_aos(getattr(lo[0], name).state.cpu().numpy().view(np.uint32), n // 2, words)
        b = layout.soa_to_aos(getattr(hi[0], name).state.cpu().numpy().view(np.uint32), n - n // 2, words)
        np.testing.assert_array_equal(np.concatenate([a, b]), w, err_msg=name)
    np.testing.assert_array_equal(np.concatenate([lo[1].cpu().numpy(), hi[1].cpu().numpy()]).view(np.uint32), cost.cpu().numpy().view(np.uint32))
