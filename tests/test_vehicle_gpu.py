"""GPU parity tests (the first gate): the CUDA path, called through the C-ABI, against the
oracles on the same seeded inputs -- bit-exact on every state word and trace word.

Tolerances: BASELINE.json asks for <=1e-5 relative per step on floats and bit-exact integer
/ mode logic.  The kernels use no FMA contraction and IEEE div/sqrt, so these tests assert
the stronger property: every 32-bit word identical (0 ulp), which implies both.
"""
import os

import numpy as np
import pytest
import torch

import oracle_lib as ol
import workloads as wl
import roboken_fmskf_robot_controller_b200 as rk
from roboken_fmskf_robot_controller_b200 import _cabi, layout, streams
from roboken_fmskf_robot_controller_b200.vehicle import Vehicle, VehicleBatch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
G = np.load(os.path.join(os.path.dirname(__file__), "golden", "vdt_golden.npz"))


def _dev(a, dtype=None):
    if a is None:
        return None
    t = torch.from_numpy(np.ascontiguousarray(a).view(dtype) if dtype is not None else np.ascontiguousarray(a))
    return t.to(DEV)


def gpu_run(inp, sensor=_cabi.RK_SENSOR_PLANT, frames=None, state=None, trace=True, chunks=None):
    n, steps = inp["n"], inp["steps"]
    vb = VehicleBatch(n, DEV)
    if state is not None:
        vb.load_state_soa(state)
    cmd = _dev(inp.get("cmd"), np.int32)
    if cmd is not None:
        cmd = cmd.reshape(-1, n, 4)
    yaw = _dev(inp.get("yaw"))
    fr = _dev(frames, np.int64)
    tr = torch.zeros((steps, 16, n), dtype=torch.int32, device=DEV) if trace else None
    if chunks is None:
        vb.rollout(steps, sensor_mode=sensor, cmd=cmd, seg_len=inp.get("seg_len", 0), yaw=yaw,
                   yaw_period=inp.get("yaw_period", 0), frames=fr, trace=tr, task_period=inp.get("task_period", 0))
    else:
        # resume: K ticks as several launches, each taking its slice of the input tables
        seg_len, yp = inp.get("seg_len", 0), inp.get("yaw_period", 0)
        assert steps % chunks == 0
        k = steps // chunks
        assert (seg_len == 0 or k % seg_len == 0) and (yp == 0 or k % yp == 0)
        for c in range(chunks):
            vb.rollout(k, sensor_mode=sensor,
                       cmd=None if cmd is None else cmd[c * k // seg_len:(c + 1) * k // seg_len].contiguous(),
                       seg_len=seg_len,
                       yaw=None if yaw is None else yaw[c * k // yp:(c + 1) * k // yp].contiguous(), yaw_period=yp,
                       frames=None if fr is None else fr[c * k:(c + 1) * k].contiguous(),
                       trace=None if tr is None else tr[c * k:(c + 1) * k], task_period=inp.get("task_period", 0))
    torch.cuda.synchronize()
    st = vb.state.cpu().numpy().view(np.uint32)
    return st, (tr.cpu().numpy().view(np.uint32) if trace else None)


def port_run(inp, sensor=_cabi.RK_SENSOR_PLANT, frames=None, state=None, trace=True, nthreads=1):
    n = inp["n"]
    st = np.zeros(layout.VS_WORDS * n, dtype=np.uint32) if state is None else state.copy()
    ro = ol.HostRollout(n, inp["steps"], sensor, inp.get("cmd"), inp.get("seg_len", 0), inp.get("yaw"),
                        inp.get("yaw_period", 0), frames=frames, trace=trace)
    ol.run_port(st, n, ro, nthreads=nthreads)
    return st, ro.trace


def host_run(kind, inp, sensor=_cabi.RK_SENSOR_PLANT, frames=None, state=None):
    n = inp["n"]
    st = np.zeros(layout.VS_WORDS * n, dtype=np.uint32) if state is None else state.copy()
    ro = ol.HostRollout(n, inp["steps"], sensor, inp.get("cmd"), inp.get("seg_len", 0), inp.get("yaw"),
                        inp.get("yaw_period", 0), frames=frames, trace=True)
    (ol.run_ref if kind == "ref" else ol.run_port)(st, n, ro)
    return st, ro.trace


def assert_same(a, b, what):
    if not np.array_equal(a, b):
        bad = np.argwhere(a != b)
        raise AssertionError(f"{what}: {len(bad)} words differ, first at {bad[0]}: {a[tuple(bad[0])]:#x} vs {b[tuple(bad[0])]:#x}")


# ---- configs[0]: the reference's own CPU-runnable case -------------------------------------
def test_c1_trace_bit_exact_vs_port_and_golden():
    st, tr = gpu_run(wl.c1_inputs())
    pst, ptr = port_run(wl.c1_inputs())
    assert_same(tr, ptr, "C1 trace vs port")
    assert_same(st, pst, "C1 final state vs port")
    assert_same(tr[G["c1_rows"]], G["c1_trace"], "C1 trace vs golden (unmodified reference)")
    assert_same(st, G["c1_state"], "C1 state vs golden")
    # SURVEY.md Appendix D known answers
    f = tr.view(np.float32)
    for step, (tgt, vel, cur) in wl.APPENDIX_D.items():
        np.testing.assert_allclose(f[step, 6:9, 0], np.float32(tgt), rtol=2e-7)
        np.testing.assert_allclose(f[step, 3:6, 0], np.float32(vel), rtol=2e-7)
        assert tuple(tr[step, 9:13, 0].view(np.int32)) == cur


def test_plant_rollout_bit_exact_vs_compiled_reference():
    inp = wl.plant_inputs(64, 1500, seed=3)
    st, tr = gpu_run(inp)
    rst, rtr = ol.reference_result("vdt_gpu_plant", lambda kind: host_run(kind, inp), "libref_vdt.so")
    assert_same(tr, rtr, "plant trace vs compiled reference")
    assert_same(st, rst, "plant state vs compiled reference")


@pytest.mark.parametrize("seed,n,steps", [(0x5EED, 256, 1000), (7, 33, 2000), (99, 1, 500)])
def test_plant_rollout_bit_exact_vs_port(seed, n, steps):
    inp = wl.plant_inputs(n, steps, seed=seed)
    st, tr = gpu_run(inp)
    pst, ptr = port_run(inp, nthreads=8)
    assert_same(tr, ptr, "plant trace")
    assert_same(st, pst, "plant state")


def test_golden_plant_and_stream_and_random():
    st, tr = gpu_run(wl.plant_inputs(16, 1000, seed=0x5EED))
    assert_same(tr[::100], G["plant_trace"], "golden plant trace")
    assert_same(st, G["plant_state"], "golden plant state")
    fr = streams.vehicle_frames(8, 300, seed=21)
    st, tr = gpu_run(wl.plant_inputs(8, 300, seed=21), sensor=_cabi.RK_SENSOR_STREAM, frames=fr)
    assert_same(tr[::30], G["stream_trace"], "golden stream trace")
    assert_same(st, G["stream_state"], "golden stream state")
    st0 = layout.aos_to_soa(wl.random_states(64, seed=9))
    st, tr = gpu_run(wl.plant_inputs(64, 24, seed=9, seg_len=6, yaw_period=3), state=st0)
    assert_same(tr[::6], G["rand_trace"], "golden random-state trace")
    assert_same(st, G["rand_state"], "golden random-state state")


def test_stream_mode_bit_exact():
    n, steps = 96, 700
    inp = wl.plant_inputs(n, steps, seed=12)
    fr = streams.vehicle_frames(n, steps, seed=12)
    st, tr = gpu_run(inp, sensor=_cabi.RK_SENSOR_STREAM, frames=fr)
    pst, ptr = port_run(inp, sensor=_cabi.RK_SENSOR_STREAM, frames=fr, nthreads=8)
    assert_same(tr, ptr, "stream trace")
    assert_same(st, pst, "stream state")


def test_stream_mode_adversarial_frames():
    """Frames with arbitrary 16-bit fields: exercises the int16 wrap / +-4096 unwrap edges of
    rx_callback (VD_motor_if_m2006.cpp:40-69) far outside what a real C610 sends."""
    n, steps = 128, 64
    rng = np.random.default_rng(5)
    fr = rng.integers(0, 1 << 63, size=(steps, 4, n), dtype=np.int64).view(np.uint64)
    edge = np.array([0, 4096, 4097, 8191, 8192, 0x7FFF, 0x8000, 0xFFFF, 4095, 12288], dtype=np.uint64)
    ang = edge[rng.integers(0, len(edge), size=(steps, 4, n))]
    be = ((ang >> np.uint64(8)) & np.uint64(0xFF)) | ((ang & np.uint64(0xFF)) << np.uint64(8))
    fr = np.where(rng.random((steps, 4, n)) < 0.5, (fr & ~np.uint64(0xFFFF)) | be, fr)
    # keep |rpm| small enough that u*1000 stays inside int16 (C++ UB beyond; SURVEY App. C)
    fr = fr & ~np.uint64(0x00000000FFFF0000)
    inp = dict(n=n, steps=steps)
    st, tr = gpu_run(inp, sensor=_cabi.RK_SENSOR_STREAM, frames=fr)
    pst, ptr = port_run(inp, sensor=_cabi.RK_SENSOR_STREAM, frames=fr)
    assert_same(tr, ptr, "adversarial stream trace")
    assert_same(st, pst, "adversarial stream state")


def test_random_initial_states_and_hold_mode():
    n = 2048
    st0 = layout.aos_to_soa(wl.random_states(n, seed=3))
    inp = wl.plant_inputs(n, 40, seed=5, seg_len=8, yaw_period=4)
    for sensor in (_cabi.RK_SENSOR_PLANT, _cabi.RK_SENSOR_HOLD):
        st, tr = gpu_run(inp, sensor=sensor, state=st0)
        pst, ptr = port_run(inp, sensor=sensor, state=st0, nthreads=8)
        assert_same(tr, ptr, f"random-state trace mode {sensor}")
        assert_same(st, pst, f"random-state state mode {sensor}")


def test_power_off_resets():
    """isPowerOn false: interpolators and controllers reset each tick, current 0
    (VD_vehicle_controller.cpp:81-98).  No command table -> power stays off."""
    n = 64
    aos = wl.random_states(n, seed=8)
    aos[:, layout.VS_FLAGS] = 0
    st0 = layout.aos_to_soa(aos)
    inp = dict(n=n, steps=5)
    st, tr = gpu_run(inp, state=st0)
    pst, ptr = port_run(inp, state=st0)
    assert_same(tr, ptr, "power-off trace")
    assert_same(st, pst, "power-off state")
    assert np.all(tr[1:, 9:13, :] == 0)


def test_resume_chunked_equals_one_launch():
    inp = wl.plant_inputs(300, 1000, seed=44, seg_len=125, yaw_period=10)
    st1, tr1 = gpu_run(inp)
    st2, tr2 = gpu_run(inp, chunks=4)
    # microsecond ids restart per launch (dead telemetry word); mask it out of the compare
    a1, a2 = layout.soa_to_aos(st1, 300, layout.VS_WORDS), layout.soa_to_aos(st2, 300, layout.VS_WORDS)
    for w in range(4):
        a1[:, layout.VS_MOTOR0 + 8 * w + layout.VM_USEC] &= 0xFFFF0000
        a2[:, layout.VS_MOTOR0 + 8 * w + layout.VM_USEC] &= 0xFFFF0000
    assert_same(tr2, tr1, "chunked trace")
    assert_same(a2, a1, "chunked state")


def test_trace_off_gives_same_state():
    inp = wl.plant_inputs(500, 600, seed=45)
    st1, _ = gpu_run(inp, trace=True)
    st2, _ = gpu_run(inp, trace=False)
    assert_same(st2, st1, "trace-off state")


def test_full_size_c2_sampled_parity_and_slice_invariance():
    """BASELINE.json configs[1]: 2^20 vehicles x 1000 fused ticks.  Size-independent checks:
    (a) a seeded sample of instances equals the oracle run on those instances alone,
    (b) instances are independent: a contiguous slice run as its own batch is identical."""
    n, steps = 1 << 20, 1000
    inp = wl.plant_inputs(n, steps, seed=0x5EED)
    st, _ = gpu_run(inp, trace=False)
    aos = layout.soa_to_aos(st, n, layout.VS_WORDS)
    rng = np.random.default_rng(1)
    idx = np.unique(np.concatenate([[0, 1, n - 1, n - 2, 127, 128], rng.integers(0, n, 90)]))
    sub = dict(n=len(idx), steps=steps, cmd=np.ascontiguousarray(inp["cmd"][:, idx]), seg_len=inp["seg_len"],
               yaw=np.ascontiguousarray(inp["yaw"][:, idx]), yaw_period=inp["yaw_period"])
    pst, _ = port_run(sub, trace=False, nthreads=8)
    assert_same(aos[idx], layout.soa_to_aos(pst, len(idx), layout.VS_WORDS), "sampled instances vs port")
    lo, hi = 500_000, 500_000 + 4096 + 17
    sl = dict(n=hi - lo, steps=steps, cmd=np.ascontiguousarray(inp["cmd"][:, lo:hi]), seg_len=inp["seg_len"],
              yaw=np.ascontiguousarray(inp["yaw"][:, lo:hi]), yaw_period=inp["yaw_period"])
    sst, _ = gpu_run(sl, trace=False)
    assert_same(layout.soa_to_aos(sst, hi - lo, layout.VS_WORDS), aos[lo:hi], "slice invariance")
    # physical sanity at full size: saturation respected everywhere, finite positions
    v = layout.vehicle_view(aos)
    assert np.all(np.abs(v["cur_tgt"]) <= 3000)
    assert np.all(np.isfinite(v["pos"]))


def test_bounded_drift_10k_steps():
    """BASELINE.json: bounded-drift check after 10k steps.  Bit-exact state after 10 000
    closed-loop ticks implies zero drift; also check it against the <=1e-5 formal bound."""
    inp = wl.plant_inputs(128, 10000, seed=77)
    st, _ = gpu_run(inp, trace=False)
    pst, _ = port_run(inp, trace=False, nthreads=8)
    a, b = layout.soa_to_aos(st, 128, layout.VS_WORDS), layout.soa_to_aos(pst, 128, layout.VS_WORDS)
    pa, pb = layout.vehicle_view(a)["pos"], layout.vehicle_view(b)["pos"]
    np.testing.assert_allclose(pa, pb, rtol=1e-5, atol=0)
    assert_same(a, b, "10k-step state")


def test_batched_setters_match_oracle():
    import ctypes as C

    n = 257
    aos = wl.random_states(n, seed=12)
    vb = VehicleBatch(n, DEV)
    vb.load_state_aos(aos)
    rng = np.random.default_rng(2)
    v = rng.uniform(-400, 400, (3, n)).astype(np.float32)
    a = rng.uniform(10, 2000, (3, n)).astype(np.float32)
    j = rng.uniform(100, 30000, (3, n)).astype(np.float32)
    vb.set_target_vel(_dev(v), _dev(a), _dev(j))
    fr = streams.vehicle_frames(n, 1, seed=3)[0]
    us = rng.integers(0, 0x7FFF, n).astype(np.int16)
    for w in range(4):
        vb.motor_rx(w, _dev(fr[w], np.int64), _dev(us))
    vb.set_power()
    torch.cuda.synchronize()
    got = vb.state_aos()
    p = rk.default_params()
    lib = ol.port()
    F3 = C.c_float * 3
    exp = aos.copy()
    for i in range(n):
        row = np.ascontiguousarray(exp[i])
        ptr = row.ctypes.data_as(C.c_void_p)
        lib.orc_vdt_set_target(C.byref(p), ptr, F3(*v[:, i]), F3(*a[:, i]), F3(*j[:, i]))
        for w in range(4):
            lib.orc_vdt_rx(C.byref(p), ptr, w, fr[w, i].tobytes(), int(us[i]))
        row[layout.VS_FLAGS] |= 1
        exp[i] = row
    assert_same(got, exp, "batched setters")


def test_single_instance_handle_c1_prefix():
    """The drop-in handle (rk_vdt_t): drive it exactly as the firmware drives its statics --
    set_now_yaw_world + rx_callback x4 + update per tick -- and compare with the oracle."""
    import ctypes as C

    steps = 300
    inp = wl.c1_inputs()
    _, ptr = port_run(dict(inp, steps=steps))
    veh = Vehicle()
    rpm, ang = [0] * 4, [0] * 4
    for t in range(steps):
        if t == 0:
            veh.start()
            veh.set_target_vel((200.0, 100.0, 1.0), (1000.0, 1000.0, 30.0), (10000.0, 10000.0, 300.0))
        veh.set_now_yaw_world(float(inp["yaw"][t // 10, 0]))
        cur = veh.get_rawCurr_tgt()
        for k in range(4):
            c = cur[k]
            rpm[k] += (c * 4 - rpm[k]) >> 4
            q = abs(rpm[k] * 8192) // 60000
            ang[k] = (ang[k] + (q if rpm[k] >= 0 else -q)) & 8191
            fr = bytes([(ang[k] >> 8) & 255, ang[k] & 255, (rpm[k] >> 8) & 255, rpm[k] & 255, (c >> 8) & 255, c & 255, 0, 0])
            veh.rx_callback(k, fr, ((t + 1) * 1000) & 0x7FFF)
        veh.update()
        if t % 25 == 0 or t == steps - 1:
            row = ptr[t, :, 0]
            np.testing.assert_array_equal(veh.get_vehicle_pos_m_latest().view(np.uint32), row[0:3])
            np.testing.assert_array_equal(veh.get_vehicle_vel_mmps_latest().view(np.uint32), row[3:6])
            np.testing.assert_array_equal(veh.get_vehicle_vel_tgt_mmps_latest().view(np.uint32), row[6:9])
            assert veh.get_rawCurr_tgt() == list(row[9:13].view(np.int32))
    veh.close()


def test_cost_epilogue():
    n = 100
    inp = wl.plant_inputs(n, 500, seed=6)
    goal = np.random.default_rng(0).uniform(-1, 1, (n, 2)).astype(np.float32)
    vb = VehicleBatch(n, DEV)
    cost = torch.zeros(n, dtype=torch.float32, device=DEV)
    cmd = _dev(inp["cmd"], np.int32).reshape(-1, n, 4)
    vb.rollout(500, cmd=cmd, seg_len=inp["seg_len"], yaw=_dev(inp["yaw"]), yaw_period=inp["yaw_period"],
               goal=_dev(goal), cost=cost)
    torch.cuda.synchronize()
    pos = layout.vehicle_view(vb.state_aos())["pos"]
    dx, dy = pos[:, 0] - goal[:, 0], pos[:, 1] - goal[:, 1]
    np.testing.assert_array_equal(cost.cpu().numpy(), dx * dx + dy * dy)


# ---- the issue-optimised kernel vs the transcription kernel --------------------------------
def test_fast_path_is_proven_and_used_for_firmware_params():
    import ctypes as C

    lib = rk.load()
    assert lib.rk_vdt_fast_path_proven(C.byref(rk.default_params())) == 1


def test_fast_kernel_equals_transcription_kernel():
    lib = rk.load()
    n = 4096 + 33
    st0 = layout.aos_to_soa(wl.random_states(n, seed=21))
    # half the instances start from the power-on state (fast path from tick 0), half from
    # random states (many of which are outside the fast path's domain -> per-thread fallback)
    aos = layout.soa_to_aos(st0, n, layout.VS_WORDS)
    aos[::2] = 0
    st0 = layout.aos_to_soa(aos)
    inp = wl.plant_inputs(n, 700, seed=22, seg_len=100, yaw_period=10)
    fast_st, fast_tr = gpu_run(inp, state=st0)
    lib.rk_set_option(_cabi.RK_OPT_FORCE_TRANSCRIPTION, 1)
    try:
        ref_st, ref_tr = gpu_run(inp, state=st0)
    finally:
        lib.rk_set_option(_cabi.RK_OPT_FORCE_TRANSCRIPTION, 0)
    assert_same(fast_tr, ref_tr, "fast vs transcription trace")
    assert_same(fast_st, ref_st, "fast vs transcription state")
    pst, ptr = port_run(inp, state=st0, nthreads=8)
    assert_same(fast_tr, ptr, "fast trace vs port")
    assert_same(fast_st, pst, "fast state vs port")


def test_float_encoder_step_zero_signs_and_crawl_speeds():
    """The packed tick forms the encoder step in float (trunc(rpm * C)): a wheel crawling backwards at less than one
    count per tick gives -0.0 where the integer path gives +0.0.  That only matters for a position word that is itself
    -0.0, which the fast path refuses (transcription instead).  Crawl commands (a few mm/s, both signs) from blocks whose
    position words are +0.0, -0.0 and tiny values of both signs, traced and untraced, against the port bit for bit."""
    n, steps = 2048, 300
    rng = np.random.default_rng(5)
    aos = np.zeros((n, layout.VS_WORDS), dtype=np.uint32)
    pos = np.zeros((n, 2), dtype=np.float32)
    kind = np.arange(n) % 4
    pos[kind == 1] = -0.0
    pos[kind == 2] = rng.uniform(-1e-30, 1e-30, ((kind == 2).sum(), 2)).astype(np.float32)
    pos[kind == 3, 0] = -0.0  # mixed: x = -0.0, y = +0.0
    aos[:, layout.VS_POS_X] = pos[:, 0].copy().view(np.uint32)
    aos[:, layout.VS_POS_Y] = pos[:, 1].copy().view(np.uint32)
    st0 = layout.aos_to_soa(aos)
    cmd = np.zeros((3, n), dtype=np.dtype([("vx", "<f4"), ("vy", "<f4"), ("vth", "<f4"), ("kind", "<i4")]))
    for sgm in range(3):
        cmd["vx"][sgm] = rng.uniform(-6.0, 6.0, n).astype(np.float32)
        cmd["vy"][sgm] = rng.uniform(-6.0, 6.0, n).astype(np.float32)
        cmd["vth"][sgm] = rng.uniform(-0.05, 0.05, n).astype(np.float32)
        cmd["kind"][sgm] = _cabi.RK_CMD_MOVE
    inp = dict(n=n, steps=steps, cmd=cmd, seg_len=100)
    pst, ptr = port_run(inp, state=st0, nthreads=8)
    gst, gtr = gpu_run(inp, state=st0)
    assert_same(gtr, ptr, "crawl trace vs port")
    assert_same(gst, pst, "crawl state vs port")
    ust, _ = gpu_run(inp, state=st0, trace=False)
    assert_same(ust, pst, "crawl state (untraced) vs port")


def test_packed_and_scalar_fast_ticks_agree():
    """The fast kernel has two bit-identical forms: packed FADD2/FFMA2 (default) and scalar
    (RK_OPT_FAST_PACKED = 0).  Every other test here runs the packed one; this one runs both."""
    lib = rk.load()
    n = 2048 + 5
    inp = wl.plant_inputs(n, 1000, seed=31, seg_len=125, yaw_period=10)
    packed_st, packed_tr = gpu_run(inp)
    lib.rk_set_option(_cabi.RK_OPT_FAST_PACKED, 0)
    try:
        scalar_st, scalar_tr = gpu_run(inp)
    finally:
        lib.rk_set_option(_cabi.RK_OPT_FAST_PACKED, 1)
    assert_same(packed_tr, scalar_tr, "packed vs scalar trace")
    assert_same(packed_st, scalar_st, "packed vs scalar state")
    pst, ptr = port_run(inp, nthreads=8)
    assert_same(packed_tr, ptr, "packed trace vs port")
    assert_same(packed_st, pst, "packed state vs port")


def test_non_finite_and_extreme_commands_fall_back_exactly():
    """Commands outside the fast path's domain (huge / tiny / NaN / Inf targets) must take the
    transcription path per thread and still match the oracle bit for bit."""
    n, steps = 256, 400
    inp = wl.plant_inputs(n, steps, seed=23, seg_len=50, yaw_period=10)
    cmd = inp["cmd"].copy()
    rng = np.random.default_rng(3)
    weird = np.array([1e-38, -1e-40, 3e38, -3e38, np.inf, -np.inf, np.nan, 1e12, -0.0, 1e-30], dtype=np.float32)
    for s in range(cmd.shape[0]):
        idx = rng.integers(0, n, 24)
        cmd["vx"][s, idx] = weird[rng.integers(0, len(weird), 24)]
        idx = rng.integers(0, n, 24)
        cmd["vth"][s, idx] = weird[rng.integers(0, len(weird), 24)]
    inp["cmd"] = cmd
    yaw = inp["yaw"].copy()
    yaw[3, :8] = [np.nan, np.inf, -np.inf, 1e30, -1e30, 1e-40, -0.0, 1e9]
    inp["yaw"] = yaw
    st, tr = gpu_run(inp)
    pst, ptr = port_run(inp, nthreads=8)
    # NaN payload propagation is not specified identically on x86 and sm_100: compare NaNs as NaNs
    def canon(a):
        a = a.copy()
        f = a.view(np.float32)
        a[np.isnan(f)] = 0x7FC00000
        return a
    ok_cols = np.ones(n, dtype=bool)
    # instances that ever saw a non-finite command/yaw: int16 conversion of NaN/Inf is C++ UB
    bad = ~np.isfinite(cmd["vx"]).all(0) | ~np.isfinite(cmd["vth"]).all(0)
    bad[:8] |= ~np.isfinite(yaw[3, :8])
    ok_cols &= ~bad
    assert ok_cols.sum() > n // 2
    assert_same(canon(tr[:, :, ok_cols]), canon(ptr[:, :, ok_cols]), "extreme-command trace")
    a, b = layout.soa_to_aos(st, n, layout.VS_WORDS), layout.soa_to_aos(pst, n, layout.VS_WORDS)
    assert_same(canon(a[ok_cols]), canon(b[ok_cols]), "extreme-command state")


def test_other_wirings_use_transcription_and_match():
    """Non-firmware parameters (different wheel directions / geometry / gains) are served by
    the transcription kernel (or the fast one if its proofs hold) -- always exact."""
    import ctypes as C

    for variant in range(3):
        p = rk.default_params()
        if variant == 0:
            p.motor_dir[:] = [1, -1, 1, -1]
        elif variant == 1:
            p.wheel_radius_mm, p.wheel_l_mm = 40.0, 15.5
            p.kd, p.kp = 0.001, 0.03
        else:
            p.raw_curr_lim = 10000
            p.i_limit = 0.25
        n, steps = 200, 500
        inp = wl.plant_inputs(n, steps, seed=30 + variant)
        vb = VehicleBatch(n, DEV, params=p)
        cmd = _dev(inp["cmd"], np.int32).reshape(-1, n, 4)
        tr = torch.zeros((steps, 16, n), dtype=torch.int32, device=DEV)
        vb.rollout(steps, cmd=cmd, seg_len=inp["seg_len"], yaw=_dev(inp["yaw"]), yaw_period=inp["yaw_period"], trace=tr)
        torch.cuda.synchronize()
        st = np.zeros(layout.VS_WORDS * n, dtype=np.uint32)
        ro = ol.HostRollout(n, steps, _cabi.RK_SENSOR_PLANT, inp["cmd"], inp["seg_len"], inp["yaw"], inp["yaw_period"], trace=True)
        ol.run_port(st, n, ro, params=p, nthreads=8)
        assert_same(tr.cpu().numpy().view(np.uint32), ro.trace, f"variant {variant} trace")
        assert_same(vb.state.cpu().numpy().view(np.uint32), st, f"variant {variant} state")


def test_yaw_register_input_equals_float_yaw_and_port():
    """rk_vdt_rollout_t::d_yaw_reg (the WT901C Yaw register, int16) on both kernels == the float stream the IMU would
    have produced == the port."""
    lib = rk.load()
    n, steps = 1500, 1000
    inp = wl.plant_inputs(n, steps, seed=41)
    reg = streams.vehicle_yaw_reg(n, steps // 10, seed=41)
    st_r, tr_r = gpu_run(dict(inp, yaw=reg))
    st_f, tr_f = gpu_run(dict(inp, yaw=streams.yaw_reg_to_rad(reg)))
    assert_same(tr_r, tr_f, "register yaw vs float yaw trace")
    assert_same(st_r, st_f, "register yaw vs float yaw state")
    lib.rk_set_option(_cabi.RK_OPT_FORCE_TRANSCRIPTION, 1)
    try:
        st_t, tr_t = gpu_run(dict(inp, yaw=reg))
    finally:
        lib.rk_set_option(_cabi.RK_OPT_FORCE_TRANSCRIPTION, 0)
    assert_same(tr_r, tr_t, "register yaw: fast vs transcription")
    pst, ptr = port_run(dict(inp, yaw=reg))
    assert_same(tr_r, ptr, "register yaw vs port trace")
    assert_same(st_r, pst, "register yaw vs port state")


def test_stream_fast_tick_equals_transcription_and_port():
    """RK_SENSOR_STREAM runs on the packed fast tick (vdt_rollout_stream_fast_kernel): same bits as the transcription
    kernel and the port -- on realistic recorded traffic with the VDT task layer active, on adversarial angle fields
    with the vehicles powered (so the fast path is really taken), and resumed over several launches."""
    lib = rk.load()
    from test_vdt_task_cpu import task_inputs

    n, steps = 1100, 1000
    rng = np.random.default_rng(8)
    fr_real = streams.vehicle_frames(n, steps, seed=31)
    fr_adv = rng.integers(0, 1 << 63, size=(steps, 4, n), dtype=np.int64).view(np.uint64) & ~np.uint64(0x00000000FFFF0000)
    cases = (("plain", wl.plant_inputs(n, steps, seed=31), fr_real), ("task", dict(task_inputs(n, steps, 32, seg_len=50), task_period=10), fr_real),
             ("adversarial", wl.plant_inputs(n, steps, seed=33), fr_adv))
    for name, inp, fr in cases:
        st, tr = gpu_run(inp, sensor=_cabi.RK_SENSOR_STREAM, frames=fr)
        lib.rk_set_option(_cabi.RK_OPT_FORCE_TRANSCRIPTION, 1)
        try:
            st_t, tr_t = gpu_run(inp, sensor=_cabi.RK_SENSOR_STREAM, frames=fr)
        finally:
            lib.rk_set_option(_cabi.RK_OPT_FORCE_TRANSCRIPTION, 0)
        assert_same(tr, tr_t, name + ": stream fast vs transcription trace")
        assert_same(st, st_t, name + ": stream fast vs transcription state")
        if name != "task":
            pst, ptr = port_run(inp, sensor=_cabi.RK_SENSOR_STREAM, frames=fr, nthreads=8)
            assert_same(tr, ptr, name + ": stream fast vs port trace")
            assert_same(st, pst, name + ": stream fast vs port state")
        if name == "plain":
            st5, _ = gpu_run(inp, sensor=_cabi.RK_SENSOR_STREAM, frames=fr, trace=False, chunks=4)
            a1, a5 = layout.soa_to_aos(st, n, layout.VS_WORDS), layout.soa_to_aos(st5, n, layout.VS_WORDS)
            for w in range(4):  # microsecond ids restart per launch (dead telemetry word)
                a1[:, layout.VS_MOTOR0 + 8 * w + layout.VM_USEC] &= 0xFFFF0000
                a5[:, layout.VS_MOTOR0 + 8 * w + layout.VM_USEC] &= 0xFFFF0000
            assert_same(a1, a5, "stream: one launch vs four")


def test_current_conversion_overflow_matches_x86():
    """(int16_t)(A * 1000.0f) beyond +-2^31: cvttss2si gives 0x80000000 (low 16 bits 0), a saturating F2I would give
    -1 for the positive side.  Gains that wrap the int16 (kp = 50: stays on the fast tick) and gains large enough to
    leave the int32 (kp = 4e3, 2e5; kff large with a wide FF limit) must
    still match the x86 port bit for bit -- the fast path's chunk bound (fast_u_bounded) sends such chunks to the
    transcription tick, whose conversion is f2i_x86."""
    for variant, (kp, kff, fflim) in enumerate([(50.0, 0.0075, 1.0), (4.0e3, 0.0075, 1.0), (2.0e5, 0.0075, 1.0), (0.02, 5.0e4, 1.0e9)]):
        p = rk.default_params()
        p.kp, p.kff, p.ff_limit = kp, kff, fflim
        n, steps = 256, 300
        inp = wl.plant_inputs(n, steps, seed=60 + variant, seg_len=50)
        vb = VehicleBatch(n, DEV, params=p)
        cmd = _dev(inp["cmd"], np.int32).reshape(-1, n, 4)
        tr = torch.zeros((steps, 16, n), dtype=torch.int32, device=DEV)
        vb.rollout(steps, cmd=cmd, seg_len=inp["seg_len"], yaw=_dev(inp["yaw"]), yaw_period=inp["yaw_period"], trace=tr)
        torch.cuda.synchronize()
        st = np.zeros(layout.VS_WORDS * n, dtype=np.uint32)
        ro = ol.HostRollout(n, steps, _cabi.RK_SENSOR_PLANT, inp["cmd"], inp["seg_len"], inp["yaw"], inp["yaw_period"], trace=True)
        ol.run_port(st, n, ro, params=p, nthreads=8)
        gtr = tr.cpu().numpy().view(np.uint32)
        assert_same(gtr, ro.trace, f"overflow variant {variant} trace")
        assert_same(vb.state.cpu().numpy().view(np.uint32), st, f"overflow variant {variant} state")


def test_yaw_from_imu_register_snapshots():
    """rk_vdt_rollout_t::d_imu_regs: the vehicle forms the yaw from the IMU's own register snapshots (Yaw register
    scaled as updateData() does, held over updates without a quaternion frame, Data.angle[2] at launch if update 0
    has none) == the float stream the IMU port emits for the same samples; fast and transcription kernels."""
    lib = rk.load()
    n, steps, slow = 777, 500, 10
    n_slow = steps // slow
    inp = wl.plant_inputs(n, steps, seed=71)
    regs, have = streams.imu_samples(n, n_slow + 1, seed=71, drop_every=5)
    have[1, : n // 2] = 0  # update 0 without a quaternion frame: the launch-time Data page is held
    ist = np.zeros(layout.IS_WORDS * n, dtype=np.uint32)
    ol.imu_port(ist, n, regs[:1], None, do_init=True)
    yaw0 = layout.soa_to_aos(ist, n, layout.IS_WORDS)[:, layout.IS_DATA + 11].copy().view(np.float32)
    out = ol.imu_port(ist, n, np.ascontiguousarray(regs[1:]), np.ascontiguousarray(have[1:]), want_out=True)
    yaw = (np.ascontiguousarray(out[:, 2, :, 3]).view(np.float32) * streams.DEG2RAD).astype(np.float32)
    pst, ptr = port_run(dict(inp, yaw=yaw, yaw_period=slow), nthreads=8)

    def run():
        vb = VehicleBatch(n, DEV)
        cmd = _dev(inp["cmd"], np.int32).reshape(-1, n, 4)
        tr = torch.zeros((steps, 16, n), dtype=torch.int32, device=DEV)
        a = vb.make_args(steps, cmd=cmd, seg_len=inp["seg_len"], trace=tr)
        regs_d, have_d, yaw0_d = _dev(streams.imu_cells(regs[1:])), _dev(have[1:]), _dev(yaw0)
        a.d_imu_regs, a.d_imu_have_quat, a.d_imu_yaw0_deg = regs_d.data_ptr(), have_d.data_ptr(), yaw0_d.data_ptr()
        a.n_yaw, a.yaw_period = n_slow, slow
        vb.rollout_args(a)
        torch.cuda.synchronize()
        return vb.state.cpu().numpy().view(np.uint32), tr.cpu().numpy().view(np.uint32)

    st, tr = run()
    assert_same(tr, ptr, "IMU-register yaw vs port trace")
    assert_same(st, pst, "IMU-register yaw vs port state")
    lib.rk_set_option(_cabi.RK_OPT_FORCE_TRANSCRIPTION, 1)
    try:
        st_t, tr_t = run()
    finally:
        lib.rk_set_option(_cabi.RK_OPT_FORCE_TRANSCRIPTION, 0)
    assert_same(tr_t, ptr, "IMU-register yaw, transcription kernel vs port trace")
    assert_same(st_t, pst, "IMU-register yaw, transcription kernel vs port state")


def test_c610_tx_frame_words_and_batch_entry():
    """SURVEY 8f-3, vehicle tx side: the C610 current frame CAN_CTRL::tx_routine() builds (VD_can_controller.hpp:43-55) --
    trace words 14-15 equal the port's (pinned against the reference's own routine in tests/test_vdt_task_cpu.py), they
    are the four currents big-endian, and rk_vdt_tx_frames / the handle's tx_routine() give the same bytes from the state."""
    n, steps = 500, 300
    inp = wl.plant_inputs(n, steps, seed=88)
    st, tr = gpu_run(inp)
    pst, ptr = port_run(inp, nthreads=8)
    assert_same(tr[:, 14:16, :], ptr[:, 14:16, :], "C610 tx frame words")
    cur = tr[:, 9:13, :].view(np.int32)
    by = np.ascontiguousarray(tr[:, 14:16, :].transpose(0, 2, 1)).view(np.uint8).reshape(steps, n, 8)
    for k in range(4):
        wire = (by[:, :, 2 * k].astype(np.int32) << 8 | by[:, :, 2 * k + 1]).astype(np.uint16).view(np.int16)
        np.testing.assert_array_equal(wire, cur[:, k, :].astype(np.int16))
    assert np.abs(cur).max() > 256  # both bytes are exercised
    vb = VehicleBatch(n, DEV)
    vb.load_state_soa(st)
    fr = vb.tx_frames()
    torch.cuda.synchronize()
    np.testing.assert_array_equal(fr.cpu().numpy().view(np.uint8).reshape(n, 8), by[-1])
    from roboken_fmskf_robot_controller_b200.vehicle import Vehicle

    v = Vehicle()
    v.set_state(layout.soa_to_aos(st, n, layout.VS_WORDS)[7])
    assert v.tx_routine() == bytes(by[-1, 7])


def test_reset_state_flag_equals_a_zeroed_block():
    """rk_vdt_rollout_t::reset_state: the rollout starts from the power-on block whatever d_state holds -- fast and
    transcription kernels, plant and stream sensors."""
    lib = rk.load()
    n, steps = 700, 300
    inp = wl.plant_inputs(n, steps, seed=55)
    st0, tr0 = gpu_run(inp)
    dirty = layout.aos_to_soa(wl.random_states(n, seed=4))
    fr = streams.vehicle_frames(n, steps, seed=55)
    for force in (0, 1):
        lib.rk_set_option(_cabi.RK_OPT_FORCE_TRANSCRIPTION, force)
        try:
            for sensor, frames in ((_cabi.RK_SENSOR_PLANT, None), (_cabi.RK_SENSOR_STREAM, fr)):
                ref_st, ref_tr = gpu_run(inp, sensor=sensor, frames=frames)
                vb = VehicleBatch(n, DEV)
                vb.load_state_soa(dirty)
                tr = torch.zeros((steps, 16, n), dtype=torch.int32, device=DEV)
                vb.rollout(steps, sensor_mode=sensor, cmd=_dev(inp["cmd"], np.int32).reshape(-1, n, 4), seg_len=inp["seg_len"],
                           yaw=_dev(inp["yaw"]), yaw_period=inp["yaw_period"], frames=_dev(frames, np.int64), trace=tr, reset_state=True)
                torch.cuda.synchronize()
                assert_same(tr.cpu().numpy().view(np.uint32), ref_tr, f"reset_state trace (force={force}, sensor={sensor})")
                assert_same(vb.state.cpu().numpy().view(np.uint32), ref_st, f"reset_state state (force={force}, sensor={sensor})")
        finally:
            lib.rk_set_option(_cabi.RK_OPT_FORCE_TRANSCRIPTION, 0)
    assert_same(st0, gpu_run(inp)[0], "sanity")
