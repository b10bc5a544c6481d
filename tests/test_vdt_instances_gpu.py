"""GPU: every compiled instantiation of the vehicle rollout kernels, bit for bit against the port.

Each row of vdt_instances.MATRIX (RK_OPT_FAST_OCCUPANCY x _FAST_PACKED x _FAST_FFSAT x kd x ff_limit, and
RK_OPT_FORCE_TRANSCRIPTION) runs the same battery: rk_vdt_rollout under RK_SENSOR_PLANT (traced and untraced, reset_state,
the cost epilogue, task_period > 0, a resume in chunks, one segment longer than a fast-kernel chunk, start states the
fast path refuses, crawl speeds from +-0 positions, and each yaw source), RK_SENSOR_STREAM, RK_SENSOR_HOLD, and the three
planner entries with discs and a path.  Each launch runs under torch.profiler and must launch exactly the instantiation
vdt_instances.expected_kernel names; the last test checks that the matrix launched every compiled instantiation.

The port's result does not depend on the options, so it is computed once per (params, workload) and every row is
compared against it.  The options are process-wide: the fixture restores their defaults whatever a case does.
"""
import ctypes as C

import numpy as np
import pytest
import torch
from torch.profiler import ProfilerActivity, profile

import oracle_lib as ol
import plan_fleet_ref as pfr
import plan_obst_ref as por
import plan_ref as pr
import vdt_instances as vi
import workloads as wl
import roboken_fmskf_robot_controller_b200 as rk
from roboken_fmskf_robot_controller_b200 import _cabi, layout, streams
from roboken_fmskf_robot_controller_b200.vehicle import VehicleBatch
from test_plan_cpu import _nominal
from test_plan_fleet_gpu import _moving_discs, _moving_rollout
from test_plan_gpu import _plan_rollout
from test_plan_obst_gpu import N_SEG, R, S, SEG_LEN, W, _discs, _obst_rollout
from test_vdt_task_cpu import task_inputs
from test_vehicle_gpu import assert_same

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
OPTIONS = {  # row key -> (option, default)
    "force_transcription": (_cabi.RK_OPT_FORCE_TRANSCRIPTION, 0),
    "packed": (_cabi.RK_OPT_FAST_PACKED, 1),
    "occupancy": (_cabi.RK_OPT_FAST_OCCUPANCY, 4),
    "ffsat": (_cabi.RK_OPT_FAST_FFSAT, 0),
}
WAVE = 148 * 4 * 128  # resident threads of the fast kernel at occupancy 4 on a B200
LAUNCHED = {}  # instantiation -> the first row that launched it
_PORT = {}
_WORK = {}


@pytest.fixture
def options():
    lib = rk.load()

    def apply(row):
        for key, (opt, _) in OPTIONS.items():
            _cabi.check(lib.rk_set_option(opt, row[key]))

    try:
        yield apply
    finally:
        for opt, default in OPTIONS.values():
            _cabi.check(lib.rk_set_option(opt, default))


def _params(row):
    p = rk.default_params()
    p.kd, p.ff_limit = row["kd"], row["ff_limit"]
    assert rk.load().rk_vdt_fast_path_proven(C.byref(p)) == 1, "the matrix's params must be on the fast path"
    return p


def _u32(t):
    return t.cpu().numpy().view(np.uint32)


def _dev(a, dtype=None):
    return None if a is None else torch.from_numpy(np.ascontiguousarray(a).view(dtype) if dtype else np.ascontiguousarray(a)).to(DEV)


def _mask_usec(st, n):
    """The microsecond ids restart with every launch (a dead telemetry word): clear them for a chunked compare."""
    a = layout.soa_to_aos(st, n, layout.VS_WORDS)
    for w in range(4):
        a[:, layout.VS_MOTOR0 + 8 * w + layout.VM_USEC] &= 0xFFFF0000
    return a


def _work(name, make):
    if name not in _WORK:
        _WORK[name] = make()
    return _WORK[name]


def _port(row, name, make):
    """make() -> the port's result for this row's params, cached per (kd, ff_limit, workload)."""
    key = (row["kd"], row["ff_limit"], name)
    if key not in _PORT:
        _PORT[key] = make()
    return _PORT[key]


def port_rollout(p, inp, sensor=_cabi.RK_SENSOR_PLANT, state=None, frames=None, trace=True, goal=None):
    n = inp["n"]
    st = np.zeros(layout.VS_WORDS * n, dtype=np.uint32) if state is None else state.copy()
    ro = ol.HostRollout(n, inp["steps"], sensor, inp.get("cmd"), inp.get("seg_len", 0), inp.get("yaw"), inp.get("yaw_period", 0),
                        frames=frames, trace=trace, goal=goal, task_period=inp.get("task_period", 0))
    ol.run_port(st, n, ro, params=p, nthreads=8)
    return st, ro.trace, ro.cost


# ---- workloads ------------------------------------------------------------------------------------------------------
def _main():
    """4096 + 33 vehicles, half from the power-on block (fast path from tick 0) and half from random states (many
    outside the fast path's domain: the per-thread fallback), with goals for the cost epilogue."""
    n = 4096 + 33
    aos = wl.random_states(n, seed=21)
    aos[::2] = 0
    inp = wl.plant_inputs(n, 600, seed=22, seg_len=100, yaw_period=10)
    goal = np.random.default_rng(0).uniform(-1, 1, (n, 2)).astype(np.float32)
    return inp, layout.aos_to_soa(aos), goal, layout.aos_to_soa(wl.random_states(n, seed=4))


def _crawl():
    """test_vehicle_gpu.test_float_encoder_step_zero_signs_and_crawl_speeds: crawl commands from +-0 / tiny positions."""
    n, steps = 2048, 300
    rng = np.random.default_rng(5)
    aos = np.zeros((n, layout.VS_WORDS), dtype=np.uint32)
    pos = np.zeros((n, 2), dtype=np.float32)
    kind = np.arange(n) % 4
    pos[kind == 1] = -0.0
    pos[kind == 2] = rng.uniform(-1e-30, 1e-30, ((kind == 2).sum(), 2)).astype(np.float32)
    pos[kind == 3, 0] = -0.0
    aos[:, layout.VS_POS_X] = pos[:, 0].copy().view(np.uint32)
    aos[:, layout.VS_POS_Y] = pos[:, 1].copy().view(np.uint32)
    cmd = np.zeros((3, n), dtype=wl.CMD_DT)
    for sgm in range(3):
        cmd["vx"][sgm] = rng.uniform(-6.0, 6.0, n).astype(np.float32)
        cmd["vy"][sgm] = rng.uniform(-6.0, 6.0, n).astype(np.float32)
        cmd["vth"][sgm] = rng.uniform(-0.05, 0.05, n).astype(np.float32)
        cmd["kind"][sgm] = _cabi.RK_CMD_MOVE
    return dict(n=n, steps=steps, cmd=cmd, seg_len=100), layout.aos_to_soa(aos)


def _imu():
    """test_vehicle_gpu.test_yaw_from_imu_register_snapshots: the IMU's register snapshots, and the float yaw the IMU
    port emits for them."""
    n, steps, slow = 777, 500, 10
    n_slow = steps // slow
    inp = wl.plant_inputs(n, steps, seed=71)
    del inp["yaw"], inp["yaw_period"]
    regs, have = streams.imu_samples(n, n_slow + 1, seed=71, drop_every=5)
    have[1, : n // 2] = 0  # update 0 without a quaternion frame: the launch-time Data page is held
    ist = np.zeros(layout.IS_WORDS * n, dtype=np.uint32)
    ol.imu_port(ist, n, regs[:1], None, do_init=True)
    yaw0 = layout.soa_to_aos(ist, n, layout.IS_WORDS)[:, layout.IS_DATA + 11].copy().view(np.float32)
    out = ol.imu_port(ist, n, np.ascontiguousarray(regs[1:]), np.ascontiguousarray(have[1:]), want_out=True)
    yaw = (np.ascontiguousarray(out[:, 2, :, 3]).view(np.float32) * streams.DEG2RAD).astype(np.float32)
    return inp, (streams.imu_cells(regs[1:]), np.ascontiguousarray(have[1:]), yaw0, n_slow, slow), yaw


def _stream():
    """The traffic of test_vehicle_gpu.test_stream_fast_tick_equals_transcription_and_port: recorded-like frames and
    adversarial angle fields."""
    n, steps = 1100, 400
    fr_adv = np.random.default_rng(8).integers(0, 1 << 63, size=(steps, 4, n), dtype=np.int64).view(np.uint64) & ~np.uint64(0x00000000FFFF0000)
    return {"plain": (wl.plant_inputs(n, steps, seed=31), streams.vehicle_frames(n, steps, seed=31)),
            "adversarial": (wl.plant_inputs(n, steps, seed=33), fr_adv)}


def _wave():
    """More than two waves of the fast kernel at either occupancy."""
    return wl.plant_inputs(2 * WAVE + 33, 96, seed=0x5EED, seg_len=32, yaw_period=8)


def _plan():
    """The planner case of test_plan_obst_gpu with source states from the port (not from a rollout under the row's
    options): R robots 300 ticks into stream commands, their candidates, references, static and moving discs."""
    inp = wl.plant_inputs(R, 300, seed=4)
    src, _, _ = port_rollout(rk.default_params(), inp, trace=False)
    ref = np.random.default_rng(1).uniform(-0.5, 0.5, (N_SEG, R, 2)).astype(np.float32)
    cand = streams.plan_commands_v2(_nominal(N_SEG, R), S, seed=5)
    P = 5
    return src, ref, cand, P, _discs(src, 3, seed=2), _moving_discs(src, N_SEG * SEG_LEN // P, 3, seed=12)


# ---- one row --------------------------------------------------------------------------------------------------------
class Battery:
    """Launches under the profiler, each checked against expected_kernel for the row."""

    def __init__(self, row, p):
        self.row, self.p, self.ran = row, p, set()

    def launch(self, entry, trace, reset, fn):
        exp = vi.expected_kernel(entry, trace=trace, reset_state=reset, **self.row)
        torch.cuda.synchronize()
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            out = fn()
            torch.cuda.synchronize()
        got = {t for t in (vi.parse(e.name) for e in prof.events()) if t is not None}
        what = f"{vi.row_id(self.row)}: {entry} trace={trace} reset_state={reset}"
        assert got, f"{what}: the profiler recorded no vehicle rollout kernel"
        assert got == {exp}, f"{what}: launched {sorted(got)}, expected {exp}"
        if exp[0] != "transcription" and self.row["ff_limit"] != 1.0:
            assert not exp[3 if exp[0] == "fast" else 2] & 1, f"{what}: FFSAT applied with ff_limit != 1"
        LAUNCHED.setdefault(exp, vi.row_id(self.row))
        self.ran.add((entry, trace, reset))
        return out

    def rollout(self, inp, entry="plant", state=None, frames=None, trace=False, goal=None, reset=False, chunks=1, imu=None):
        """rk_vdt_rollout, in `chunks` launches; returns (state, trace or None, cost or None) as uint32 / float32."""
        n, steps = inp["n"], inp["steps"]
        vb = VehicleBatch(n, DEV, params=self.p)
        if state is not None:
            vb.load_state_soa(state)
        cmd = _dev(inp.get("cmd"), np.int32)
        cmd = None if cmd is None else cmd.reshape(-1, n, 4)
        yaw = _dev(inp.get("yaw"))
        fr = _dev(frames, np.int64)
        tr = torch.zeros((steps, _cabi.RK_VDT_TRACE_WORDS, n), dtype=torch.int32, device=DEV) if trace else None
        gl = _dev(goal)
        cost = None if goal is None else torch.full((n,), float("nan"), dtype=torch.float32, device=DEV)
        imu_d = None if imu is None else (_dev(imu[0]), _dev(imu[1]), _dev(imu[2]))
        seg_len, yp, k = inp.get("seg_len", 0), inp.get("yaw_period", 0), steps // chunks
        assert steps % chunks == 0 and (chunks == 1 or goal is None)
        for c in range(chunks):
            # launch c takes its slice of the input tables (the whole tables for one launch)
            a = vb.make_args(k, sensor_mode=vi.MODES[entry], seg_len=seg_len, yaw_period=yp, goal=gl, cost=cost, task_period=inp.get("task_period", 0),
                             reset_state=reset, cmd=cmd if cmd is None or chunks == 1 else cmd[c * k // seg_len:(c + 1) * k // seg_len],
                             yaw=yaw if yaw is None or chunks == 1 else yaw[c * k // yp:(c + 1) * k // yp],
                             frames=None if fr is None else fr[c * k:(c + 1) * k], trace=None if tr is None else tr[c * k:(c + 1) * k])
            if imu is not None:
                a.d_imu_regs, a.d_imu_have_quat, a.d_imu_yaw0_deg = (t.data_ptr() for t in imu_d)
                a.n_yaw, a.yaw_period = imu[3], imu[4]
            self.launch(entry, trace, reset, lambda: vb.rollout_args(a))
        return _u32(vb.state), None if tr is None else _u32(tr), None if cost is None else cost.cpu().numpy()


def _plant_cases(b, row):
    p = b.p
    inp, st0, goal, dirty = _work("main", _main)
    n = inp["n"]
    pst, ptr, pcost = _port(row, "main", lambda: port_rollout(p, inp, state=st0, goal=goal))
    st, tr, cost = b.rollout(inp, state=st0, trace=True, goal=goal)
    assert_same(tr, ptr, "traced trace")
    assert_same(st, pst, "traced state")
    assert_same(cost.view(np.uint32), pcost.view(np.uint32), "traced cost")
    st, _, cost = b.rollout(inp, state=st0, goal=goal)
    assert_same(st, pst, "untraced state")
    assert_same(cost.view(np.uint32), pcost.view(np.uint32), "untraced cost")
    st, _, _ = b.rollout(inp, state=st0, chunks=3)
    assert_same(_mask_usec(st, n), _mask_usec(pst, n), "state resumed over three launches")
    zst, ztr, _ = _port(row, "main from power-on", lambda: port_rollout(p, inp))
    for trace in (True, False):
        st, tr, _ = b.rollout(inp, state=dirty, trace=trace, reset=True)
        assert_same(st, zst, f"reset_state state (trace={trace})")
        if trace:
            assert_same(tr, ztr, "reset_state trace")

    one = _work("one", lambda: wl.plant_inputs(1, 500, seed=99))
    ost, otr, _ = _port(row, "one", lambda: port_rollout(p, one))
    for trace in (True, False):
        st, tr, _ = b.rollout(one, trace=trace)
        assert_same(st, ost, f"n = 1 state (trace={trace})")
        if trace:
            assert_same(tr, otr, "n = 1 trace")

    task = _work("task", lambda: dict(task_inputs(333, 500, 32, seg_len=50), task_period=10))
    tst, ttr, _ = _port(row, "task", lambda: port_rollout(p, task))
    st, tr, _ = b.rollout(task, trace=True)
    assert_same(tr, ttr, "task_period trace")
    assert_same(st, tst, "task_period state")

    # one segment of 2600 ticks and no yaw stream: the fast kernel's chunks end at kMaxChunk (2048 ticks)
    long = _work("long", lambda: dict(n=131, steps=2600, cmd=streams.vehicle_commands(131, 1, 17), seg_len=2600))
    lst, _, _ = _port(row, "long", lambda: port_rollout(p, long, trace=False))
    st, _, _ = b.rollout(long)
    assert_same(st, lst, "one 2600-tick segment")

    crawl, cst0 = _work("crawl", _crawl)
    cst, ctr, _ = _port(row, "crawl", lambda: port_rollout(p, crawl, state=cst0))
    for trace in (True, False):
        st, tr, _ = b.rollout(crawl, state=cst0, trace=trace)
        assert_same(st, cst, f"crawl state (trace={trace})")
        if trace:
            assert_same(tr, ctr, "crawl trace")

    reg = _work("yaw register", lambda: dict(wl.plant_inputs(777, 500, seed=41), yaw=streams.vehicle_yaw_reg(777, 50, seed=41)))
    rst, rtr, _ = _port(row, "yaw register", lambda: port_rollout(p, reg))
    st, tr, _ = b.rollout(reg, trace=True)
    assert_same(tr, rtr, "d_yaw_reg trace")
    assert_same(st, rst, "d_yaw_reg state")

    iinp, imu, iyaw = _work("imu", _imu)
    ist, itr, _ = _port(row, "imu", lambda: port_rollout(p, dict(iinp, yaw=iyaw, yaw_period=imu[4])))
    st, tr, _ = b.rollout(iinp, trace=True, imu=imu)
    assert_same(tr, itr, "d_imu_regs trace")
    assert_same(st, ist, "d_imu_regs state")

    wave = _work("waves", _wave)
    wst, _, _ = _port(row, "waves", lambda: port_rollout(p, wave, trace=False))
    st, _, _ = b.rollout(wave)
    assert_same(st, wst, "multi-wave launch")


def _stream_and_hold_cases(b, row):
    p = b.p
    for name, (inp, fr) in _work("stream", _stream).items():
        sst, stt, _ = _port(row, "stream " + name, lambda: port_rollout(p, inp, sensor=_cabi.RK_SENSOR_STREAM, frames=fr))
        for trace in (True, False):
            st, tr, _ = b.rollout(inp, entry="stream", frames=fr, trace=trace)
            assert_same(st, sst, f"stream {name} state (trace={trace})")
            if trace:
                assert_same(tr, stt, f"stream {name} trace")
    hinp, hst0 = _work("hold", lambda: (wl.plant_inputs(257, 40, seed=5, seg_len=8, yaw_period=4), layout.aos_to_soa(wl.random_states(257, seed=3))))
    hst, htr, _ = _port(row, "hold", lambda: port_rollout(p, hinp, sensor=_cabi.RK_SENSOR_HOLD, state=hst0))
    for trace in (True, False):
        st, tr, _ = b.rollout(hinp, entry="hold", state=hst0, trace=trace)
        assert_same(st, hst, f"hold state (trace={trace})")
        if trace:
            assert_same(tr, htr, "hold trace")


def _plan_cases(b, row):
    p = b.p
    src, ref, cand, P, obs, mobs = _work("plan", _plan)
    vb = VehicleBatch(R, DEV)
    vb.load_state_soa(src)
    w_obst = 3.0e3
    exp = _port(row, "plan", lambda: pr.candidate_costs(src, R, S, cand, SEG_LEN, ref, *W, params=p))
    got = b.launch("plan", False, False, lambda: _plan_rollout(vb, R, S, cand, N_SEG, SEG_LEN, ref, W, params=p))
    assert_same(got.view(np.uint32), exp.view(np.uint32), "rk_plan_rollout costs")
    exp, O = _port(row, "obstacles", lambda: por.candidate_costs_obst(src, R, S, cand, SEG_LEN, ref, *W, obs, P, w_obst, params=p))
    assert (O == 0).any() and (O > 0).any(), "the discs must be entered by some candidates and missed by others"
    got = b.launch("obstacles", False, False, lambda: _obst_rollout(vb, cand, ref, obs, P, w_obst, params=p))
    assert_same(got.view(np.uint32), exp.view(np.uint32), "rk_plan_rollout_obstacles costs")
    exp, O, exp_path = _port(row, "moving", lambda: pfr.candidate_costs_moving(src, R, S, cand, SEG_LEN, ref, *W, mobs, P, w_obst, params=p))
    assert (O == 0).any() and (O > 0).any(), "the moving discs must be entered by some candidates and missed by others"
    got, path = b.launch("moving", False, False, lambda: _moving_rollout(vb, cand, ref, mobs, P, w_obst, params=p, path=True))
    assert_same(got.view(np.uint32), exp.view(np.uint32), "rk_plan_rollout_moving costs")
    assert_same(path.view(np.uint32), exp_path.view(np.uint32), "rk_plan_rollout_moving paths")
    assert_same(_u32(vb.state), src, "the planner wrote the source states")


@pytest.mark.parametrize("row", vi.MATRIX, ids=vi.row_id)
def test_row_launches_its_instantiations_bit_exact_vs_port(row, options):
    p = _params(row)
    options(row)
    b = Battery(row, p)
    _plant_cases(b, row)
    _stream_and_hold_cases(b, row)
    _plan_cases(b, row)
    assert b.ran == vi.BATTERY, f"the battery ran {sorted(b.ran)}, vdt_instances.BATTERY declares {sorted(vi.BATTERY)}"


def test_defaults_restored_and_default_launch_runs_the_default_kernel():
    """After the matrix the options are back at their defaults: a plain traced-off launch runs the default kernel."""
    row = dict(vi.MATRIX[0], occupancy=4, packed=1, ffsat=0, force_transcription=0, kd=0.0, ff_limit=1.0)
    b = Battery(row, _params(row))
    inp = wl.plant_inputs(300, 200, seed=3)
    st, _, _ = b.rollout(inp)
    assert b.ran == {("plant", False, False)}
    assert_same(st, port_rollout(b.p, inp, trace=False)[0], "default launch state")


def test_matrix_launched_every_compiled_instantiation():
    if vi.tool("cuobjdump") is None or vi.tool("cu++filt") is None:
        pytest.skip("cuobjdump / cu++filt not found")
    compiled = vi.inventory()
    never = sorted(compiled - set(LAUNCHED))
    assert not never, f"{len(never)} of {len(compiled)} compiled instantiations were never launched: {never}"
    assert set(LAUNCHED) == compiled, f"launched instantiations not in the library: {sorted(set(LAUNCHED) - compiled)}"
