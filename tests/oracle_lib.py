"""TEST INFRASTRUCTURE: ctypes loaders for the oracles.

  port()  -> oracle/liboracle_port.so   plain-C restatement (always available; built by
             oracle/Makefile / __graft_entry__.build())
  ref()   -> oracle/_ref/libref_vdt.so  the UNMODIFIED reference compiled for x86 (built
             where /root/reference exists; the prebuilt .so travels to the GPU box)
"""
import ctypes as C
import hashlib
import json
import os
import subprocess

import numpy as np

import roboken_fmskf_robot_controller_b200 as rk
from roboken_fmskf_robot_controller_b200 import _cabi, layout, streams

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE = os.path.join(ROOT, "oracle")

_cache = {}


def _build(target):
    subprocess.run(["make", "-s", "-C", ORACLE, target], check=True, capture_output=True)


def port():
    if "port" not in _cache:
        path = os.path.join(ORACLE, "liboracle_port.so")
        if not os.path.exists(path):
            _build("port")
        lib = C.CDLL(path)
        vp = C.c_void_p
        lib.orc_vdt_rollout.argtypes = [C.POINTER(_cabi.VdtParams), vp, C.c_int64, C.c_int64, C.c_int64,
                                        C.POINTER(_cabi.VdtRollout), C.c_int]
        lib.orc_vdt_rollout.restype = None
        f3 = C.POINTER(C.c_float)
        lib.orc_vdt_set_target.argtypes = [C.POINTER(_cabi.VdtParams), vp, f3, f3, f3]
        lib.orc_vdt_rx.argtypes = [C.POINTER(_cabi.VdtParams), vp, C.c_int, C.c_char_p, C.c_int16]
        lib.orc_vdt_update.argtypes = [C.POINTER(_cabi.VdtParams), vp]
        lib.orc_imt_update.argtypes = [vp, C.c_int64, C.c_int64, C.c_int64, C.c_int, vp, vp, vp, C.c_int]
        lib.orc_imt_update.restype = None
        lib.orc_imt_feed_bytes.argtypes = [vp, vp, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int, vp, vp, vp, vp, C.c_int]
        lib.orc_imt_feed_bytes.restype = None
        lib.orc_rmt_guard.argtypes = [C.POINTER(_cabi.RmtParams), vp, C.c_int64, C.c_int64, C.c_int64, C.c_int, vp, vp, vp]
        lib.orc_rmt_guard.restype = None
        lib.orc_atanf.argtypes = [C.c_float]
        lib.orc_atanf.restype = C.c_float
        lib.orc_atan2f.argtypes = [C.c_float, C.c_float]
        lib.orc_atan2f.restype = C.c_float
        lib.orc_adt_batch.argtypes = [C.c_int, C.POINTER(_cabi.AdtParams), vp, vp, C.c_int64, C.c_int64, C.c_int64, C.c_int,
                                      vp, vp, vp, vp, vp]
        lib.orc_adt_batch.restype = None
        lib.orc_adt_rx_batch.argtypes = [C.c_int, C.POINTER(_cabi.AdtParams), vp, C.c_int64, C.c_int64, C.c_int64, vp, vp, vp]
        lib.orc_adt_rx_batch.restype = None
        lib.orc_adp_batch.argtypes = lib.orc_adt_batch.argtypes
        lib.orc_adp_batch.restype = None
        lib.orc_adh_batch.argtypes = [C.c_int, C.POINTER(_cabi.AdtParams), vp, vp, C.c_int64, C.c_int64, C.c_int64, C.c_int, vp, vp]
        lib.orc_adh_batch.restype = None
        for nm in ("orc_sin", "orc_cos", "orc_normalize_rad_0to2pi", "orc_normalize_deg_0to360"):
            getattr(lib, nm).argtypes = [C.c_float]
            getattr(lib, nm).restype = C.c_float
        _cache["port"] = lib
    return _cache["port"]


REF_DIGESTS = os.path.join(ROOT, "tests", "golden", "ref_digests.json")


def digest(out):
    """SHA-256 over every array in a (nested) result: dtype, shape and bytes."""
    h = hashlib.sha256()

    def walk(x):
        if isinstance(x, (list, tuple)):
            for y in x:
                walk(y)
        elif isinstance(x, dict):
            for k in sorted(x):
                h.update(k.encode())
                walk(x[k])
        elif x is not None:
            a = np.ascontiguousarray(x)
            h.update(f"{a.dtype.str}{a.shape}".encode())
            h.update(a.tobytes())

    walk(out)
    return h.hexdigest()


def reference_result(key, run, *libs):
    """What the compiled reference returns for one test case: run("ref") where oracle/_ref has every library in `libs`,
    run("port") elsewhere.  Either way the result must match the SHA-256 recorded under `key` in tests/golden/ref_digests.json,
    so a checkout without the reference still holds the port (and the GPU tests built on it) to the reference's answer.
    With ROBOTICK_RECORD_REF_DIGESTS=1 a missing key is recorded instead, noting which implementation produced it."""
    kind = "ref" if all(os.path.exists(os.path.join(ORACLE, "_ref", name)) for name in libs) else "port"
    out = run(kind)
    with open(REF_DIGESTS) as f:
        table = json.load(f)
    d = digest(out)
    if key not in table and os.environ.get("ROBOTICK_RECORD_REF_DIGESTS") == "1":
        table[key] = {"sha256": d, "from": kind}
        with open(REF_DIGESTS, "w") as f:
            json.dump(table, f, indent=1, sort_keys=True)
            f.write("\n")
    assert key in table, f"no recorded reference result for {key!r} in {REF_DIGESTS}"
    assert d == table[key]["sha256"], f"{key}: the {kind} result differs from the recorded reference result"
    return out


def have_ref(name="libref_vdt.so"):
    return os.path.exists(os.path.join(ORACLE, "_ref", name)) or os.path.isdir("/root/reference/src")


def ref(name="libref_vdt.so"):
    if name not in _cache:
        path = os.path.join(ORACLE, "_ref", name)
        if not os.path.exists(path):
            _build("ref")
        lib = C.CDLL(path)
        vp = C.c_void_p
        if name.startswith("libref_vdt") and not name.startswith("libref_vdt_task"):
            lib.ref_vdt_create.restype = vp
            lib.ref_vdt_destroy.argtypes = [vp]
            lib.ref_vdt_start.argtypes = [vp]
            lib.ref_vdt_stop.argtypes = [vp]
            f3 = C.POINTER(C.c_float)
            lib.ref_vdt_set_target.argtypes = [vp, f3, f3, f3]
            lib.ref_vdt_set_yaw.argtypes = [vp, C.c_float]
            lib.ref_vdt_rx.argtypes = [vp, C.c_int, C.c_char_p, C.c_int16]
            lib.ref_vdt_update.argtypes = [vp]
            lib.ref_vdt_export.argtypes = [vp, vp]
            lib.ref_vdt_import.argtypes = [vp, vp]
            lib.ref_vdt_get.argtypes = [vp, f3, f3, f3, C.POINTER(C.c_int16)]
            lib.ref_vdt_rollout.argtypes = [vp, C.c_int64, C.c_int64, C.c_int64, C.POINTER(_cabi.VdtRollout), C.c_int]
            lib.ref_vdt_rollout.restype = None
            for nm in ("ref_normalize_rad_0to2pi", "ref_normalize_deg_0to360", "ref_atanf", "ref_sinf",
                       "ref_cosf", "ref_sqrtf"):
                getattr(lib, nm).argtypes = [C.c_float]
                getattr(lib, nm).restype = C.c_float
            lib.ref_atan2f.argtypes = [C.c_float, C.c_float]
            lib.ref_atan2f.restype = C.c_float
        if name.startswith("libref_vdt_task"):
            lib.ref_vdt_task_rollout.argtypes = [vp, C.c_int64, C.c_int64, C.c_int64, C.POINTER(_cabi.VdtRollout), vp]
            lib.ref_vdt_task_rollout.restype = None
        if name.startswith("libref_rm"):
            lib.ref_rmt_guard.argtypes = [C.POINTER(_cabi.RmtParams), vp, C.c_int64, C.c_int64, C.c_int64, C.c_int, vp, vp, vp]
            lib.ref_rmt_guard.restype = None
            lib.ref_rm_atanf.argtypes = [C.c_float]
            lib.ref_rm_atanf.restype = C.c_float
            lib.ref_rm_atan2f.argtypes = [C.c_float, C.c_float]
            lib.ref_rm_atan2f.restype = C.c_float
            lib.ref_rm_atan_tables.argtypes = [vp, vp, vp]
        if name.startswith("libref_imu"):
            lib.ref_imt_create.restype = vp
            lib.ref_imt_destroy.argtypes = [vp]
            R = C.POINTER(C.c_int16)
            lib.ref_imt_init.argtypes = [vp, R]
            lib.ref_imt_update.argtypes = [vp, R, C.c_int]
            lib.ref_imt_yaw.argtypes = [vp]
            lib.ref_imt_yaw.restype = C.c_float
            lib.ref_imt_is_error.argtypes = [vp]
            lib.ref_imt_get.argtypes = [vp, C.POINTER(C.c_float)]
            lib.ref_imt_export.argtypes = [vp, vp]
            lib.ref_imt_import.argtypes = [vp, vp]
            lib.ref_imt_rollout.argtypes = [vp, C.c_int64, C.c_int64, C.c_int64, C.c_int, vp, vp, vp, C.c_int]
            lib.ref_imt_rollout.restype = None
            lib.ref_imt_bytes_rollout.argtypes = [vp, C.c_int64, C.c_int64, C.c_int64, C.c_int, C.c_int, vp, vp, vp, vp]
            lib.ref_imt_bytes_rollout.restype = None
        if name.startswith("libref_arm"):
            lib.ref_adh_batch.argtypes = [C.c_int, vp, vp, C.c_int64, C.c_int64, C.c_int64, C.c_int, vp, vp]
            lib.ref_adh_batch.restype = None
            lib.ref_adt_create.restype = vp
            for nm in ("ref_adt_destroy", "ref_adt_bringup", "ref_adt_tick"):
                getattr(lib, nm).argtypes = [vp]
                getattr(lib, nm).restype = None
            lib.ref_adt_push.argtypes = [vp, C.POINTER(_cabi.AdtPosCmdSeq)]
            lib.ref_adt_status.argtypes = [vp, C.c_uint32]
            lib.ref_adt_targets.argtypes = [vp, C.POINTER(C.c_float)]
            lib.ref_adt_export.argtypes = [vp, vp]
            lib.ref_adt_import.argtypes = [vp, vp]
            lib.ref_adt_trace_row.argtypes = [vp, vp]
            lib.ref_adt_debug_seq.argtypes = [C.c_int, C.POINTER(_cabi.AdtPosCmdSeq)]
            lib.ref_adt_batch.argtypes = [C.c_int, vp, vp, C.c_int64, C.c_int64, C.c_int64, C.c_int, vp, vp, vp, vp, vp]
            lib.ref_adt_batch.restype = None
            lib.ref_adt_rx_batch.argtypes = [C.c_int, vp, C.c_int64, C.c_int64, C.c_int64, vp, vp, vp]
            lib.ref_adt_rx_batch.restype = None
            lib.ref_adp_batch.argtypes = lib.ref_adt_batch.argtypes
            lib.ref_adp_batch.restype = None
        _cache[name] = lib
    return _cache[name]


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


class HostRollout:
    """Builds an rk_vdt_rollout_t over HOST numpy arrays and keeps them alive."""

    def __init__(self, n, steps, sensor_mode, cmd=None, seg_len=0, yaw=None, yaw_period=0, frames=None,
                 trace=False, goal=None, task_period=0):
        self.n = n
        self.keep = [cmd, yaw, frames, goal]
        self.trace = np.zeros((steps, _cabi.RK_VDT_TRACE_WORDS, n), dtype=np.uint32) if trace else None
        self.cost = np.zeros(n, dtype=np.float32) if goal is not None else None
        a = _cabi.VdtRollout()
        a.steps, a.sensor_mode = steps, sensor_mode
        a.d_cmd, a.n_seg, a.seg_len = _ptr(cmd), (0 if cmd is None else cmd.shape[0]), seg_len
        a.n_yaw, a.yaw_period = (0 if yaw is None else yaw.shape[0]), yaw_period
        if yaw is not None and yaw.dtype == np.int16:
            a.d_yaw_reg = _ptr(yaw)  # the WT901C Yaw register stream
        else:
            a.d_yaw = _ptr(yaw)
        a.d_frames = _ptr(frames)
        a.d_trace = _ptr(self.trace)
        a.d_goal, a.d_cost = _ptr(goal), _ptr(self.cost)
        a.task_period = task_period
        self.args = a


def run_port(state_soa, n, ro, params=None, nthreads=1):
    p = params or rk.default_params()
    port().orc_vdt_rollout(C.byref(p), _ptr(state_soa), n, 0, n, C.byref(ro.args), nthreads)


def run_ref(state_soa, n, ro, nthreads=1, name="libref_vdt.so"):
    ref(name).ref_vdt_rollout(_ptr(state_soa), n, 0, n, C.byref(ro.args), nthreads)


def run_task_ref(state_soa, n, ro, yaw_deg):
    """The reference's whole vehicle task (VD_task_main.cpp compiled unmodified) from the power-on state."""
    ref("libref_vdt_task.so").ref_vdt_task_rollout(_ptr(state_soa), n, 0, n, C.byref(ro.args), _ptr(yaw_deg))


def imu_port(state_soa, n, regs, have=None, want_out=False, do_init=False):
    K = regs.shape[0]
    out = np.zeros((K, 4, n, 4), dtype=np.uint32) if want_out else None
    cells = streams.imu_cells(regs)  # regs: logical int16 [K, 16, n]
    port().orc_imt_update(_ptr(state_soa), n, 0, n, K, _ptr(cells), _ptr(have), _ptr(out), int(do_init))
    return out


def imu_ref(state_soa, n, regs, have=None, want_out=False, do_init=False):
    K = regs.shape[0]
    out = np.zeros((K, 4, n, 4), dtype=np.uint32) if want_out else None
    cells = streams.imu_cells(regs)
    ref("libref_imu.so").ref_imt_rollout(_ptr(state_soa), n, 0, n, K, _ptr(cells), _ptr(have), _ptr(out), int(do_init))
    return out


def imu_bytes_port(state_soa, parser_soa, n, cells, nbytes=None, want_out=False, want_yaw=False, do_init=False):
    """rk_imt_feed_bytes on host arrays (the port).  cells: uint32 [K, ncells, n, 4]; nbytes: uint16 [K, n] or None."""
    K, ncells = cells.shape[0], cells.shape[1]
    assert cells.dtype == np.uint32 and cells.shape[2:] == (n, 4) and cells.flags.c_contiguous
    assert nbytes is None or (nbytes.dtype == np.uint16 and nbytes.shape == (K, n) and nbytes.flags.c_contiguous)
    out = np.zeros((K, 4, n, 4), dtype=np.uint32) if want_out else None
    yaw = np.zeros((K, n), dtype=np.float32) if want_yaw else None
    port().orc_imt_feed_bytes(_ptr(state_soa), _ptr(parser_soa), n, 0, n, K, ncells, _ptr(cells), _ptr(nbytes), _ptr(out), _ptr(yaw),
                              int(do_init))
    return (out, yaw) if want_yaw else out


def imu_bytes_ref(state_soa, n, cells, nbytes=None, want_out=False):
    """The compiled reference (vendor parser + IMU_IF_WT901C) replayed from power-on: update 0 is init().
    Returns (out, sreg int16 [n, 16])."""
    K, ncells = cells.shape[0], cells.shape[1]
    assert ncells * 16 <= 512  # the fake Serial6 FIFO
    assert cells.dtype == np.uint32 and cells.shape[2:] == (n, 4) and cells.flags.c_contiguous
    assert nbytes is None or (nbytes.dtype == np.uint16 and nbytes.shape == (K, n) and nbytes.flags.c_contiguous)
    out = np.zeros((K, 4, n, 4), dtype=np.uint32) if want_out else None
    sreg = np.zeros((n, 16), dtype=np.int16)
    ref("libref_imu.so").ref_imt_bytes_rollout(_ptr(state_soa), n, 0, n, K, ncells, _ptr(cells), _ptr(nbytes), _ptr(out), _ptr(sreg))
    return out, sreg


def arm_homing(kind, op, state, hstate, n, K=0, mode=0, now=None, trace=False, params=None):
    """rk_adh_mode_init ("init", mode) / rk_adh_update ("update", K ticks) on host arrays via the port or the compiled
    reference modes.  now: float32 [K, 4, n] servo feedback or None.  Returns the trace (uint32 [K, 16, n]) or None."""
    p = params or _cabi.default_arm_params()
    tr = np.zeros((K, layout.ADT_TRACE_WORDS, n), dtype=np.uint32) if (trace and op == "update") else None
    if now is not None:
        assert now.dtype == np.float32 and now.shape == (K, 4, n) and now.flags.c_contiguous
    o, k = (0, mode) if op == "init" else (2, K)
    if kind == "port":
        port().orc_adh_batch(o, C.byref(p), _ptr(state), _ptr(hstate), n, 0, n, k, _ptr(now), _ptr(tr))
    else:
        ref("libref_arm.so").ref_adh_batch(o, _ptr(state), _ptr(hstate), n, 0, n, k, _ptr(now), _ptr(tr))
    return tr


def rm_default_params():
    return _cabi.RmtParams(200, 200, 100)


def rm_guard(kind, state_soa, n, inp, params=None, want_abort=True):
    """rk_rmt_guard on host arrays through the port ("port") or the compiled RobotManager task ("ref").
    inp: uint32 [K, 3, n, 4].  Returns (cmd uint32 [K, n, 4], abort uint32 [K, n])."""
    K = inp.shape[0]
    assert inp.dtype == np.uint32 and inp.shape[1:] == (3, n, 4) and inp.flags.c_contiguous
    p = params or rm_default_params()
    cmd = np.zeros((K, n, 4), dtype=np.uint32)
    ab = np.zeros((K, n), dtype=np.uint32) if want_abort else None
    fn = port().orc_rmt_guard if kind == "port" else ref("libref_rm.so").ref_rmt_guard
    fn(C.byref(p), _ptr(state_soa), n, 0, n, K, _ptr(inp), _ptr(cmd), _ptr(ab))
    return cmd, ab


# ---- arm ---------------------------------------------------------------------------------
ARM_OPS = {"init": 0, "push": 1, "update": 2, "status": 3}


def arm_batch(kind, op, state, cmdtab, n, K=0, seq=None, valid=None, trace=False, ids=None, params=None):
    """Runs one rk_adt_* batch op on HOST SoA arrays through the port ("port") or the compiled
    reference ("ref").  Returns (trace or None, status or None); state/cmdtab updated in place."""
    tr = np.zeros((K, layout.ADT_TRACE_WORDS, n), dtype=np.uint32) if (trace and op == "update") else None
    status = np.zeros(n, dtype=np.int32) if op == "status" else None
    if kind == "port":
        p = params or _cabi.default_arm_params()
        port().orc_adt_batch(ARM_OPS[op], C.byref(p), _ptr(state), _ptr(cmdtab), n, 0, n, K, _ptr(seq), _ptr(valid),
                             _ptr(tr), _ptr(ids), _ptr(status))
    else:
        assert params is None, "the compiled reference has the firmware constants wired in"
        ref("libref_arm.so").ref_adt_batch(ARM_OPS[op], _ptr(state), _ptr(cmdtab), n, 0, n, K, _ptr(seq), _ptr(valid),
                                           _ptr(tr), _ptr(ids), _ptr(status))
    return tr, status


def arm_rx(kind, which, state, n, frames, cmdid=None, cur=None, params=None):
    """Servo feedback frames through the rx callbacks (rk_adt_bldc_rx: which = 0..2, rk_adt_mg_rx: which = 3) on HOST
    SoA arrays, port or compiled reference.  frames: uint64 [n]; cmdid: uint32 [n] or None; cur: float32 [n] (in/out) or None."""
    assert frames.dtype == np.uint64 and frames.shape == (n,)
    if kind == "port":
        p = params or _cabi.default_arm_params()
        port().orc_adt_rx_batch(which, C.byref(p), _ptr(state), n, 0, n, _ptr(frames), _ptr(cmdid), _ptr(cur))
    else:
        assert params is None, "the compiled reference has the firmware constants wired in"
        ref("libref_arm.so").ref_adt_rx_batch(which, _ptr(state), n, 0, n, _ptr(frames), _ptr(cmdid), _ptr(cur))


def armpos_batch(kind, op, state, pstate, n, K=0, cmd=None, valid=None, trace=False, ids=None, params=None):
    """ADTModePositioning (single-command mode) batch op on HOST SoA arrays; cmd = uint32 [2, n, 4] planes."""
    tr = np.zeros((K, layout.ADT_TRACE_WORDS, n), dtype=np.uint32) if (trace and op == "update") else None
    status = np.zeros(n, dtype=np.int32) if op == "status" else None
    if kind == "port":
        p = params or _cabi.default_arm_params()
        port().orc_adp_batch(ARM_OPS[op], C.byref(p), _ptr(state), _ptr(pstate), n, 0, n, K, _ptr(cmd), _ptr(valid), _ptr(tr),
                             _ptr(ids), _ptr(status))
    else:
        ref("libref_arm.so").ref_adp_batch(ARM_OPS[op], _ptr(state), _ptr(pstate), n, 0, n, K, _ptr(cmd), _ptr(valid), _ptr(tr),
                                           _ptr(ids), _ptr(status))
    return tr, status


def seq_struct_to_image(q):
    """rk_adt_poscmdseq_t -> uint32[260] slot image"""
    img = np.zeros(layout.ACMD_SLOT_WORDS, dtype=np.uint32)
    img[0], img[1] = q.id, q.len
    for k in range(32):
        img[4 + 8 * k] = q.cmd[k].dt_ms
        img[5 + 8 * k : 10 + 8 * k] = np.array(q.cmd[k].tgt_deg[:], dtype=np.float32).view(np.uint32)
    return img


def image_to_seq_struct(img):
    q = _cabi.AdtPosCmdSeq()
    q.id, q.len = int(img[0]), int(img[1]) & 0xFF
    for k in range(32):
        q.cmd[k].dt_ms = int(img[4 + 8 * k])
        q.cmd[k].tgt_deg[:] = [float(x) for x in np.asarray(img[5 + 8 * k : 10 + 8 * k], dtype=np.uint32).view(np.float32)]
    return q


# ---- full tick (vehicle + IMU + arm) ---------------------------------------------------------
def full_tick(kind, n, steps, slow_period, cmd, seg_len, regs, have, vstate, istate, astate, atab, trace=False, goal=None,
              nthreads=1):
    """The firmware's coupling restated on the HOST from the per-module oracles: IMU update k runs
    before vehicle tick k*slow_period and the vehicle ISR reads deg2rad(getYawDate())
    (VD_task_main.cpp:368, util_mymath.hpp:13,16); the arm ticks at the IMU rate.  `kind` selects
    the plain-C port or the compiled reference for every module.  States updated in place."""
    from roboken_fmskf_robot_controller_b200 import streams

    n_slow = (steps + slow_period - 1) // slow_period
    out = (imu_port if kind == "port" else imu_ref)(istate, n, regs[:n_slow], None if have is None else have[:n_slow], want_out=True)
    yaw_deg = np.ascontiguousarray(out[:, 2, :, 3]).view(np.float32)  # Data.angle[2] = word 11
    yaw = (yaw_deg * streams.DEG2RAD).astype(np.float32)
    ro = HostRollout(n, steps, _cabi.RK_SENSOR_PLANT, cmd, seg_len, yaw, slow_period, trace=trace, goal=goal)
    if kind == "port":
        run_port(vstate, n, ro, nthreads=nthreads)
    else:
        run_ref(vstate, n, ro, nthreads=nthreads)
    atr, _ = arm_batch(kind, "update", astate, atab, n, K=n_slow, trace=trace)
    return ro.trace, atr, yaw, ro.cost
