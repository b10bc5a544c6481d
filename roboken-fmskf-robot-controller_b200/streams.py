"""Seeded synthetic command / sensor streams (SURVEY.md section 8d).

Everything here is host-side input generation: counter-based (splitmix64 of
(seed, stream, instance, index)), vectorised numpy, float32 results produced only from
exactly-representable integer arithmetic or IEEE float32 ops, so the SAME arrays feed the
CUDA engine, the C port and the compiled reference.
"""
import numpy as np

from . import _cabi

_M64 = np.uint64(0xFFFFFFFFFFFFFFFF)


def splitmix64(x):
    x = (np.asarray(x, dtype=np.uint64) + np.uint64(0x9E3779B97F4A7C15)) & _M64
    z = x
    z = ((z ^ (z >> np.uint64(30))) * np.uint64(0xBF58476D1CE4E5B9)) & _M64
    z = ((z ^ (z >> np.uint64(27))) * np.uint64(0x94D049BB133111EB)) & _M64
    return z ^ (z >> np.uint64(31))


def _hash(seed, stream, inst, idx):
    with np.errstate(over="ignore"):
        h = splitmix64(np.uint64(seed) ^ (np.uint64(stream) * np.uint64(0xD6E8FEB86659FD93)))
        h = splitmix64(h ^ np.asarray(inst, dtype=np.uint64))
        h = splitmix64(h ^ (np.asarray(idx, dtype=np.uint64) * np.uint64(0xA0761D6478BD642F)))
    return h


def _u01(h):
    """24-bit uniform in [0,1) as exact float32."""
    return (h >> np.uint64(40)).astype(np.float32) * np.float32(1.0 / 16777216.0)


def vehicle_commands(n, n_seg, seed=0x5EED, first=0, stop_every=8):
    """C2 command schedule: [n_seg, n] rk_vdt_cmd_t records (structured array).

    vx, vy ~ U[-400, 400] mm/s norm-clamped to 400 exactly as speed_limit_xy() does
    (VD_task_main.cpp:127-137); vth ~ U[-2*pi, 2*pi] clamped by speed_limit_rot() (:139-142);
    one segment in `stop_every` is a MOVE_STOP (zero target, STOP accel/jerk tables).
    """
    inst = (np.arange(n, dtype=np.uint64) + np.uint64(first))[None, :]
    seg = np.arange(n_seg, dtype=np.uint64)[:, None]
    f32 = np.float32
    vx = _u01(_hash(seed, 1, inst, seg)) * f32(800.0) - f32(400.0)
    vy = _u01(_hash(seed, 2, inst, seg)) * f32(800.0) - f32(400.0)
    vth = _u01(_hash(seed, 3, inst, seg)) * f32(4.0 * np.pi) - f32(2.0 * np.pi)
    # speed_limit_xy: sqrt, clamp, x*lim/len  (all IEEE float32, left to right)
    ln = np.sqrt(vx * vx + vy * vy, dtype=np.float32)
    lim = np.minimum(ln, f32(400.0))
    nz = ln != 0
    safe = np.where(nz, ln, f32(1.0))
    vx = np.where(nz, (vx * lim) / safe, f32(0.0)).astype(np.float32)
    vy = np.where(nz, (vy * lim) / safe, f32(0.0)).astype(np.float32)
    rl = f32(6.0 * np.pi)
    vth = np.clip(vth, -rl, rl).astype(np.float32)
    stop = (_hash(seed, 4, inst, seg) % np.uint64(stop_every)) == 0
    cmd = np.zeros((n_seg, n), dtype=np.dtype([("vx", "<f4"), ("vy", "<f4"), ("vth", "<f4"), ("kind", "<i4")]))
    cmd["vx"] = np.where(stop, f32(0), vx)
    cmd["vy"] = np.where(stop, f32(0), vy)
    cmd["vth"] = np.where(stop, f32(0), vth)
    cmd["kind"] = np.where(stop, _cabi.RK_CMD_STOP, _cabi.RK_CMD_MOVE)
    return cmd


DEG2RAD = np.float32(np.float32(3.14159265358979) / np.float32(180.0))  # util_mymath.hpp:13


def vehicle_yaw(n, n_yaw, seed=0x5EED, first=0, degrees=False):
    """Yaw stream at the IMU rate: integer-stepped triangle wave in whole degrees in
    [-180, 180), converted with mymath::deg2rad (util_mymath.hpp:16).  [n_yaw, n] float32."""
    inst = (np.arange(n, dtype=np.uint64) + np.uint64(first))[None, :]
    k = np.arange(n_yaw, dtype=np.int64)[:, None]
    phase = (_hash(seed, 5, inst, 0) % np.uint64(720)).astype(np.int64)
    rate = (_hash(seed, 6, inst, 0) % np.uint64(5)).astype(np.int64) + 1  # deg per IMU sample
    u = (phase + rate * k) % 720
    deg = np.where(u < 360, u - 180, 539 - u)  # -180..179 then 179..-180
    if degrees:  # what IMT::get_status_now_yaw() reports; the ISR applies mymath::deg2rad itself (VD_task_main.cpp:368)
        return deg.astype(np.float32)
    return (deg.astype(np.float32) * DEG2RAD).astype(np.float32)


def vehicle_yaw_reg(n, n_yaw, seed=0x5EED, first=0):
    """The same kind of yaw stream as the sensor delivers it: the WT901C Yaw register, int16 [n_yaw, n], 180/32768
    degrees per count.  Per instance a constant turn rate of 1..5 steps of 182 counts (about one degree) per IMU sample
    from a random phase, wrapping at +-180 degrees like the real heading (int16 overflow)."""
    inst = (np.arange(n, dtype=np.uint64) + np.uint64(first))[None, :]
    k = np.arange(n_yaw, dtype=np.int64)[:, None]
    phase = (_hash(seed, 5, inst, 0) % np.uint64(65536)).astype(np.int64)
    rate = ((_hash(seed, 6, inst, 0) % np.uint64(5)).astype(np.int64) + 1) * 182
    sign = np.where((_hash(seed, 9, inst, 0) % np.uint64(2)) == 0, 1, -1)
    return ((phase + sign * rate * k) & 0xFFFF).astype(np.uint16).view(np.int16)


def yaw_reg_to_rad(reg):
    """What the vehicle ISR sees for a Yaw register value: reg / 32768.0f * 180.0f (imu_if_wt901c.cpp:100), then
    mymath::deg2rad (VD_task_main.cpp:368); float32, one rounding per operation."""
    deg = (reg.astype(np.float32) / np.float32(32768.0)) * np.float32(180.0)
    return (deg * DEG2RAD).astype(np.float32)


def vehicle_frames(n, steps, seed=0x5EED, first=0):
    """RK_SENSOR_STREAM input: [steps, 4, n] uint64 M2006 feedback frames
    (VD_motor_if_m2006.hpp:13-21, big-endian angle/speed/current) from a per-wheel random
    walk: rpm wanders within +-8000, the angle integrates it and wraps at 8192."""
    inst = (np.arange(n, dtype=np.uint64) + np.uint64(first))[None, None, :]
    w = np.arange(4, dtype=np.uint64)[None, :, None]
    t = np.arange(steps, dtype=np.uint64)[:, None, None]
    dr = (_hash(seed, 7, inst * np.uint64(4) + w, t) % np.uint64(401)).astype(np.int64) - 200
    rpm = np.clip(np.cumsum(dr, axis=0), -8000, 8000)
    ang = np.cumsum((rpm * 8192) // 60000, axis=0) % 8192
    cur = (_hash(seed, 8, inst * np.uint64(4) + w, t) % np.uint64(6001)).astype(np.int64) - 3000
    b = np.zeros((steps, 4, n, 8), dtype=np.uint8)
    b[..., 0] = (ang >> 8) & 255
    b[..., 1] = ang & 255
    b[..., 2] = (rpm >> 8) & 255
    b[..., 3] = rpm & 255
    b[..., 4] = (cur >> 8) & 255
    b[..., 5] = cur & 255
    return b.view(np.uint64).reshape(steps, 4, n)


def imu_samples(n, n_upd, seed=0x5EED, first=0, drop_every=64):
    """C3 stream: WT901 register snapshots, int16 [n_upd, 16, n] (+ have_quat uint8 [n_upd, n]).

    AX..Yaw ~ U{-32768..32767}; q0..q3 a random unit quaternion x 32767 rounded; one update in
    `drop_every` carries no quaternion frame (error / hold path, imu_if_wt901c.cpp:83-89)."""
    inst = (np.arange(n, dtype=np.uint64) + np.uint64(first))[None, None, :]
    u = np.arange(n_upd, dtype=np.uint64)[:, None, None]
    r = np.arange(16, dtype=np.uint64)[None, :, None]
    h = _hash(seed, 20, inst * np.uint64(16) + r, u)
    regs = ((h >> np.uint64(13)) & np.uint64(0xFFFF)).astype(np.uint16).view(np.int16).copy()
    g = _u01(_hash(seed, 21, inst * np.uint64(16) + r, u))[:, 12:16, :].astype(np.float64) * 2.0 - 1.0
    nrm = np.sqrt((g * g).sum(axis=1, keepdims=True))
    nrm[nrm == 0] = 1.0
    regs[:, 12:16, :] = np.rint(g / nrm * 32767.0).astype(np.int16)
    have = (_hash(seed, 22, inst[:, 0, :], u[:, 0, :]) % np.uint64(drop_every) != 0).astype(np.uint8)
    return np.ascontiguousarray(regs), np.ascontiguousarray(have)


def imu_cells(regs):
    """Register snapshots int16 [K, 16, n] -> the two-128-bit-cells-per-sample layout rk_imt_update takes:
    int16 [K, 2, n, 8] (register r of sample u, IMU i at ((u*2 + r//8)*n + i)*8 + r%8)."""
    K, _, n = regs.shape
    return np.ascontiguousarray(regs.reshape(K, 2, 8, n).transpose(0, 1, 3, 2))


def arm_sequences(n, seed=0x5EED, first=0, max_len=32, min_len=2, seq_id=1, dt_zero_every=4):
    """C4 command sequences: one PosCmdSeq per arm as an AoS slot image, uint32 [n, 260]
    (word 0 u32_id, 1 u8_cmd_seq_len, 2-3 zero, then 32 x {u32_dt_ms, fl_tgt_pos_deg[5], 0, 0};
    AD_mode_positioning_seq.hpp:15-24).  len ~ U{min_len..max_len}; dt_ms absolute and
    non-decreasing, increments ~ U{10..1000} (1 in 8 is 0: a zero-length segment, one cycle);
    1 arm in `dt_zero_every` starts with dt=0 like POS_CMD_SEQ_DEBUG_2; angles ~ U[-150,150]
    deg in whole 1/64 deg (exact float32).  Entries past len hold stale random waypoints, as a
    reused firmware buffer would."""
    inst = (np.arange(n, dtype=np.uint64) + np.uint64(first))[:, None]
    k = np.arange(32, dtype=np.uint64)[None, :]
    ln = (_hash(seed, 30, inst[:, 0], 0) % np.uint64(max_len - min_len + 1)).astype(np.int64) + min_len
    inc = (_hash(seed, 31, inst, k) % np.uint64(991)).astype(np.int64) + 10
    inc[(_hash(seed, 32, inst, k) % np.uint64(8)) == 0] = 0
    z = (_hash(seed, 33, inst[:, 0], 0) % np.uint64(dt_zero_every)) == 0
    inc[z, 0] = 0
    dt = np.cumsum(inc, axis=1)
    img = np.zeros((n, 260), dtype=np.uint32)
    img[:, 0] = seq_id
    img[:, 1] = ln
    wp = img[:, 4:].reshape(n, 32, 8)
    wp[:, :, 0] = dt.astype(np.uint32)
    for j in range(5):
        q = (_hash(seed, 34 + j, inst, k) % np.uint64(300 * 64 + 1)).astype(np.int64) - 150 * 64
        wp[:, :, 1 + j] = (q.astype(np.float32) * np.float32(1.0 / 64.0)).view(np.uint32)
    return img


def arm_seq_image(seq_id, waypoints):
    """One slot image (uint32 [260]) from [(dt_ms, (5 deg)), ...]."""
    img = np.zeros(260, dtype=np.uint32)
    img[0], img[1] = seq_id, len(waypoints)
    for k, (dt, deg) in enumerate(waypoints):
        img[4 + 8 * k] = dt
        img[5 + 8 * k : 10 + 8 * k] = np.asarray(deg, dtype=np.float32).view(np.uint32)
    return img


def vehicle_messages(n, n_seg, seed=0x5EED, first=0):
    """VDT::main message schedule (VD_task_main.hpp:8-60): [n_seg, n] rk_vdt_cmd_t records of kind
    RK_CMD_MSG_*: 5/8 REQ_MOVE_DIR (direction 0..12 incl. two undefined codes, speed 0 = default / up to 700
    = over the limit, time 0..1500 ms), 2/8 REQ_MOVE_CONT_DIR (vx, vy ~ U[-600, 600] mm/s, vth ~ U[-25, 25]
    rad/s: both limiters act; 1 in 16 is exactly zero), 1/8 nothing / an ignored MsgId."""
    inst = (np.arange(n, dtype=np.uint64) + np.uint64(first))[None, :]
    seg = np.arange(n_seg, dtype=np.uint64)[:, None]
    f32 = np.float32
    sel = (_hash(seed, 40, inst, seg) % np.uint64(8)).astype(np.int64)
    time_ms = (_hash(seed, 41, inst, seg) % np.uint64(1501)).astype(np.uint32)
    time_ms[(_hash(seed, 42, inst, seg) % np.uint64(6)) == 0] = 0
    d = (_hash(seed, 43, inst, seg) % np.uint64(13)).astype(np.uint32)
    spd = (_hash(seed, 44, inst, seg) % np.uint64(701)).astype(np.uint32)
    spd[(_hash(seed, 45, inst, seg) % np.uint64(5)) == 0] = 0
    vx = _u01(_hash(seed, 46, inst, seg)) * f32(1200.0) - f32(600.0)
    vy = _u01(_hash(seed, 47, inst, seg)) * f32(1200.0) - f32(600.0)
    vth = _u01(_hash(seed, 48, inst, seg)) * f32(50.0) - f32(25.0)
    zero = (_hash(seed, 49, inst, seg) % np.uint64(16)) == 0
    vx, vy = np.where(zero, f32(0), vx), np.where(zero, f32(0), vy)
    cmd = np.zeros((n_seg, n), dtype=np.dtype([("vx", "<f4"), ("vy", "<f4"), ("vth", "<f4"), ("kind", "<i4")]))
    is_dir, is_cont, is_unk = sel < 5, (sel == 5) | (sel == 6), (sel == 7) & (time_ms % 2 == 1)
    cmd["vx"] = np.where(is_dir, d.view(np.float32), np.where(is_cont, vx, f32(0)))
    cmd["vy"] = np.where(is_dir, spd.view(np.float32), np.where(is_cont, vy, f32(0)))
    cmd["vth"] = np.where(is_cont, vth, f32(0))
    kind = np.where(is_dir, _cabi.RK_CMD_MSG_MOVE_DIR, np.where(is_cont, _cabi.RK_CMD_MSG_MOVE_CONT_DIR,
                                                               np.where(is_unk, _cabi.RK_CMD_MSG_UNKNOWN, 0))).astype(np.uint32)
    cmd["kind"] = (kind | np.where(kind != 0, time_ms << np.uint32(8), np.uint32(0))).view(np.int32)
    return cmd


# ---- WIT serial wire (lib/wt901c/wit_c_sdk.c:132-164: 0x55, type, 4 x LE int16, byte-sum) ----------
WIT_ACC, WIT_GYRO, WIT_ANGLE, WIT_MAGNETIC, WIT_QUATER, WIT_REGVALUE = 0x51, 0x52, 0x53, 0x54, 0x59, 0x5F


def wit_frame(ftype, d):
    """One 11-byte WIT frame: header 0x55, type, four little-endian int16, checksum = byte sum of the first ten."""
    b = [0x55, int(ftype) & 0xFF]
    for v in d:
        v = int(v) & 0xFFFF
        b += [v & 0xFF, v >> 8]
    return bytes(b + [sum(b) & 0xFF])


def imu_wire_clean(regs, ncells=4):
    """The byte stream a healthy WT901C would send for the register snapshots `regs` (int16 [K, 16, n], as
    imu_samples): per update the five frames ACC, GYRO, ANGLE, MAGNETIC, QUATER (4th words: TEMP / VERSION = 0),
    55 bytes.  Returns (cells uint32 [K, ncells, n, 4], nbytes uint16 [K, n]) in rk_imt_feed_bytes layout."""
    K, _, n = regs.shape
    assert ncells * 16 >= 55
    b = np.zeros((K, ncells * 16, n), dtype=np.uint8)
    r = regs.astype(np.int16).view(np.uint16)
    plan = ((WIT_ACC, (0, 1, 2, None)), (WIT_GYRO, (3, 4, 5, None)), (WIT_ANGLE, (9, 10, 11, None)),
            (WIT_MAGNETIC, (6, 7, 8, None)), (WIT_QUATER, (12, 13, 14, 15)))
    for f, (t, slots) in enumerate(plan):
        o = 11 * f
        b[:, o, :], b[:, o + 1, :] = 0x55, t
        for k, s in enumerate(slots):
            if s is not None:
                b[:, o + 2 + 2 * k, :] = r[:, s, :] & 0xFF
                b[:, o + 3 + 2 * k, :] = r[:, s, :] >> 8
        b[:, o + 10, :] = b[:, o : o + 10, :].astype(np.uint32).sum(axis=1).astype(np.uint8)
    return _pack_wire(b), np.full((K, n), 55, dtype=np.uint16)


def _pack_wire(b):
    """uint8 [K, 16*ncells, n] (wire order) -> uint32 [K, ncells, n, 4]: 128-bit cells, first byte in the low byte."""
    K, nb, n = b.shape
    q = b.reshape(K, nb // 16, 4, 4, n).astype(np.uint32)  # [K, cell, word, byte, n]
    w = q[:, :, :, 0] | (q[:, :, :, 1] << 8) | (q[:, :, :, 2] << 16) | (q[:, :, :, 3] << 24)  # [K, cell, word, n]
    return np.ascontiguousarray(w.transpose(0, 1, 3, 2))


def imu_wire_fuzz(n, K, ncells=4, seed=0x5EED, first=0, full_slots=False):
    """Adversarial serial traffic: per IMU one continuous byte stream cut into K updates of 0 .. 16*ncells bytes
    (1 update in 8 sees an idle line; full_slots: every update carries exactly 16*ncells bytes), so frames straddle
    update boundaries.  Items: valid frames of every type CopeWitData knows (0x50..0x5A, 0x5F) and of unknown
    types, frames with a broken checksum, truncated frames, 0x55 runs, zeros and random garbage; data words are
    biased towards 0x55 bytes so that false headers occur inside payloads.  The stream always opens with a valid
    quaternion frame inside update 0 (IMU_IF_WT901C::init() spins until one arrives).
    Returns (cells uint32 [K, ncells, n, 4], nbytes uint16 [K, n])."""
    cap = 16 * ncells
    out = np.zeros((n, K, cap), dtype=np.uint8)
    nbytes = np.zeros((K, n), dtype=np.uint16)
    for i in range(n):
        rng = np.random.default_rng([int(seed) & 0xFFFFFFFF, int(first) + i, 0x317])
        if full_slots:
            lens = np.full(K, cap, dtype=np.int64)
        else:
            lens = rng.integers(0, cap + 1, size=K)
            lens[rng.integers(0, 8, size=K) == 0] = 0
            lens[0] = rng.integers(11, cap + 1)
        total = int(lens.sum())
        buf = bytearray()

        def words():
            w = rng.integers(-32768, 32768, size=4)
            m = rng.integers(0, 8, size=4)
            w = np.where(m == 0, 0x5555, np.where(m == 1, (w & 0xFF00) | 0x55, w))
            return [int(x) for x in w]

        buf += wit_frame(WIT_QUATER if rng.integers(0, 2) else WIT_REGVALUE, words())
        while len(buf) < total:
            kind = int(rng.integers(0, 16))
            if kind < 8:
                t = (WIT_ACC, WIT_GYRO, WIT_ANGLE, WIT_MAGNETIC, WIT_QUATER, WIT_QUATER, WIT_QUATER, WIT_REGVALUE)[kind]
                buf += wit_frame(t, words())
            elif kind == 8:
                buf += wit_frame(int(rng.integers(0x50, 0x5B)), words())
            elif kind == 9:
                buf += wit_frame(int(rng.integers(0, 256)), words())
            elif kind == 10:  # broken checksum
                f = bytearray(wit_frame(WIT_QUATER, words()))
                f[int(rng.integers(2, 11))] ^= 1 << int(rng.integers(0, 8))
                buf += f
            elif kind == 11:  # truncated frame
                buf += wit_frame(WIT_QUATER, words())[: int(rng.integers(1, 11))]
            elif kind == 12:
                buf += bytes([0x55] * int(rng.integers(1, 14)))
            elif kind == 13:
                buf += bytes(int(x) for x in rng.integers(0, 256, size=int(rng.integers(1, 24))))
            else:
                buf += bytes(int(rng.integers(1, 20)))
        o = 0
        for u in range(K):
            out[i, u, : lens[u]] = np.frombuffer(bytes(buf[o : o + lens[u]]), dtype=np.uint8)
            # bytes past the count are junk the engine must not look at
            out[i, u, lens[u] :] = rng.integers(0, 256, size=cap - lens[u])
            o += int(lens[u])
        nbytes[:, i] = lens
    return _pack_wire(np.ascontiguousarray(out.transpose(1, 2, 0))), nbytes


# ---- RobotManager cycles (src/RobotManager/RM_task_main.cpp:484-767) ----------------------------------
def rm_inputs(n, K, seed=0x5EED, first=0, idle_every=4):
    """Manager cycles: uint32 [K, 3, n, 4] rk_rmt_guard input records (RK_RI_* words in three 128-bit cells).

    Per cycle one of: nothing (45 %; robots with index % idle_every == 0 stay silent for 3/4 of their cycles
    so the 200-cycle watchdog fires), MecanumCommand (direction 0..12 incl. undefined codes, time 0..1500,
    speed 0..700), MecanumContOrder (mm/s doubles: U[-600, 600], 1 in 8 below the 0.01 dead band on both axes, 1 in
    8 exactly on a heading k * pi/50 so sector edges are probed, doubles that do not fit a float exactly), cmd_vel
    Twist (m/s), Command (RELAX, MOVE_READY, MOVE_START x3, QUIT_PG, INIT, HW_DEBUG, SWITCH_FLOOR_SENSOR, 77).
    Floor sensors: 70 % floor, 15 % nothing, 15 % wall per sensor; 1 cycle in 16 is mostly-nothing / mostly-wall."""
    inst = (np.arange(n, dtype=np.uint64) + np.uint64(first))[None, :]
    u = np.arange(K, dtype=np.uint64)[:, None]
    sel = (_hash(seed, 60, inst, u) % np.uint64(100)).astype(np.int64)
    silent = ((inst % np.uint64(idle_every)) == 0) & ((_hash(seed, 61, inst, u // np.uint64(300)) % np.uint64(4)) != 0)
    kind = np.where(sel < 45, 0, np.where(sel < 65, 1, np.where(sel < 80, 2, np.where(sel < 88, 3, 4))))
    kind = np.where(silent, 0, kind).astype(np.uint32)
    w = np.zeros((K, n, 12), dtype=np.uint32)
    w[..., 0] = kind
    d = (_hash(seed, 62, inst, u) % np.uint64(13)).astype(np.uint32)
    tm = (_hash(seed, 63, inst, u) % np.uint64(1501)).astype(np.uint32)
    sp = (_hash(seed, 64, inst, u) % np.uint64(701)).astype(np.uint32)
    cmds = np.array([0, 1, 2, 2, 2, 3, 4, 5, 10, 77], dtype=np.uint32)
    command = cmds[(_hash(seed, 65, inst, u) % np.uint64(len(cmds))).astype(np.int64)]
    w[..., 1] = np.where(kind == 1, d, np.where(kind == 2, tm, np.where(kind == 4, command, 0)))
    w[..., 2] = np.where(kind == 1, tm, 0)
    w[..., 3] = np.where(kind == 1, sp, 0)
    def u53(stream):  # full-mantissa uniform doubles in [0, 1)
        return (_hash(seed, stream, inst, u) >> np.uint64(11)).astype(np.float64) * (1.0 / 9007199254740992.0)
    vx, vy, vz = u53(66) * 1200.0 - 600.0, u53(67) * 1200.0 - 600.0, u53(68) * 50.0 - 25.0
    mode = (_hash(seed, 69, inst, u) % np.uint64(8)).astype(np.int64)
    tiny = mode == 0
    vx, vy = np.where(tiny, vx * 1e-5, vx), np.where(tiny, vy * 1e-5, vy)
    edge = mode == 1
    k50 = (_hash(seed, 70, inst, u) % np.uint64(101)).astype(np.float64) - 50.0
    r = 50.0 + u53(71) * 400.0
    vx, vy = np.where(edge, r * np.cos(k50 * np.pi / 50.0), vx), np.where(edge, r * np.sin(k50 * np.pi / 50.0), vy)
    axis = mode == 2  # on an axis: one component exactly zero
    vx = np.where(axis & (sel % 2 == 0), 0.0, vx)
    vy = np.where(axis & (sel % 2 == 1), 0.0, vy)
    scale = np.where(kind == 3, 1e-3, 1.0)
    for k, v in ((4, vx * scale), (6, vy * scale), (8, vz)):
        bits = np.ascontiguousarray(v).view(np.uint64)
        w[..., k] = np.where(kind >= 2, bits & np.uint64(0xFFFFFFFF), 0).astype(np.uint32)
        w[..., k + 1] = np.where((kind == 2) | (kind == 3), bits >> np.uint64(32), 0).astype(np.uint32)
    w[..., 4:10] = np.where(((kind == 2) | (kind == 3))[..., None], w[..., 4:10], 0)
    s = np.arange(8, dtype=np.uint64)[None, None, :]
    fsel = (_hash(seed, 72, inst[..., None] * np.uint64(8) + s, u[..., None]) % np.uint64(100)).astype(np.int64)
    fl = np.where(fsel < 70, 1, np.where(fsel < 85, 0, 2)).astype(np.uint32)
    bulk = (_hash(seed, 73, inst, u) % np.uint64(16)).astype(np.int64)
    bsel = (_hash(seed, 74, inst[..., None] * np.uint64(8) + s, u[..., None]) % np.uint64(8)).astype(np.int64)
    fl = np.where((bulk == 0)[..., None] & (bsel < 6), 0, fl)
    fl = np.where((bulk == 1)[..., None] & (bsel < 6), 2, fl).astype(np.uint32)
    w[..., 10] = fl[..., 0] | (fl[..., 1] << 8) | (fl[..., 2] << 16) | (fl[..., 3] << 24)
    w[..., 11] = fl[..., 4] | (fl[..., 5] << 8) | (fl[..., 6] << 16) | (fl[..., 7] << 24)
    return np.ascontiguousarray(w.reshape(K, n, 3, 4).transpose(0, 2, 1, 3))


# ---- v2 streams: the same distributions on a 32-bit counter hash -------------------------------------------------
# The generators above hash with splitmix64 three times per value: fine on the host, but a rollout engine that is fed
# over PCIe is bound by the host link (4.5 KB of tables per robot for the full tick), so the bench's workload is
# generated ON THE DEVICE from a 48-byte descriptor (csrc/rk_stream.cu, rk_stream_* in include/robotick.h).  These
# numpy restatements are the definition; the device kernels must reproduce them bit for bit
# (tests/test_streams_gpu.py).  All float32 results come from exactly representable integers or single IEEE float32 /
# float64 operations in a fixed order.
_U32 = np.uint32


def mix32(x):
    """32-bit finaliser (two odd multiplies, three xor-shifts)."""
    x = np.asarray(x, dtype=np.uint32)
    with np.errstate(over="ignore"):
        x = x ^ (x >> _U32(16))
        x = x * _U32(0x7FEB352D)
        x = x ^ (x >> _U32(15))
        x = x * _U32(0x846CA68B)
        x = x ^ (x >> _U32(16))
    return x


def h32(seed, stream, inst, idx):
    """Counter hash of (seed, stream, instance, index); instance and index are taken modulo 2^32."""
    with np.errstate(over="ignore"):
        h = mix32(_U32(int(seed) & 0xFFFFFFFF) ^ (_U32(stream) * _U32(0x9E3779B9)))
        h = mix32(h ^ (np.asarray(inst, dtype=np.uint64) & np.uint64(0xFFFFFFFF)).astype(np.uint32))
        h = mix32(h ^ ((np.asarray(idx, dtype=np.uint64) & np.uint64(0xFFFFFFFF)).astype(np.uint32) * _U32(0x85EBCA6B)))
    return h


def sub32(h, k):
    """k-th draw under one hash."""
    with np.errstate(over="ignore"):
        return mix32(np.asarray(h, dtype=np.uint32) + _U32(((k + 1) * 0x9E3779B9) & 0xFFFFFFFF))


def lite32(h, k):
    """k-th draw under one (already mixed) hash at a fraction of sub32's cost: the 64-bit product with an odd per-draw
    constant, high half folded onto the low half (one wide multiply and one xor on the device).  The per-sample streams
    (IMU registers, arm waypoints) use it; 16.8 M robots x 100 samples are expanded per pass."""
    m = np.uint64(((0x85EBCA6B + 2 * (k + 1) * 0x9E3779B9) | 1) & 0xFFFFFFFF)
    x = np.asarray(h, dtype=np.uint32).astype(np.uint64) * m
    return ((x & np.uint64(0xFFFFFFFF)) ^ (x >> np.uint64(32))).astype(np.uint32)


def _u01_32(h):
    """24-bit uniform in [0,1) as exact float32."""
    return (np.asarray(h, dtype=np.uint32) >> _U32(8)).astype(np.float32) * np.float32(1.0 / 16777216.0)


def _inst(n, first, inst):
    return (np.arange(n, dtype=np.uint64) + np.uint64(first)) if inst is None else np.asarray(inst, dtype=np.uint64)


def vehicle_commands_v2(n, n_seg, seed=0x5EED, first=0, stop_every=8, inst=None):
    """vehicle_commands() on the 32-bit hash.  `inst` (optional): explicit global instance indices instead of
    first .. first + n - 1 (spot checks generate just the sampled robots)."""
    inst = _inst(n, first, inst)[None, :]
    seg = np.arange(n_seg, dtype=np.uint64)[:, None]
    f32 = np.float32
    b = h32(seed, 1, inst, seg)
    vx = _u01_32(sub32(b, 0)) * f32(800.0) - f32(400.0)
    vy = _u01_32(sub32(b, 1)) * f32(800.0) - f32(400.0)
    vth = _u01_32(sub32(b, 2)) * f32(4.0 * np.pi) - f32(2.0 * np.pi)
    ln = np.sqrt(vx * vx + vy * vy, dtype=np.float32)
    lim = np.minimum(ln, f32(400.0))
    nz = ln != 0
    safe = np.where(nz, ln, f32(1.0))
    vx = np.where(nz, (vx * lim) / safe, f32(0.0)).astype(np.float32)
    vy = np.where(nz, (vy * lim) / safe, f32(0.0)).astype(np.float32)
    rl = f32(6.0 * np.pi)
    vth = np.clip(vth, -rl, rl).astype(np.float32)
    stop = (sub32(b, 3) % _U32(stop_every)) == 0
    cmd = np.zeros(b.shape, dtype=np.dtype([("vx", "<f4"), ("vy", "<f4"), ("vth", "<f4"), ("kind", "<i4")]))
    cmd["vx"] = np.where(stop, f32(0), vx)
    cmd["vy"] = np.where(stop, f32(0), vy)
    cmd["vth"] = np.where(stop, f32(0), vth)
    cmd["kind"] = np.where(stop, _cabi.RK_CMD_STOP, _cabi.RK_CMD_MOVE)
    return cmd


def vehicle_yaw_reg_v2(n, n_yaw, seed=0x5EED, first=0, inst=None):
    """vehicle_yaw_reg() on the 32-bit hash: int16 [n_yaw, n]."""
    inst = _inst(n, first, inst)[None, :]
    k = np.arange(n_yaw, dtype=np.int64)[:, None]
    b = h32(seed, 5, inst, 0)
    phase = (sub32(b, 0) & _U32(0xFFFF)).astype(np.int64)
    rate = ((sub32(b, 1) % _U32(5)).astype(np.int64) + 1) * 182
    sign = np.where((sub32(b, 2) & _U32(1)) == 0, 1, -1)
    return ((phase + sign * rate * k) & 0xFFFF).astype(np.uint16).view(np.int16)


def imu_samples_v2(n, n_upd, seed=0x5EED, first=0, drop_every=64, inst=None, first_update=0):
    """imu_samples() on the 32-bit hash: int16 [n_upd, 16, n] (+ have_quat uint8 [n_upd, n]).  One hash per
    (IMU, update); its lite32 draws 0-5 are AX..Yaw two registers a word, 6-7 four 16-bit uniforms in (-1, 1) normalised in
    float32 (IEEE sqrt / division, fixed order) to a unit quaternion x 32767 (rounded half to even), 8 the
    missing-quaternion-frame flag."""
    inst = _inst(n, first, inst)[None, :]
    u = (np.arange(n_upd, dtype=np.uint64) + np.uint64(first_update))[:, None]
    b = h32(seed, 20, inst, u)  # [n_upd, n]
    regs = np.zeros((n_upd, 16, b.shape[1]), dtype=np.int16)
    for k in range(6):
        w = lite32(b, k)
        regs[:, 2 * k, :] = (w & _U32(0xFFFF)).astype(np.uint16).view(np.int16)
        regs[:, 2 * k + 1, :] = (w >> _U32(16)).astype(np.uint16).view(np.int16)
    w6, w7 = lite32(b, 6), lite32(b, 7)
    f32 = np.float32
    g = [((x.astype(np.float32) + f32(0.5)) * f32(1.0 / 32768.0)) - f32(1.0) for x in (w6 & _U32(0xFFFF), w6 >> _U32(16), w7 & _U32(0xFFFF), w7 >> _U32(16))]
    nrm = np.sqrt(((g[0] * g[0] + g[1] * g[1]) + g[2] * g[2]) + g[3] * g[3], dtype=np.float32)
    sc = f32(32767.0) / nrm
    for k in range(4):
        regs[:, 12 + k, :] = np.rint(g[k] * sc).astype(np.int16)
    if drop_every:
        have = ((lite32(b, 8) % _U32(drop_every)) != 0).astype(np.uint8)
    else:
        have = np.ones(b.shape, dtype=np.uint8)
    return regs, np.ascontiguousarray(have)


def arm_sequences_v2(n, seed=0x5EED, first=0, max_len=32, min_len=2, seq_id=1, dt_zero_every=4, inst=None):
    """arm_sequences() on the 32-bit hash: uint32 [n, 260] slot images; waypoints past the sequence length are zero."""
    inst = _inst(n, first, inst)
    m = len(inst)
    k = np.arange(32, dtype=np.uint64)[None, :]
    b0 = h32(seed, 30, inst, 0)
    ln = (sub32(b0, 0) % _U32(max_len - min_len + 1)).astype(np.int64) + min_len
    z = (sub32(b0, 1) % _U32(dt_zero_every)) == 0
    b = h32(seed, 31, inst[:, None], k)  # [m, 32]
    inc = (lite32(b, 0) % _U32(991)).astype(np.int64) + 10
    inc[(lite32(b, 1) % _U32(8)) == 0] = 0
    inc[z, 0] = 0
    dt = np.cumsum(inc, axis=1)
    img = np.zeros((m, 260), dtype=np.uint32)
    img[:, 0] = seq_id
    img[:, 1] = ln
    wp = img[:, 4:].reshape(m, 32, 8)
    wp[:, :, 0] = dt.astype(np.uint32)
    for j in range(5):
        q = (lite32(b, 2 + j) % _U32(300 * 64 + 1)).astype(np.int64) - 150 * 64
        wp[:, :, 1 + j] = (q.astype(np.float32) * np.float32(1.0 / 64.0)).view(np.uint32)
    wp[np.arange(32)[None, :] >= ln[:, None]] = 0
    return img


def plan_xi_v2(h):
    """The candidate noise of plan_commands_v2 under hash(es) h: float32 [..., 3] Irwin-Hall draws (four uniforms of lite32
    draws 4a .. 4a+3 for axis a, summed left to right, centred and scaled to unit variance)."""
    f32 = np.float32
    xi = []
    for a in range(3):
        u = [_u01_32(lite32(h, 4 * a + k)) for k in range(4)]
        xi.append((((u[0] + u[1]) + u[2]) + u[3] - f32(2.0)) * f32(1.7320508))
    return np.stack(xi, axis=-1).astype(np.float32)


def plan_commands_v2(nominal, S, seed=0x5EED, first=0, sigma=(100.0, 100.0, 1.0), params=None):
    """Sampling-planner candidates around a nominal plan (rk_plan_sample_commands): nominal [n_seg, R] rk_vdt_cmd_t records
    -> [n_seg, R*S], candidate j of robot r at column r*S + j.  Candidate 0 is the nominal; candidate j > 0 of segment s adds
    sigma_a * xi_a with xi = plan_xi_v2(h32(seed, 40, first + r, s*S + j)).  Then the vehicle's limiters (params: the
    rk_vdt_params_t, default firmware constants): |(vx, vy)| above limit_speed_mmps is scaled back onto it as
    (v * L) / |v|, vth is clamped to +-limit_rot_radps; kind = RK_CMD_MOVE.  float32, one rounding per operation."""
    p = params or _cabi.default_params()
    f32 = np.float32
    nominal = np.asarray(nominal)
    if nominal.dtype.names is None:  # int32 / float32 [n_seg, R, 4] cells
        cells = np.ascontiguousarray(nominal).view(np.uint32)
        nominal = cells.view(np.dtype([("vx", "<f4"), ("vy", "<f4"), ("vth", "<f4"), ("kind", "<i4")])).reshape(cells.shape[:2])
    n_seg, R = nominal.shape
    inst = (np.arange(R, dtype=np.uint64) + np.uint64(first))[None, :, None]
    idx = np.arange(n_seg, dtype=np.uint64)[:, None, None] * np.uint64(S) + np.arange(S, dtype=np.uint64)[None, None, :]
    xi = plan_xi_v2(h32(seed, 40, inst, idx))  # [n_seg, R, S, 3]
    v = []
    for a, name in enumerate(("vx", "vy", "vth")):
        nom = np.broadcast_to(nominal[name].astype(np.float32)[:, :, None], (n_seg, R, S))
        noisy = (nom + f32(sigma[a]) * xi[..., a]).astype(np.float32)
        noisy[:, :, 0] = nom[:, :, 0]  # j == 0: the nominal itself
        v.append(noisy)
    vx, vy, vth = v
    L, rl = f32(p.limit_speed_mmps), f32(p.limit_rot_radps)
    ln = np.sqrt(vx * vx + vy * vy, dtype=np.float32)
    over = ln > L
    safe = np.where(over, ln, f32(1.0))
    vx = np.where(over, (vx * L) / safe, vx).astype(np.float32)
    vy = np.where(over, (vy * L) / safe, vy).astype(np.float32)
    vth = np.where(vth > rl, rl, np.where(vth < -rl, -rl, vth)).astype(np.float32)
    cmd = np.zeros((n_seg, R * S), dtype=np.dtype([("vx", "<f4"), ("vy", "<f4"), ("vth", "<f4"), ("kind", "<i4")]))
    cmd["vx"], cmd["vy"], cmd["vth"] = vx.reshape(n_seg, -1), vy.reshape(n_seg, -1), vth.reshape(n_seg, -1)
    cmd["kind"] = _cabi.RK_CMD_MOVE
    return cmd
