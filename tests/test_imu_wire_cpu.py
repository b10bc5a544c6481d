"""CPU: pin the WIT serial codec of the plain-C oracle (orc_imt_feed_bytes) against the compiled reference --
the vendor parser lib/wt901c/wit_c_sdk.c and IMU_IF_WT901C::init/update, both unmodified -- on clean and on
adversarial byte streams (SURVEY 8f-3)."""
import os

import numpy as np
import pytest

import oracle_lib as ol
from roboken_fmskf_robot_controller_b200 import layout, streams

GOLD = os.path.join(os.path.dirname(__file__), "golden", "imu_wire_golden.npz")


def parser_sreg(parser_soa, n):
    """The 16 tracked sReg words of every IMU out of the RK_IP_* block: int16 [n, 16]."""
    a = layout.soa_to_aos(parser_soa, n, layout.IP_WORDS)[:, layout.IP_SREG : layout.IP_SREG + 8]
    return np.ascontiguousarray(a).view(np.int16).reshape(n, 16)


def wire_run(kind, n, cells, nbytes):
    """Raw bytes into the IMU from power-on (update 0 is init()): (out, state, sReg int16 [n, 16]), port or compiled reference."""
    st = np.zeros(layout.IS_WORDS * n, dtype=np.uint32)
    if kind == "ref":
        out, sreg = ol.imu_bytes_ref(st, n, cells, nbytes, want_out=True)
        return out, st, sreg
    ps = np.zeros(layout.IP_WORDS * n, dtype=np.uint32)
    out = ol.imu_bytes_port(st, ps, n, cells, nbytes, want_out=True, do_init=True)
    return out, st, parser_sreg(ps, n)


def test_wit_frame_checksum():
    f = streams.wit_frame(streams.WIT_QUATER, [1, -2, 0x1234, -32768])
    assert len(f) == 11 and f[0] == 0x55 and f[1] == 0x59 and f[10] == sum(f[:10]) & 0xFF
    assert f[2:10] == bytes([1, 0, 0xFE, 0xFF, 0x34, 0x12, 0x00, 0x80])


def test_clean_wire_equals_register_path():
    """The five frames of a healthy sensor give exactly what the register-level entry gives."""
    n, K = 50, 12
    regs, _ = streams.imu_samples(n, K, seed=11)
    cells, nbytes = streams.imu_wire_clean(regs)
    a = np.zeros(layout.IS_WORDS * n, dtype=np.uint32)
    oa = ol.imu_port(a, n, regs, None, want_out=True, do_init=True)
    b, pb = np.zeros(layout.IS_WORDS * n, dtype=np.uint32), np.zeros(layout.IP_WORDS * n, dtype=np.uint32)
    ob, yaw = ol.imu_bytes_port(b, pb, n, cells, nbytes, want_out=True, want_yaw=True, do_init=True)
    np.testing.assert_array_equal(oa, ob)
    np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(parser_sreg(pb, n), regs[-1].T)
    ang_yaw = ob.view(np.float32)[:, 2, :, 3]  # Data word 11 = angle[2]
    np.testing.assert_array_equal(yaw, (ang_yaw * streams.DEG2RAD).astype(np.float32))


@pytest.mark.parametrize("n,K,ncells,seed,full", [(64, 24, 4, 1, False), (48, 40, 1, 2, False), (32, 10, 16, 3, False),
                                                   (40, 64, 1, 4, True), (24, 12, 3, 5, True)])
def test_port_equals_ref_fuzzed_wire(n, K, ncells, seed, full):
    cells, nbytes = streams.imu_wire_fuzz(n, K, ncells=ncells, seed=seed, full_slots=full)
    if full:
        nbytes = None
    a, pa = np.zeros(layout.IS_WORDS * n, dtype=np.uint32), np.zeros(layout.IP_WORDS * n, dtype=np.uint32)
    oa = ol.imu_bytes_port(a, pa, n, cells, nbytes, want_out=True, do_init=True)
    ob, b, sreg = ol.reference_result(f"imu_wire_fuzz_{seed}", lambda kind: wire_run(kind, n, cells, nbytes), "libref_imu.so")
    np.testing.assert_array_equal(oa, ob)
    np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(parser_sreg(pa, n), sreg)
    # the stream exercised both outcomes of isComComp()
    err = layout.soa_to_aos(a, n, layout.IS_WORDS)[:, layout.IS_FLAGS] & 1
    assert 0 < err.sum() < n


def test_port_chunked_equals_ref_one_pass():
    """Parser state carried across calls (window, fill count, read index, sReg) == one uninterrupted replay."""
    n, K, ncells = 40, 30, 2
    cells, nbytes = streams.imu_wire_fuzz(n, K, ncells=ncells, seed=9)
    a, pa = np.zeros(layout.IS_WORDS * n, dtype=np.uint32), np.zeros(layout.IP_WORDS * n, dtype=np.uint32)
    outs, k0 = [], 0
    for k1 in (1, 2, 9, 10, 23, 30):
        outs.append(ol.imu_bytes_port(a, pa, n, np.ascontiguousarray(cells[k0:k1]), np.ascontiguousarray(nbytes[k0:k1]),
                                      want_out=True, do_init=(k0 == 0)))
        k0 = k1
    ob, b, sreg = ol.reference_result("imu_wire_one_pass", lambda kind: wire_run(kind, n, cells, nbytes), "libref_imu.so")
    np.testing.assert_array_equal(np.concatenate(outs), ob)
    np.testing.assert_array_equal(a, b)
    np.testing.assert_array_equal(parser_sreg(pa, n), sreg)


def test_false_header_resync_known_answer():
    """Hand-built stream: garbage with a false 0x55 header, then a frame.  The parser slides one byte per
    incoming byte (wit_c_sdk.c:139-144,148-153) and must still find the frame."""
    q = streams.wit_frame(streams.WIT_QUATER, [16384, 0, 0, 0])
    acc = streams.wit_frame(streams.WIT_ACC, [2048, -1024, 512, 77])
    raw = q + bytes([0x55, 0x51, 1, 2, 3]) + acc + bytes(3)
    nb = np.array([[len(raw)]], dtype=np.uint16)
    raw += bytes([0xEE] * (-len(raw) % 16))  # junk past the count
    cells = np.frombuffer(raw, dtype="<u4").reshape(1, len(raw) // 16, 1, 4).copy()
    st, ps = np.zeros(layout.IS_WORDS, dtype=np.uint32), np.zeros(layout.IP_WORDS, dtype=np.uint32)
    out = ol.imu_bytes_port(st, ps, 1, cells, nb, want_out=True, do_init=True)
    d = out.view(np.float32).reshape(16)
    # the false header swallowed the real header: 0x55 0x51 01 02 03 55 51 00 08 00 fc | sum mismatch -> slide
    sreg = parser_sreg(ps, 1)[0]
    assert list(sreg[12:16]) == [16384, 0, 0, 0]
    assert list(sreg[0:3]) == [2048, -1024, 512]
    assert d[0] == 1.0 and d[1] == 0.5 and d[2] == -0.25


def test_golden_imu_wire():
    g = np.load(GOLD)
    n, K, ncells = 48, 20, 2
    cells, nbytes = streams.imu_wire_fuzz(n, K, ncells=ncells, seed=0x5EED)
    np.testing.assert_array_equal(cells, g["cells"])
    np.testing.assert_array_equal(nbytes, g["nbytes"])
    st, ps = np.zeros(layout.IS_WORDS * n, dtype=np.uint32), np.zeros(layout.IP_WORDS * n, dtype=np.uint32)
    out = ol.imu_bytes_port(st, ps, n, cells, nbytes, want_out=True, do_init=True)
    np.testing.assert_array_equal(out, g["out"])
    np.testing.assert_array_equal(st, g["state"])
    np.testing.assert_array_equal(parser_sreg(ps, n), g["sreg"])


def late_quaternion_wire(n, K, seed):
    """Healthy traffic (five frames per update) in which the FIRST quaternion frame is late for most IMUs: the
    quaternion frame of updates 0 .. late-1 never makes it onto the wire (44 bytes instead of 55), so
    IMU_IF_WT901C::init() -- update slot 0 -- keeps waiting in getDataImmediately() through those slots."""
    regs, _ = streams.imu_samples(n, K, seed=seed)
    cells, nb = streams.imu_wire_clean(regs, ncells=4)
    late = np.arange(n) % 4  # 0: on time, 1..3: that many slots late
    for i in range(n):
        nb[: late[i], i] = 44
    return cells, nb, late


def test_init_waits_for_a_late_first_quaternion_frame_like_the_reference():
    """ADVICE r1: init() must not latch q_init (or publish) before its first quaternion frame.  Port == the compiled
    reference, whose blocking init() is fed the following update slots while it spins."""
    n, K = 64, 12
    cells, nb, late = late_quaternion_wire(n, K, 77)
    out_r, st_r, sreg_r = ol.reference_result("imu_wire_late_quaternion", lambda kind: wire_run(kind, n, cells, nb), "libref_imu.so")
    st_p, ps_p = np.zeros(layout.IS_WORDS * n, dtype=np.uint32), np.zeros(layout.IP_WORDS * n, dtype=np.uint32)
    out_p = ol.imu_bytes_port(st_p, ps_p, n, cells, nb, want_out=True, do_init=True)
    np.testing.assert_array_equal(out_p, out_r)
    np.testing.assert_array_equal(st_p, st_r)
    np.testing.assert_array_equal(parser_sreg(ps_p, n), sreg_r)
    # nothing is published while init() waits, and q_init is the quaternion of the frame that ended the wait
    o = np.ascontiguousarray(out_p.transpose(0, 2, 1, 3)).reshape(K, n, 16)
    for i in range(n):
        assert not o[: late[i], i].any() and o[late[i], i].any()
    regs, _ = streams.imu_samples(n, K, seed=77)
    qi = layout.soa_to_aos(st_p, n, layout.IS_WORDS)[:, :4].view(np.float32)
    for i in range(n):
        np.testing.assert_array_equal(qi[i], regs[late[i], 12:16, i].astype(np.float32) / np.float32(32768.0))


def test_pending_init_is_carried_across_launches_port():
    """The wait survives a launch boundary: slots 0..1 in one call (no quaternion frame), the rest in the next."""
    n, K = 32, 8
    cells, nb, late = late_quaternion_wire(n, K, 78)
    st_a, ps_a = np.zeros(layout.IS_WORDS * n, dtype=np.uint32), np.zeros(layout.IP_WORDS * n, dtype=np.uint32)
    out_a = ol.imu_bytes_port(st_a, ps_a, n, cells, nb, want_out=True, do_init=True)
    st_b, ps_b = np.zeros(layout.IS_WORDS * n, dtype=np.uint32), np.zeros(layout.IP_WORDS * n, dtype=np.uint32)
    o1 = ol.imu_bytes_port(st_b, ps_b, n, np.ascontiguousarray(cells[:2]), np.ascontiguousarray(nb[:2]), want_out=True, do_init=True)
    pend = layout.soa_to_aos(ps_b, n, layout.IP_WORDS)[:, 3] & 0x10000
    assert ((pend != 0) == (late >= 2)).all()
    o2 = ol.imu_bytes_port(st_b, ps_b, n, np.ascontiguousarray(cells[2:]), np.ascontiguousarray(nb[2:]), want_out=True, do_init=False)
    np.testing.assert_array_equal(np.concatenate([o1, o2]), out_a)
    np.testing.assert_array_equal(st_b, st_a)
    np.testing.assert_array_equal(ps_b, ps_a)
