"""GPU parity: the arm kernels behind the C-ABI (rk_adt_*) vs the oracle port / compiled
reference / golden fixture.  Everything here is integer state or float words compared as bits."""
import os

import numpy as np
import pytest
import torch

import oracle_lib as ol
from roboken_fmskf_robot_controller_b200 import _cabi, layout, streams
from roboken_fmskf_robot_controller_b200.arm import DONE, NO_DATA, PROCESSING, Arm, ArmBatch
from test_arm_cpu import fresh, random_arm_states, run_script

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def gpu_script(n, script, state=None, tab=None):
    ab = ArmBatch(n, DEV)
    if state is not None:
        ab.load_state_soa(state, tab)
    outs = []
    for step in script:
        if step[0] == "init":
            ab.mode_init()
        elif step[0] == "push":
            seq = torch.from_numpy(layout.aos_to_soa(step[1]).view(np.int32)).to(DEV)
            ab.push_cmdseq(seq, None if step[2] is None else torch.from_numpy(step[2]).to(DEV))
        elif step[0] == "update":
            tr = torch.zeros((step[1], layout.ADT_TRACE_WORDS, n), dtype=torch.int32, device=DEV)
            ab.update(step[1], tr)
            outs.append(tr.cpu().numpy().view(np.uint32))
        elif step[0] == "status":
            ids = torch.from_numpy(np.asarray(step[1], dtype=np.uint32).view(np.int32)).to(DEV)
            outs.append(ab.cmdseq_status(ids).cpu().numpy())
        torch.cuda.synchronize()
        outs.append(ab.state_host().copy())
    return ab.state_host(), ab.cmdtab_host(), outs


def assert_same(a, b):
    assert len(a[2]) == len(b[2])
    for x, y in zip(a[2], b[2]):
        np.testing.assert_array_equal(x, y)
    np.testing.assert_array_equal(a[0], b[0])
    np.testing.assert_array_equal(a[1], b[1])


def test_arm_golden_fixture():
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "arm_golden.npz"))
    n = int(g["n"])
    script = [("init",), ("push", g["seq_a"], None), ("push", g["seq_b"], g["valid_b"]), ("update", int(g["K"])),
              ("status", g["ids"])]
    st, tb, outs = gpu_script(n, script)
    np.testing.assert_array_equal(outs[-4], g["trace"])
    np.testing.assert_array_equal(outs[-2], g["status"])
    np.testing.assert_array_equal(st, g["state"])
    np.testing.assert_array_equal(tb, g["cmdtab"])


@pytest.mark.parametrize("n,seed", [(1, 1), (257, 2), (4099, 3)])
def test_arm_random_sequences_vs_port(n, seed):
    s1 = streams.arm_sequences(n, seed=seed, seq_id=1, max_len=8)
    s2 = streams.arm_sequences(n, seed=seed + 50, seq_id=2, max_len=6)
    valid = (np.arange(n) % 3 != 0).astype(np.uint8)
    script = [("init",), ("push", s1, None), ("update", 37), ("push", s2, valid), ("status", np.full(n, 1)),
              ("update", 300), ("status", np.full(n, 2)), ("status", np.full(n, 7))]
    assert_same(gpu_script(n, script), run_script("port", n, script))


def test_arm_ring_overflow_and_id0_vs_port():
    n = 8
    seqs = [streams.arm_sequences(n, seed=10 + k, seq_id=k, max_len=3) for k in range(6)]
    script = [("init",), ("status", np.zeros(n)), ("push", seqs[0], None), ("status", np.zeros(n)), ("update", 1),
              ("status", np.zeros(n))]
    for k in range(1, 6):
        script += [("push", seqs[k], None)] + [("status", np.full(n, j)) for j in range(6)]
    script += [("update", 900)] + [("status", np.full(n, j)) for j in range(6)]
    script += [("push", seqs[5], None), ("update", 5)] + [("status", np.full(n, j)) for j in range(6)]
    assert_same(gpu_script(n, script), run_script("port", n, script))


def test_arm_random_states_vs_port():
    n = 3000
    st0 = random_arm_states(n, seed=4)
    taos = np.zeros((n, layout.ACMD_WORDS), dtype=np.uint32)
    for s in range(4):
        taos[:, s * 260 : (s + 1) * 260] = streams.arm_sequences(n, seed=20 + s, seq_id=s + 1, max_len=5)
    tab = layout.aos_to_soa(taos)
    script = [("update", 3), ("status", np.full(n, 2)), ("update", 120)]
    assert_same(gpu_script(n, script, st0, tab), run_script("port", n, script, st0, tab))


@pytest.mark.parametrize("mg_any", [False, True])
def test_arm_untraced_launches_of_any_length_vs_port(mg_any):
    """The kernel WITHOUT a trace attached (what rk_tick_rollout and the bench launch) forms values nobody can read inside
    a launch lazily -- the MG position frame once after the last tick, targets of axes 1..4 on ticks that end a segment and
    on the last two ticks, the torque-edge logic from the second tick on.  Launch lengths 1, 2, 3, ... from random mid-move
    states (and with MG joints in every control branch) must leave the same block as the port after every launch."""
    n = 2500
    st0 = random_arm_states(n, seed=11, mg_any_branch=mg_any)
    taos = np.zeros((n, layout.ACMD_WORDS), dtype=np.uint32)
    for s in range(4):
        taos[:, s * 260 : (s + 1) * 260] = streams.arm_sequences(n, seed=40 + s, seq_id=s + 1, max_len=6)
    tab = layout.aos_to_soa(taos)
    ab = ArmBatch(n, DEV)
    ab.load_state_soa(st0, tab)
    es, et = st0.copy(), tab.copy()
    for K in (1, 1, 2, 3, 2, 5, 1, 17, 64, 2, 1, 200):
        ab.update(K)
        torch.cuda.synchronize()
        ol.arm_batch("port", "update", es, et, n, K=K)
        np.testing.assert_array_equal(ab.state_host(), es, err_msg=f"after a launch of {K} ticks")
    np.testing.assert_array_equal(ab.cmdtab_host(), et)


def test_mg_torque_control_branches_vs_port():
    """Every flag combination of the MG joint: PI_D reset on the torque-off edge, torque control while not
    initialised / limp (CMSIS sine, double-precision current->raw map), position control."""
    n = 2048
    st0 = random_arm_states(n, seed=6, mg_any_branch=True)
    taos = np.zeros((n, layout.ACMD_WORDS), dtype=np.uint32)
    for s in range(4):
        taos[:, s * 260 : (s + 1) * 260] = streams.arm_sequences(n, seed=30 + s, seq_id=s + 1, max_len=4)
    tab = layout.aos_to_soa(taos)
    script = [("update", 1), ("update", 2), ("update", 60)]
    assert_same(gpu_script(n, script, st0, tab), run_script("port", n, script, st0, tab))


def test_arm_extreme_waypoints_vs_port():
    wp = [(0, (170, 10, 10, 10, 10)), (50, (-190, 20, -20, 5, 5)), (50, (140, 0, 0, 0, 0)), (40, (0, 0, 0, 0, 0)),
          (45, (100, -100, 100, -100, 100))]
    img = np.stack([streams.arm_seq_image(3, wp), streams.arm_seq_image(4, []), streams.arm_seq_image(5, wp[:2])])
    script = [("init",), ("push", img, None), ("update", 40), ("status", [3, 4, 5]), ("update", 40)]
    assert_same(gpu_script(3, script), run_script("port", 3, script))


def test_arm_mg_velocity_division_domains_vs_port():
    """The MG velocity limit divides the per-tick target step by the control period through the exact reciprocal form
    only where rk_exact.cu proves it (0 and 2^-40 <= |step| <= 2^64 for 0.01 s); J1 targets that make the step tiny,
    denormal, huge or overflowing (quotient = inf) must take the IEEE division and still match the port bit for bit.  (A step
    that is itself inf - inf is left out: NaN payloads differ between x86 and the GPU.)"""
    mags = [0.0, 1e-45, 1e-38, 1e-30, 3e-13, 9.2e-13, 1e-6, 1.0, 1e6, 1e18, 1.9e19, 3e19, 1e30, 1e37]
    imgs = []
    for k, m in enumerate(mags):
        wp = [(10, (0, m, 0, 0, 0)), (20, (0, -m, 0, 0, 0)), (40, (0, m * 0.5, 0, 0, 0)), (50, (0, 0, 0, 0, 0))]
        imgs.append(streams.arm_seq_image(7, wp))
    img = np.stack(imgs)
    script = [("init",), ("push", img, None), ("update", 12)]
    assert_same(gpu_script(len(mags), script), run_script("port", len(mags), script))


def test_arm_vs_compiled_reference():
    n = 64
    s1 = streams.arm_sequences(n, seed=77, seq_id=5, max_len=10)
    script = [("init",), ("push", s1, None), ("update", 250), ("status", np.full(n, 5))]
    assert_same(gpu_script(n, script), ol.reference_result("arm_gpu", lambda kind: run_script(kind, n, script), "libref_arm.so"))


def test_arm_full_size_c4():
    """BASELINE.json configs[3]: 2^20 arms, one sequence each, K = 1000 fused ticks.  Sampled
    bit-exact parity + size-independent properties: every finished arm sits exactly on its last
    waypoint (the interpolation's final step has zero remaining count) and reports DONE."""
    n, K = 1 << 20, 1000
    seq = streams.arm_sequences(n, seed=0xC4, seq_id=9, max_len=32)
    ab = ArmBatch(n, DEV)
    ab.mode_init()
    ab.push_cmdseq(torch.from_numpy(layout.aos_to_soa(seq).view(np.int32)).to(DEV))
    ab.update(K)
    torch.cuda.synchronize()
    st = layout.soa_to_aos(ab.state_host(), n, layout.AS_WORDS)
    status = ab.cmdseq_status(torch.full((n,), 9, dtype=torch.int32, device=DEV)).cpu().numpy()
    idx = np.unique(np.random.default_rng(0).integers(0, n, 400))
    es, et = fresh(len(idx))
    ol.arm_batch("port", "init", es, et, len(idx))
    ol.arm_batch("port", "push", es, et, len(idx), seq=layout.aos_to_soa(seq[idx]))
    ol.arm_batch("port", "update", es, et, len(idx), K=K)
    np.testing.assert_array_equal(st[idx], layout.soa_to_aos(es, len(idx), layout.AS_WORDS))
    ln = seq[:, 1].astype(np.int64)
    done = (st[:, layout.AS_CMD_IDX] & 0xFF) >= ln  # the status query's criterion with one sequence in the ring
    assert done.sum() > n // 20 and (~done).sum() > n // 20
    np.testing.assert_array_equal(status[done], DONE)
    np.testing.assert_array_equal(status[~done], PROCESSING)
    last = seq[:, 4:].reshape(n, 32, 8)[np.arange(n), ln - 1, 1:6].view(np.float32)
    tgt = np.stack([st[:, layout.AS_JOINT0 + 4 * k + layout.AJ_RAW_TGT].view(np.float32) for k in layout.ADT_AXIS], axis=1)
    np.testing.assert_array_equal(tgt[done], last[done])  # offsets are zero: raw target == commanded angle


def test_arm_single_instance_handle_debug_2():
    """POS_CMD_SEQ_DEBUG_2 (AD_mode_positioning_seq_debug_data.cpp:43-64) through the handle API."""
    wp = [(0, (0, 120, -90, 0, 45)), (1000, (20, 60, -30, 45, -60)), (2000, (-20, 90, 0, 0, 0)), (3000, (0, 120, -60, 0, 45))]
    arm = Arm()
    arm.init()
    assert arm.get_q_cmdseq_status(0) == NO_DATA
    arm.push_cmdseq(0, wp)
    assert arm.get_q_cmdseq_status(0) == NO_DATA  # isModeFirstCall && id == 0
    arm.update()
    assert arm.get_q_cmdseq_status(0) == PROCESSING
    arm.update()  # dt = 0: a one-cycle move, reached on the second tick
    np.testing.assert_array_equal(arm.get_tgt_deg(), np.float32([0, 120, -90, 0, 45]))
    for _ in range(101):  # MOVE_START + 100 cycles
        arm.update()
    np.testing.assert_array_equal(arm.get_tgt_deg(), np.float32([20, 60, -30, 45, -60]))
    for _ in range(2 * 101):
        arm.update()
    assert arm.get_q_cmdseq_status(0) == DONE  # u8_nowcmd_idx_ == len
    arm.update()
    np.testing.assert_array_equal(arm.get_tgt_deg(), np.float32([0, 120, -60, 0, 45]))
    assert arm.get_state()[layout.AS_FSM] & 0xFF == layout.ASTATE_STANDBY
    st, tb = fresh(1)
    ol.arm_batch("port", "init", st, tb, 1)
    ol.arm_batch("port", "push", st, tb, 1, seq=streams.arm_seq_image(0, wp))
    ol.arm_batch("port", "update", st, tb, 1, K=2 + 3 * 101 + 1)
    np.testing.assert_array_equal(arm.get_state(), st)
    arm.close()


def test_shared_reciprocal_division_is_ieee():
    """div_by_rcp64 (the arm tick's five per-segment divisions by one count) == div.rn.f32: 2^32 pseudo-random (x, c)
    pairs on the device -- every bit pattern class of x; c alternately an arbitrary float and an integer 1 .. 2^24."""
    import ctypes as C

    from roboken_fmskf_robot_controller_b200 import _cabi

    bad = C.c_uint32(123)
    _cabi.check(_cabi.load().rk_selftest_div_rcp64(1 << 32, 2024, C.byref(bad)))
    assert bad.value == 0
