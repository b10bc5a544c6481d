"""SURVEY 8f-3, arm side on the device: rk_adt_bldc_rx / rk_adt_mg_rx against the port (every frame, the Cortex-M7
reading of the MG multi-turn angle included) and against the reference's own rx callbacks compiled for x86 (frames on
which the two architectures agree)."""
import numpy as np
import pytest
import torch

import oracle_lib as ol
from roboken_fmskf_robot_controller_b200.arm import ArmBatch
from test_armrx_cpu import rx_cases

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def gpu_rx(state, n, frames, cmdid):
    ab = ArmBatch(n, DEV)
    ab.state.copy_(torch.from_numpy(state.view(np.int32)))
    curs = []
    for which in range(4):
        cur = torch.full((n,), 123.25, dtype=torch.float32, device=DEV)
        fr = torch.from_numpy(frames[which].view(np.int64)).to(DEV)
        if which < 3:
            ab.bldc_rx(which, fr, torch.from_numpy(cmdid.view(np.int32)).to(DEV), cur)
        else:
            ab.mg_rx(fr, cur)
        curs.append(cur.cpu().numpy())
    torch.cuda.synchronize()
    return ab.state.cpu().numpy().view(np.uint32), curs


def host_rx(kind, state, n, frames, cmdid):
    st = state.copy()
    curs = []
    for which in range(4):
        cur = np.full(n, 123.25, dtype=np.float32)
        ol.arm_rx(kind, which, st, n, frames[which], cmdid if which < 3 else None, cur)
        curs.append(cur)
    return st, curs


@pytest.mark.parametrize("n,seed,upper_zero", [(5000, 11, False), (1, 12, False), (3333, 13, True)])
def test_rx_vs_port(n, seed, upper_zero):
    state, frames, cmdid = rx_cases(n, seed, mg_upper_zero=upper_zero)
    gst, gcur = gpu_rx(state, n, frames, cmdid)
    pst, pcur = host_rx("port", state, n, frames, cmdid)
    np.testing.assert_array_equal(gst, pst)
    for a, b in zip(gcur, pcur):
        np.testing.assert_array_equal(a.view(np.uint32), b.view(np.uint32))


def test_rx_vs_compiled_reference():
    n = 4096
    state, frames, cmdid = rx_cases(n, 21, mg_upper_zero=True)
    gst, gcur = gpu_rx(state, n, frames, cmdid)
    rst, rcur = ol.reference_result("armrx_gpu", lambda kind: host_rx(kind, state, n, frames, cmdid), "libref_arm.so")
    np.testing.assert_array_equal(gst, rst)
    for a, b in zip(gcur, rcur):
        np.testing.assert_array_equal(a.view(np.uint32), b.view(np.uint32))


def test_rx_none_optionals_and_feedback_into_homing_words():
    """cmdid / cur may be NULL; the angle the decoder stores is the fl_raw_now_deg word the homing modes read."""
    from roboken_fmskf_robot_controller_b200 import layout

    n = 64
    state, frames, _ = rx_cases(n, 31)
    ab = ArmBatch(n, DEV)
    ab.state.copy_(torch.from_numpy(state.view(np.int32)))
    ab.bldc_rx(1, torch.from_numpy(frames[1].view(np.int64)).to(DEV))
    ab.mg_rx(torch.from_numpy(frames[3].view(np.int64)).to(DEV))
    torch.cuda.synchronize()
    st = state.copy()
    ol.arm_rx("port", 1, st, n, frames[1])
    ol.arm_rx("port", 3, st, n, frames[3])
    np.testing.assert_array_equal(ab.state.cpu().numpy().view(np.uint32), st)
    a = layout.soa_to_aos(st, n, layout.AS_WORDS)
    assert (a[:, layout.AS_JOINT0 + 4 * 3 + 3] != layout.soa_to_aos(state, n, layout.AS_WORDS)[:, layout.AS_JOINT0 + 4 * 3 + 3]).any()
