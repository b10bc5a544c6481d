"""GPU parity of the VDT::main command layer inside rk_vdt_rollout (RK_CMD_MSG_* records, speed limiters,
move-time auto-stop with task_period = 10) against the oracle port and the reference's whole vehicle task
(VD_task_main.cpp compiled unmodified)."""
import numpy as np
import pytest

import oracle_lib as ol
import roboken_fmskf_robot_controller_b200 as rk
from roboken_fmskf_robot_controller_b200 import _cabi, layout
from test_vdt_task_cpu import run, task_inputs
from test_vehicle_gpu import assert_same, gpu_run

pytestmark = pytest.mark.gpu


def gpu_task(inp, trace=True):
    return gpu_run(dict(inp, task_period=10), trace=trace)


@pytest.mark.parametrize("n,steps,seed,seg_len", [(1, 300, 1, 50), (700, 1200, 2, 30), (2100, 1000, 3, 200)])
def test_task_layer_vs_port(n, steps, seed, seg_len):
    inp = task_inputs(n, steps, seed, seg_len=seg_len)
    st, tr = gpu_task(inp)
    pst, ptr = run("port", inp)
    assert_same(tr, ptr, "task-layer trace vs port")
    assert_same(st, pst, "task-layer state vs port")


def test_task_layer_vs_reference_task():
    inp = task_inputs(96, 1500, 7, seg_len=70)
    st, tr = gpu_task(inp)
    rst, rtr = ol.reference_result("vdt_task_gpu", lambda kind: run(kind, inp), "libref_vdt_task.so")
    assert_same(tr, rtr, "task-layer trace vs the compiled VDT task")
    assert_same(st, rst, "task-layer state vs the compiled VDT task")


def test_task_layer_fast_equals_transcription_and_chunked():
    """The countdown's data-dependent stop tick splits the fast kernel's chunks; the transcription kernel and a
    rollout resumed in five launches (countdown carried in the state block) must give the same bits."""
    lib = rk.load()
    inp = task_inputs(1500, 1000, 11, seg_len=100)
    st, tr = gpu_task(inp)
    lib.rk_set_option(_cabi.RK_OPT_FORCE_TRANSCRIPTION, 1)
    try:
        st2, tr2 = gpu_task(inp)
    finally:
        lib.rk_set_option(_cabi.RK_OPT_FORCE_TRANSCRIPTION, 0)
    assert_same(tr, tr2, "fast vs transcription trace")
    assert_same(st, st2, "fast vs transcription state")
    st3, _ = gpu_run(dict(inp, task_period=10), trace=False, chunks=5)
    # microsecond ids restart per launch (dead telemetry word); mask it out of the compare
    a1, a3 = layout.soa_to_aos(st, inp["n"], layout.VS_WORDS), layout.soa_to_aos(st3, inp["n"], layout.VS_WORDS)
    for w in range(4):
        a1[:, layout.VS_MOTOR0 + 8 * w + layout.VM_USEC] &= 0xFFFF0000
        a3[:, layout.VS_MOTOR0 + 8 * w + layout.VM_USEC] &= 0xFFFF0000
    assert_same(a1, a3, "one launch vs five")
    st4, _ = gpu_task(inp, trace=False)
    assert_same(st, st4, "trace off")
