"""GPU parity: ADTModePositioning kernels (rk_adp_*) vs the oracle port / compiled reference."""
import numpy as np
import pytest
import torch

import oracle_lib as ol
from roboken_fmskf_robot_controller_b200 import layout
from roboken_fmskf_robot_controller_b200.arm import ArmBatch, ArmPositioningBatch
from test_armpos_cpu import bringup_state, pos_script, run_pos_script

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def gpu_pos_script(n, script, astate, trace=True):
    """The script's outputs; without `trace` each update's trace output is None (the kernel runs untraced)."""
    ab = ArmBatch(n, DEV)
    ab.load_state_soa(astate)
    pb = ArmPositioningBatch(ab)
    outs = []
    for step in script:
        if step[0] == "init":
            pb.mode_init()
        elif step[0] == "push":
            pb.push_cmd(torch.from_numpy(step[1].view(np.int32)).to(DEV), None if step[2] is None else torch.from_numpy(step[2]).to(DEV))
        elif step[0] == "update":
            tr = torch.zeros((step[1], layout.ADT_TRACE_WORDS, n), dtype=torch.int32, device=DEV) if trace else None
            pb.update(step[1], tr)
            outs.append(tr.cpu().numpy().view(np.uint32) if trace else None)
        elif step[0] == "status":
            outs.append(pb.cmd_status(torch.from_numpy(np.asarray(step[1], dtype=np.uint32).view(np.int32)).to(DEV)).cpu().numpy())
        torch.cuda.synchronize()
        outs += [ab.state_host().copy(), pb.pstate.cpu().numpy().view(np.uint32)]
    return outs


_POS_CASES = [(1, 1), (300, 2), (4100, 3)]


# Untraced runs launch the kernel instantiations without a trace; they are held to the state blocks after every step.
@pytest.mark.parametrize("n,seed,trace", [(n, s, True) for n, s in _POS_CASES] + [(n, s, False) for n, s in _POS_CASES],
                         ids=[f"{n}-{s}" for n, s in _POS_CASES] + [f"{n}-{s}-untraced" for n, s in _POS_CASES])
def test_positioning_mode_vs_port(n, seed, trace):
    st0 = bringup_state(n, seed)
    sc = pos_script(n, seed)
    got, exp = gpu_pos_script(n, sc, st0, trace), run_pos_script("port", n, sc, st0)[2]
    assert len(got) == len(exp)
    for k, (x, y) in enumerate(zip(got, exp)):
        if x is not None:
            np.testing.assert_array_equal(x, y, err_msg=f"output {k}")


def test_positioning_mode_vs_compiled_reference():
    n = 48
    st0 = bringup_state(n, 9)
    sc = pos_script(n, 9)
    got = gpu_pos_script(n, sc, st0)
    exp = ol.reference_result("armpos_gpu", lambda kind: run_pos_script(kind, n, sc, st0), "libref_arm.so")[2]
    for k, (x, y) in enumerate(zip(got, exp)):
        np.testing.assert_array_equal(x, y, err_msg=f"output {k}")
