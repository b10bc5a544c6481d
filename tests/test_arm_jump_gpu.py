"""GPU parity of the untraced arm launch where it jumps over ticks (loop_jump in rk_arm.cu): the inside of a positioning
segment in one step, and the idle ticks after a finished queue.  The ICS joint (J0) is the only servo that looks at the
target inside a segment, so its waypoints are chosen to move the target across the bounds of its position word
(about +-135 deg) and of its degree range (+-180 deg) in the middle of segments, in both directions, and out of the range
of its integer conversion (3e7 deg; 3e38 deg, where the conversion overflows to +-inf), which runs tick by tick.  The
states are random (ICS servo connected or not, torque on or off, mid-move FSMs), segments run from one tick (dt = 0) to
longer than a launch, and each arm's sequences are shifted by its own number of ticks, so that the launch lengths end
before, on and after the final tick of segments.  Every launch must leave the same block as the port.  (J0 waypoints of
+-inf are left out: the interpolation then forms inf - inf, and NaN payloads differ between x86 and the GPU.)"""
import numpy as np
import pytest
import torch

import oracle_lib as ol
from roboken_fmskf_robot_controller_b200 import layout, streams
from roboken_fmskf_robot_controller_b200.arm import ArmBatch
from test_arm_cpu import random_arm_states

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

J0_PATHS = [
    [0.0, 170.0, -170.0, 200.0, -200.0, 0.0],
    [140.0, 140.0, -140.0, 185.0, -185.0, 134.0, 136.0],
    [0.0, 3e7, 0.0, -3e7, 0.0],
    [0.0, 3e38, 0.0, -3e38, 0.0],
    [-179.0, 179.0, -90.0],
    [100.0],
]
SEG_MS = [0, 0, 10, 20, 450, 1000, 3000]  # at the default 10 ms tick: 1 tick, 1, 2, 45, 100, 300 ticks
LAUNCHES = (1, 2, 3, 44, 45, 46, 1, 7, 100, 299, 300, 301, 2, 1000, 1, 500, 3)


def j0_ring(n, seed):
    rng = np.random.default_rng(seed)
    taos = np.zeros((n, layout.ACMD_WORDS), dtype=np.uint32)
    for i in range(n):
        for s in range(layout.ACMD_SLOTS):
            path = J0_PATHS[rng.integers(len(J0_PATHS))]
            t = 10 * (i % 61) if s == 0 else 0
            wp = []
            for x in path:
                wp.append((t, (x, rng.uniform(-90, 90), rng.uniform(-90, 90), rng.uniform(-90, 90), rng.uniform(-90, 90))))
                t += int(SEG_MS[rng.integers(len(SEG_MS))])
            img = streams.arm_seq_image(s + 1, wp)
            taos[i, s * layout.ACMD_SLOT_WORDS : (s + 1) * layout.ACMD_SLOT_WORDS] = img
    return layout.aos_to_soa(taos)


@pytest.mark.parametrize("seed", [1, 2])
def test_arm_jump_over_segments_and_idle_ticks_vs_port(seed):
    n = 2048
    st0 = random_arm_states(n, seed=100 + seed)
    tab = j0_ring(n, seed)
    ab = ArmBatch(n, DEV)
    ab.load_state_soa(st0, tab)
    es, et = st0.copy(), tab.copy()
    for K in LAUNCHES:
        ab.update(K)
        torch.cuda.synchronize()
        ol.arm_batch("port", "update", es, et, n, K=K)
        np.testing.assert_array_equal(ab.state_host(), es, err_msg=f"after a launch of {K} ticks")
    np.testing.assert_array_equal(ab.cmdtab_host(), et)
