#!/usr/bin/env python3
"""Where the kernels of rk_tick_rollout run relative to each other: a few chunks back to back on one or two lanes with
the library's diagnostic timestamps (rk_tick_debug_timeline), plus CUDA events around the caller-side setup kernels.

    python tools/tick_timeline.py [--n 1048576] [--chunks 4] [--lanes 2] [--side-ctas 0]"""
import argparse
import ctypes as C
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from roboken_fmskf_robot_controller_b200 import _cabi, layout  # noqa: E402
from roboken_fmskf_robot_controller_b200.devstreams import DeviceStreams  # noqa: E402
from roboken_fmskf_robot_controller_b200.robot import RobotBatch  # noqa: E402

ap = argparse.ArgumentParser()
ap.add_argument("--n", type=int, default=1 << 20)
ap.add_argument("--chunks", type=int, default=4)
ap.add_argument("--lanes", type=int, default=2)
ap.add_argument("--side-ctas", type=int, default=0)
ap.add_argument("--ticks", type=int, default=1000)
a = ap.parse_args()
dev = torch.device("cuda", 0)
lib = _cabi.load()
lib.rk_set_option(_cabi.RK_OPT_TICK_SIDE_CTAS, a.side_ctas)
n, T, slow = a.n, a.ticks, 10
n_seg, n_slow = (T + 124) // 125, (T + slow - 1) // slow
ds = DeviceStreams(dev, first_update=1)
cmd = ds.vehicle_commands(torch.empty((n_seg, n, 4), dtype=torch.int32, device=dev))
regs, have = ds.imu_samples(torch.empty((n_slow, 2, n, 8), dtype=torch.int16, device=dev), torch.empty((n_slow, n), dtype=torch.uint8, device=dev))
seq = ds.arm_sequences(torch.empty(layout.ACMD_SLOT_WORDS * n, dtype=torch.int32, device=dev))
lanes = [torch.cuda.Stream(dev) for _ in range(a.lanes)]
rbs, args = [], []
for c in range(a.chunks):
    rb = RobotBatch(n, dev)
    rb.imu.update(regs[:1].contiguous(), None, None, do_init=True)
    rbs.append(rb)
    args.append(rb.make_args(T, slow, cmd=cmd, seg_len=125, regs=regs, have_quat=have, yaw=torch.zeros(n, dtype=torch.float32, device=dev)))
main = torch.cuda.current_stream(dev)


def one_pass(timed):
    ev = []
    for ls in lanes:
        ls.wait_stream(main)
    for c, rb in enumerate(rbs):
        ls = lanes[c % len(lanes)]
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        e[0].record(ls)
        rb.arm.mode_init(stream=ls)
        rb.arm.push_cmdseq(seq, stream=ls)
        e[1].record(ls)
        rb.rollout_args(args[c], stream=ls)
        e[2].record(ls)
        ev.append(e)
    for ls in lanes:
        main.wait_stream(ls)
    return ev


one_pass(False)
one_pass(False)
torch.cuda.synchronize()
t0 = torch.cuda.Event(enable_timing=True)
t1 = torch.cuda.Event(enable_timing=True)
t0.record(main)
ev = one_pass(True)
t1.record(main)
torch.cuda.synchronize()
print(f"pass of {a.chunks} chunks x {n} robots x {T} ticks, lanes={a.lanes}, side_ctas={a.side_ctas}: {t0.elapsed_time(t1):.3f} ms")
for c, e in enumerate(ev):
    print(f"  chunk {c} lane {c % len(lanes)}: setup starts {t0.elapsed_time(e[0]):8.3f}  setup done {t0.elapsed_time(e[1]):8.3f}  tick (incl. join) done {t0.elapsed_time(e[2]):8.3f}")
# the library's own timestamps of ONE chunk run alone after the pass, then inside a pass of two
lib.rk_tick_debug_timeline(1, None)
out = (C.c_float * 5)()
rbs[0].rollout_args(args[0], stream=lanes[0])
lib.rk_tick_debug_timeline(1, out)
print("  one chunk alone     [side start, imu done, arm done, vehicle start, vehicle done] ms:", [round(x, 3) for x in out])
ev = one_pass(True)
lib.rk_tick_debug_timeline(0, out)
print("  last chunk of a pass [side start, imu done, arm done, vehicle start, vehicle done] ms:", [round(x, 3) for x in out])
