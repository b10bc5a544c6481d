#!/usr/bin/env python3
"""One planning step of the vehicle sampling planner at size: R robots x S candidates, n_seg segments of seg_len ticks.

Times (CUDA events) rk_plan_sample_commands, rk_plan_rollout and rk_plan_select, and, alternated with the plan rollout in
the same run, a plain rk_vdt_rollout of the same candidates on the S-fold forked state block (the fork is rewritten
before every plain rollout, outside the timed window).  Prints one JSON line with the device name and power limit.

With --obstacles M (M > 0 discs per robot; a comma list or repeated) the same run also times rk_plan_rollout_obstacles
for every M and every --check-period P (default seg_len), each alternated with rk_plan_rollout on the same candidates,
and reports obst_over_plan.  The discs are seeded around the robots' positions, within the candidates' reach, so that
part of the candidates enter them.

    python tools/bench_plan.py [--R 4096] [--S 256] [--n-seg 8] [--seg-len 125] [--reps 10] [--out FILE]
                               [--obstacles 1,8 --check-period 125,25,10]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import roboken_fmskf_robot_controller_b200 as rk  # noqa: E402
from roboken_fmskf_robot_controller_b200 import _cabi, layout, streams  # noqa: E402
from roboken_fmskf_robot_controller_b200.planner import VehiclePlanner  # noqa: E402
from roboken_fmskf_robot_controller_b200.vehicle import VehicleBatch  # noqa: E402


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return out or "unknown"
    except Exception:
        return "unknown"


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    b.synchronize()
    return a.elapsed_time(b)


def int_list(args):
    return [int(x) for a in args for x in str(a).split(",") if x != ""]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--R", type=int, default=4096)
    ap.add_argument("--S", type=int, default=256)
    ap.add_argument("--n-seg", type=int, default=8)
    ap.add_argument("--seg-len", type=int, default=125)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    ap.add_argument("--obstacles", action="append", default=[], help="discs per robot (comma list or repeated; 0: none)")
    ap.add_argument("--check-period", action="append", default=[], help="obstacle check period in ticks (comma list or repeated)")
    a = ap.parse_args()
    obst_m = [m for m in int_list(a.obstacles) if m > 0]
    obst_p = int_list(a.check_period) or [a.seg_len]
    if not torch.cuda.is_available():
        sys.exit("bench_plan.py needs a CUDA device")
    dev = "cuda:0"
    R, S, n_seg, seg_len = a.R, a.S, a.n_seg, a.seg_len
    n, K = R * S, n_seg * seg_len

    # R robots in mid-move: two segments of stream commands from power-on
    nominal = torch.from_numpy(streams.vehicle_commands_v2(R, n_seg, seed=17, stop_every=1 << 30).view(np.int32)).reshape(n_seg, R, 4).to(dev)
    src = VehicleBatch(R, dev)
    src.rollout(2 * seg_len, sensor_mode=_cabi.RK_SENSOR_PLANT, cmd=nominal[:2].contiguous(), seg_len=seg_len)
    goal = torch.from_numpy(np.random.default_rng(3).uniform(-0.3, 0.3, (R, 2)).astype(np.float32)).to(dev)
    ref = goal.unsqueeze(0).expand(n_seg, R, 2).contiguous()
    pl = VehiclePlanner(R, S, n_seg, seg_len, dev)
    plain = VehicleBatch(n, dev)
    src_planes = src.state.view(layout.VS_WORDS // 4, R, 4)

    def fork():
        plain.state.view(layout.VS_WORDS // 4, n, 4).copy_(src_planes.repeat_interleave(S, dim=1))

    def sample():
        pl.sample(nominal=nominal, seed=5)

    def plan_rollout():
        pl.rollout(src, ref, 1.0, 10.0, 1e-9)

    def select():
        pl.select(0.0, 1)

    def plain_rollout():
        plain.rollout(K, sensor_mode=_cabi.RK_SENSOR_PLANT, cmd=pl.candidates, seg_len=seg_len)

    # keep-out discs: centres within 0.15 m of each robot's position, radii 20 - 80 mm (the candidates travel up to
    # 0.4 m in 1000 ticks)
    discs = {}
    if obst_m:
        aos = layout.soa_to_aos(src.state.cpu().numpy().view(np.uint32), R, layout.VS_WORDS)
        pos = aos[:, [layout.VS_POS_X, layout.VS_POS_Y]].view(np.float32)
        rng = np.random.default_rng(11)
    for m in obst_m:
        d = np.zeros((m, R, 4), dtype=np.float32)
        d[:, :, :2] = pos[None] + rng.uniform(-0.15, 0.15, (m, R, 2))
        d[:, :, 2] = rng.uniform(0.02, 0.08, (m, R))
        discs[m] = torch.from_numpy(d).to(dev)

    def obst_rollout(m, P):
        pl.rollout(src, ref, 1.0, 10.0, 1e-9, obstacles=discs[m], w_obst=1e3, check_period=P)

    # warm-up: every shape once (the first rollout also runs the fast path's on-device proofs)
    sample(), plan_rollout(), select(), fork(), plain_rollout()
    for m in obst_m:
        for P in obst_p:
            obst_rollout(m, P)
    torch.cuda.synchronize()
    src_before = src.state.clone()
    t = {"sample": [], "plan_rollout": [], "select": [], "plain_rollout": []}
    t_obst = {}
    for _ in range(a.reps):
        t["sample"].append(timed(sample))
        t["plan_rollout"].append(timed(plan_rollout))
        t["select"].append(timed(select))
        fork()
        torch.cuda.synchronize()
        t["plain_rollout"].append(timed(plain_rollout))
        for m in obst_m:
            for P in obst_p:  # alternated with the plan rollout of the same candidates
                tp, to = t_obst.setdefault((m, P), ([], []))
                tp.append(timed(plan_rollout))
                to.append(timed(lambda: obst_rollout(m, P)))
    assert torch.equal(src.state, src_before), "the plan rollout modified its source states"
    med = {k: float(np.median(v)) for k, v in t.items()}
    res = {
        "bench": "plan_step",
        "device": torch.cuda.get_device_name(0),
        "power_limit": power_limit(),
        "R": R, "S": S, "candidates": n, "n_seg": n_seg, "seg_len": seg_len, "ticks": K, "reps": a.reps,
        "ms_median": {k: round(v, 4) for k, v in med.items()},
        "ms_min": {k: round(float(np.min(v)), 4) for k, v in t.items()},
        "ms_max": {k: round(float(np.max(v)), 4) for k, v in t.items()},
        "plan_candidate_steps_per_s": n * K / (med["plan_rollout"] * 1e-3),
        "plain_candidate_steps_per_s": n * K / (med["plain_rollout"] * 1e-3),
        "plan_over_plain": med["plan_rollout"] / med["plain_rollout"],
        "sample_plus_select_over_rollout": (med["sample"] + med["select"]) / med["plan_rollout"],
        "step_ms": med["sample"] + med["plan_rollout"] + med["select"],
    }
    if obst_m:
        plan_rollout()
        plan_cost = pl.cost.clone()
        rows = []
        for (m, P), (tp, to) in t_obst.items():
            obst_rollout(m, P)
            hit = (pl.cost != plan_cost).float().mean().item()  # candidates with O > 0
            mp, mo = float(np.median(tp)), float(np.median(to))
            rows.append({"m": m, "check_period": P, "ms_median_plan": round(mp, 4), "ms_median_obst": round(mo, 4),
                         "ms_min_obst": round(float(np.min(to)), 4), "ms_max_obst": round(float(np.max(to)), 4),
                         "obst_over_plan": mo / mp, "penetrating_fraction": hit})
        res["obstacles"] = rows
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
