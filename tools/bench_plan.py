#!/usr/bin/env python3
"""One planning step of the vehicle sampling planner at size: R robots x S candidates, n_seg segments of seg_len ticks.

Times (CUDA events) rk_plan_sample_commands, rk_plan_rollout and rk_plan_select, and, alternated with the plan rollout in
the same run, a plain rk_vdt_rollout of the same candidates on the S-fold forked state block (the fork is rewritten
before every plain rollout, outside the timed window).  Prints one JSON line with the device name and power limit.

With --obstacles M (M > 0 discs per robot; a comma list or repeated) the same run also times rk_plan_rollout_obstacles
for every M and every --check-period P (default seg_len), each alternated with rk_plan_rollout on the same candidates,
and reports obst_over_plan.  The discs are seeded around the robots' positions, within the candidates' reach, so that
part of the candidates enter them.

With --cem ITERS:ELITE the run also times the two ends of a cross-entropy round, rk_plan_sample_commands_sigma and
rk_plan_refit (ELITE elites), each alternated with its counterpart rk_plan_sample_commands / rk_plan_select, and reports
them against the plan rollout.  Then, from the same robots, it plans --cem-steps closed-loop steps three ways at the same
rollout budget -- CEM with ITERS rounds of S / ITERS candidates, argmin and MPPI (--lam) over S candidates -- executing
the first segment of each new plan, and reports the last step's best cost and the final distance to the goal.

With --moving M:P (a comma list or repeated) the run also times, for every pair, rk_plan_rollout_moving with a table of
M discs per robot that differs at every checkpoint, alternated with rk_plan_rollout_obstacles at the same M and P and with
rk_plan_rollout_moving writing every candidate's path; then VehiclePlanner.predict (S = 1 over the R robots) and
rk_plan_peer_discs of fleets of --fleet G robots (default 8).  It reports moving_over_static and path_over_moving.

With --fleet G the run also plays the circle swap at size: R / G groups of G robots on a --fleet-circle (m) circle, each
heading for the antipodal point, with and without peer discs (radius 2 * --fleet-body + --fleet-margin, weight
--fleet-w, checked every --fleet-period ticks), under argmin (S candidates) and CEM (--cem ITERS:ELITE, default 4:8, at
the same rollout budget), for --fleet-steps steps.  It reports the share of groups in which two robots came closer than
2 * body radius, the median / minimum over groups of the least pairwise distance, and the median distance to the goal.

    python tools/bench_plan.py [--R 4096] [--S 256] [--n-seg 8] [--seg-len 125] [--reps 10] [--out FILE]
                               [--obstacles 1,8 --check-period 125,25,10] [--cem 4:8 --cem-steps 8 --lam 1e-3]
                               [--moving 1:125,8:25] [--fleet 8 --fleet-steps 60]
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
from roboken_fmskf_robot_controller_b200.planner import VehiclePlanner, fleet_peers  # noqa: E402
from roboken_fmskf_robot_controller_b200.vehicle import VehicleBatch  # noqa: E402


def power_limit(query="power.limit"):
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={query}", "--format=csv,noheader", "-i", str(torch.cuda.current_device())],
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


def compare_planners(a, src, goal, ref, iters, elite):
    """--cem-steps closed-loop steps from the robots in src (left untouched) for CEM (iters x S/iters, elite), argmin and
    MPPI (S candidates): the last step's best cost and the final distance to the goal, median and mean over the robots."""
    R, S, n_seg, seg_len, dev = a.R, a.S, a.n_seg, a.seg_len, src.state.device
    out = {}
    for name, s_step in (("cem", S // iters), ("argmin", S), ("mppi", S)):
        pl = VehiclePlanner(R, s_step, n_seg, seg_len, dev)
        vb = VehicleBatch(R, dev)
        vb.state.copy_(src.state)
        for step in range(a.cem_steps):
            if name == "cem":
                pl.plan_cem(vb, ref, 1.0, 10.0, 1e-9, iters, elite, seed=step)
            else:
                pl.plan(vb, ref, 1.0, 10.0, 1e-9, lam=a.lam if name == "mppi" else 0.0, seed=step)
            vb.rollout(seg_len, sensor_mode=_cabi.RK_SENSOR_PLANT, cmd=pl.first_command(), seg_len=seg_len)
        torch.cuda.synchronize()
        aos = layout.soa_to_aos(vb.state.cpu().numpy().view(np.uint32), R, layout.VS_WORDS)
        pos = aos[:, [layout.VS_POS_X, layout.VS_POS_Y]].view(np.float32).astype(np.float64)
        d = np.hypot(*(pos - goal.cpu().numpy()).T)
        bc = pl.best_cost.cpu().numpy().astype(np.float64)
        out[name] = {"rollouts_per_step": S if name != "cem" else iters * s_step,
                     "best_cost_median": float(np.median(bc)), "best_cost_mean": float(np.mean(bc)),
                     "goal_dist_m_median": float(np.median(d)), "goal_dist_m_mean": float(np.mean(d))}
    out["steps"], out["lam"] = a.cem_steps, a.lam
    return out


def circle_swap(R, G, circle, dev):
    """Start states and goals float32 [R, 2] of the circle swap: group g = r // G on a circle of radius `circle` around its
    own centre (a grid 3 circles apart), robot r at angle 2 pi (r % G) / G + 0.3 g, the goal at the antipodal point."""
    g = np.arange(R) // G
    side = int(np.ceil(np.sqrt(R // G + 1)))
    centre = 3.0 * circle * np.stack([g % side, g // side], axis=1).astype(np.float64)
    ang = 2.0 * np.pi * (np.arange(R) % G) / G + 0.3 * g
    u = np.stack([np.cos(ang), np.sin(ang)], axis=1)
    start, goal = (centre + circle * u).astype(np.float32), (centre - circle * u).astype(np.float32)
    aos = np.zeros((R, layout.VS_WORDS), dtype=np.uint32)
    aos[:, layout.VS_POS_X], aos[:, layout.VS_POS_Y] = start[:, 0].view(np.uint32), start[:, 1].view(np.uint32)
    vb = VehicleBatch(R, dev)
    vb.load_state_aos(aos)
    return vb, torch.from_numpy(goal).to(dev)


def fleet_report(a, G, dev):
    """The circle swap with and without peer discs, under argmin and CEM at the same rollout budget (see the docstring)."""
    R, S, n_seg, seg_len, P = a.R, a.S, a.n_seg, a.seg_len, a.fleet_period
    iters, elite = (int(x) for x in (a.cem or "4:8").split(":"))
    body, radius = a.fleet_body, 2 * a.fleet_body + a.fleet_margin
    peers = fleet_peers(R, G, dev)
    out = {"G": G, "groups": R // G, "circle_m": a.fleet_circle, "body_radius_m": body, "disc_radius_m": radius, "w_obst": a.fleet_w,
           "check_period": P, "steps": a.fleet_steps, "cem": {"iters": iters, "elite": elite}}
    for mode in ("argmin", "cem"):
        for avoid in (False, True):
            vb, goal = circle_swap(R, G, a.fleet_circle, dev)
            ref = goal.unsqueeze(0).expand(n_seg, R, 2).contiguous()
            pl = VehiclePlanner(R, S // iters if mode == "cem" else S, n_seg, seg_len, dev)
            tr = torch.zeros((seg_len, _cabi.RK_VDT_TRACE_WORDS, R), dtype=torch.int32, device=dev)
            least = torch.full((R // G,), float("inf"), dtype=torch.float64, device=dev)
            eye = torch.eye(G, dtype=torch.bool, device=dev)
            for step in range(a.fleet_steps):
                discs = None
                if avoid:
                    discs = pl.peer_discs(pl.predict(vb, check_period=P), peers, radius=radius)
                kw = dict(shift=0, seed=step, obstacles=discs, w_obst=a.fleet_w, check_period=P)
                if mode == "cem":
                    pl.plan_cem(vb, ref, 1.0, 10.0, 1e-9, iters, elite, **kw)
                else:
                    pl.plan(vb, ref, 1.0, 10.0, 1e-9, lam=0.0, **kw)
                vb.rollout(seg_len, sensor_mode=_cabi.RK_SENSOR_PLANT, cmd=pl.first_command(), seg_len=seg_len, trace=tr)
                pos = tr[:, :2].view(torch.float32).double().reshape(seg_len, 2, R // G, G)
                d = torch.hypot(pos[:, 0, :, :, None] - pos[:, 0, :, None, :], pos[:, 1, :, :, None] - pos[:, 1, :, None, :])
                least = torch.minimum(least, d.masked_fill(eye, float("inf")).amin(dim=(0, 2, 3)))
            aos = layout.soa_to_aos(vb.state.cpu().numpy().view(np.uint32), R, layout.VS_WORDS)
            pos = aos[:, [layout.VS_POS_X, layout.VS_POS_Y]].view(np.float32).astype(np.float64)
            dg = np.hypot(*(pos - goal.cpu().numpy()).T)
            lc = least.cpu().numpy()
            out[f"{mode}_{'peer_discs' if avoid else 'none'}"] = {
                "rollouts_per_step": S if mode == "argmin" else iters * (S // iters),
                "groups_with_collision": float(np.mean(lc < 2 * body)), "least_pair_m_median": float(np.median(lc)),
                "least_pair_m_min": float(np.min(lc)), "goal_dist_m_median": float(np.median(dg))}
    return out


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
    ap.add_argument("--cem", default=None, help="ITERS:ELITE: time the cross-entropy round's sampler and refit, and compare planners")
    ap.add_argument("--cem-steps", type=int, default=8, help="closed-loop planning steps of the planner comparison")
    ap.add_argument("--lam", type=float, default=1e-3, help="MPPI temperature of the planner comparison")
    ap.add_argument("--moving", action="append", default=[], help="M:P pairs (comma list or repeated): time moving discs and paths")
    ap.add_argument("--fleet", type=int, default=None, help="G: play the circle swap with fleets of G robots")
    ap.add_argument("--fleet-steps", type=int, default=60)
    ap.add_argument("--fleet-circle", type=float, default=1.0)
    ap.add_argument("--fleet-body", type=float, default=0.15)
    ap.add_argument("--fleet-margin", type=float, default=0.1)
    ap.add_argument("--fleet-w", type=float, default=1e3)
    ap.add_argument("--fleet-period", type=int, default=25)
    a = ap.parse_args()
    moving = [tuple(int(v) for v in x.split(":")) for arg in a.moving for x in arg.split(",") if x]
    cem_iters, cem_elite = (int(x) for x in a.cem.split(":")) if a.cem else (0, 0)
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

    # moving discs: a table per checkpoint, the discs of the static table moved by up to 20 mm per checkpoint
    mov, static_m = {}, {}
    if moving:
        aos = layout.soa_to_aos(src.state.cpu().numpy().view(np.uint32), R, layout.VS_WORDS)
        pos0 = aos[:, [layout.VS_POS_X, layout.VS_POS_Y]].view(np.float32)
        rng_m = np.random.default_rng(12)
    for m, P in moving:
        n_ck = K // P
        d = np.zeros((m, R, 4), dtype=np.float32)
        d[:, :, :2] = pos0[None] + rng_m.uniform(-0.15, 0.15, (m, R, 2))
        d[:, :, 2] = rng_m.uniform(0.02, 0.08, (m, R))
        static_m[m] = torch.from_numpy(d).to(dev)
        walk = np.cumsum(rng_m.uniform(-0.02, 0.02, (n_ck, m, R, 2)), axis=0).astype(np.float32)
        t4 = np.repeat(d[None], n_ck, axis=0)
        t4[..., :2] += walk
        mov[(m, P)] = torch.from_numpy(t4).to(dev)
    if moving:
        n_ck_max = max(K // P for _, P in moving)
        path_buf = torch.empty((n_ck_max, n, 2), dtype=torch.float32, device=dev)
        G_m = a.fleet or 8
        peers_m = fleet_peers(R, G_m, dev)

    def static_rollout(m, P):
        pl.rollout(src, ref, 1.0, 10.0, 1e-9, obstacles=static_m[m], w_obst=1e3, check_period=P)

    def moving_rollout(m, P, path=False):
        p = path_buf[: K // P] if path else None
        pl.rollout(src, ref, 1.0, 10.0, 1e-9, obstacles=mov[(m, P)], w_obst=1e3, check_period=P, path=p)

    def sample_sigma():
        pl.sample(nominal=nominal, seed=5, sigma_table=pl.sigma_table)

    def refit():
        pl.refit(cem_elite, shift=1)

    # warm-up: every shape once (the first rollout also runs the fast path's on-device proofs)
    sample(), plan_rollout(), select(), fork(), plain_rollout()
    if a.cem:
        sample_sigma(), refit()
    for m in obst_m:
        for P in obst_p:
            obst_rollout(m, P)
    for m, P in moving:
        static_rollout(m, P), moving_rollout(m, P), moving_rollout(m, P, True)
    if moving:
        pred = {P: pl.predict(src, P) for P in sorted({P for _, P in moving})}
        for P in pred:
            pl.peer_discs(pred[P], peers_m, 0.4)
    torch.cuda.synchronize()
    src_before = src.state.clone()
    t = {"sample": [], "plan_rollout": [], "select": [], "plain_rollout": []}
    if a.cem:
        t.update(sample_sigma=[], refit=[])
    t_obst, t_mov = {}, {}
    for _ in range(a.reps):
        t["sample"].append(timed(sample))
        if a.cem:
            t["sample_sigma"].append(timed(sample_sigma))
        t["plan_rollout"].append(timed(plan_rollout))
        t["select"].append(timed(select))
        if a.cem:
            t["refit"].append(timed(refit))
        fork()
        torch.cuda.synchronize()
        t["plain_rollout"].append(timed(plain_rollout))
        for m in obst_m:
            for P in obst_p:  # alternated with the plan rollout of the same candidates
                tp, to = t_obst.setdefault((m, P), ([], []))
                tp.append(timed(plan_rollout))
                to.append(timed(lambda: obst_rollout(m, P)))
        for m, P in moving:  # static, moving and moving with paths, alternated
            ts, tm, tpth = t_mov.setdefault((m, P), ([], [], []))
            ts.append(timed(lambda: static_rollout(m, P)))
            tm.append(timed(lambda: moving_rollout(m, P)))
            tpth.append(timed(lambda: moving_rollout(m, P, True)))
        if moving:
            for P in pred:
                t_mov.setdefault(("predict", P), []).append(timed(lambda: pl.predict(src, P)))
                t_mov.setdefault(("peer_discs", P), []).append(timed(lambda: pl.peer_discs(pred[P], peers_m, 0.4)))
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
    if moving:
        rows = []
        for m, P in moving:
            ts, tm, tpth = (float(np.median(v)) for v in t_mov[(m, P)])
            moving_rollout(m, P)
            mc = pl.cost.clone()
            moving_rollout(m, P, True)
            same = bool(torch.equal(pl.cost.view(torch.int32), mc.view(torch.int32)))
            rows.append({"m": m, "check_period": P, "ms_median_static": round(ts, 4), "ms_median_moving": round(tm, 4),
                         "ms_median_moving_path": round(tpth, 4), "moving_over_static": tm / ts, "path_over_moving": tpth / tm,
                         "path_bytes": (K // P) * n * 8, "path_store_ms": tpth - tm, "cost_same_with_path": same})
        res["moving"] = rows
        res["predict"] = [{"check_period": P, "robots": R, "ms_median": round(float(np.median(t_mov[("predict", P)])), 4),
                           "ms_min": round(float(np.min(t_mov[("predict", P)])), 4)} for P in pred]
        res["peer_discs"] = [{"check_period": P, "G": G_m, "cells": (K // P) * (G_m - 1) * R,
                              "ms_median": round(float(np.median(t_mov[("peer_discs", P)])), 4)} for P in pred]
    if moving or a.fleet:
        res["max_sm_clock"] = power_limit("clocks.max.sm")
    if a.fleet:
        res["fleet"] = fleet_report(a, a.fleet, dev)
    if a.cem:
        res["cem"] = {"iters": cem_iters, "elite": cem_elite,
                      "sample_sigma_over_sample": med["sample_sigma"] / med["sample"],
                      "refit_over_select": med["refit"] / med["select"],
                      "sample_sigma_plus_refit_over_rollout": (med["sample_sigma"] + med["refit"]) / med["plan_rollout"],
                      "compare": compare_planners(a, src, goal, ref, cem_iters, cem_elite)}
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
