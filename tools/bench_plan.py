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

With --map CELLS:P (a comma list or repeated) the run also times rk_plan_rollout_map on a square world of CELLS x CELLS
5 cm cells (800 cells: 40 m, 2.56 MB) holding random rectangular walls, with m = 0 and 8 moving discs per robot checked
every P ticks, each alternated with rk_plan_rollout_moving on the same discs (m = 0: with a path, so that the moving
kernel runs), and reports map_over_moving.  Then it plays the wall scenario at size (R robots, each in its own lane with
a wall across it and a gap to the side, --map-steps steps under argmin and CEM --cem ITERS:ELITE, default 4:8) and
reports the share of robots that ever enter a wall cell, with and without the map, and the distance to the goal.
--parent-lib LIB also times LIB's rk_plan_rollout_moving (a build of another tree, loaded side by side) alternated with
this tree's on the same inputs, and checks that both give the same bits.

With --field CELLS:G the run also times rk_plan_cost_to_go on the random-wall world of --map (CELLS x CELLS cells, walls
lethal) with G whole-map fields, and on a serpentine maze of the same size as the worst case (one path that crosses
every tile row back and forth), reporting ms and relaxation rounds; then rk_plan_rollout_field (field of robot r: r % G)
alternated with rk_plan_rollout_map on the same inputs at P = 125, 25 and 5, with a path and no discs, and with
--parent-lib LIB's rk_plan_rollout_map alternated with this tree's.  Then it plays the wall scenario and a dead end (a U
of shelving that opens toward the robot, its goal straight behind the U's bottom) at size, under argmin and CEM, with
the map and with or without each robot's cost-to-go field over its 20-cell lane, and reports the share of robots within
0.1 m of their goals.

With --inflate the run also times rk_plan_inflate (CostMap.inflate) on 1 and 16 maps of the --map world's 800 x 800
random walls at table radii of 4, 10 and 40 cells (CUDA events around a batch of calls; median over --reps), against the
bytes a separable transform moves (16 per cell); then it plays the narrow-gap scenario of tests/plan_inflate_ref.py at
size (R lanes, each with a gap narrower than the body straight ahead and wide gaps on the lane boundaries, --inflate-steps
steps under argmin and CEM, each robot with its lane's cost-to-go field) on the raw walls and on the inflated map, and
reports the share of robots whose 0.15 m body ever overlapped a wall cell and the share within 0.1 m of the goal.

    python tools/bench_plan.py [--R 4096] [--S 256] [--n-seg 8] [--seg-len 125] [--reps 10] [--out FILE]
                               [--obstacles 1,8 --check-period 125,25,10] [--cem 4:8 --cem-steps 8 --lam 1e-3]
                               [--moving 1:125,8:25] [--fleet 8 --fleet-steps 60] [--map 800:125,800:25,800:5]
                               [--field 800:16] [--inflate] [--parent-lib path/to/librobotick_b200.so]
"""
import ctypes as C
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import roboken_fmskf_robot_controller_b200 as rk  # noqa: E402
from roboken_fmskf_robot_controller_b200 import _cabi, layout, streams  # noqa: E402
from roboken_fmskf_robot_controller_b200.planner import CostMap, CostToGo, VehiclePlanner, fleet_peers, inflation_table  # noqa: E402
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


def wall_world(R, dev, cell=0.05):
    """The wall scenario of tests/plan_map_ref.py at size: robot r in lane x in [r - 0.5, r + 0.5), a 0.1 m wall band across
    y = 0 with a 0.3 m gap centred 0.25 m east (even r) or west (odd r) of the lane's line, start 0.35 m south of the band,
    goal 0.35 m north.  Returns (wall bool [H, W] on the host, CostMap of the wall inflated by one cell, starts, goals)."""
    W, H = 20 * R, 24
    x0, y0 = -0.5, -0.6
    xc = x0 + (np.arange(W) + 0.5) * cell
    yc = y0 + (np.arange(H) + 0.5) * cell
    lane = np.floor(xc - x0).astype(np.int64)
    gap = np.abs(xc - (lane + 0.25 * np.where(lane % 2 == 0, 1.0, -1.0))) < 0.15
    wall = (np.abs(yc) < 0.05)[:, None] & ~gap[None, :]
    g = np.pad(wall, 1)
    grown = np.zeros_like(wall)
    for dy in range(3):
        for dx in range(3):
            grown |= g[dy:dy + H, dx:dx + W]
    cm = CostMap(torch.from_numpy(grown.astype(np.float32)).to(dev), (x0, y0), cell)
    starts = np.stack([np.arange(R, dtype=np.float64), np.full(R, -0.40)], axis=1).astype(np.float32)
    goals = np.stack([np.arange(R, dtype=np.float64), np.full(R, 0.40)], axis=1).astype(np.float32)
    return wall, cm, starts, goals


def random_walls(cells_n, rng):
    """The --map world: CELLS x CELLS cells, walls of 1 - 4 by 4 - 40 cells at random (one per 160 cells of area) costing 1."""
    g = np.zeros((cells_n, cells_n), dtype=np.float32)
    for _ in range(cells_n * cells_n // 160):
        h, w = (rng.integers(1, 5), rng.integers(4, 41))[:: 1 if rng.random() < 0.5 else -1]
        y, x = rng.integers(0, cells_n - h), rng.integers(0, cells_n - w)
        g[y:y + h, x:x + w] = 1.0
    return g


def serpentine(cells_n, corridor=3):
    """A maze of cells_n x cells_n: a +inf wall row after every `corridor` free rows, open at alternating ends."""
    g = np.zeros((cells_n, cells_n), np.float32)
    for k, y in enumerate(range(corridor, cells_n, corridor + 1)):
        g[y, :] = np.inf
        g[y, -1 if k % 2 == 0 else 0] = 0.0
    return g


def inflate(wall, n=1):
    H, W = wall.shape
    grown = wall.copy()
    for _ in range(n):
        g = np.pad(grown, 1)
        grown = np.zeros_like(wall)
        for dy in range(3):
            for dx in range(3):
                grown |= g[dy:dy + H, dx:dx + W]
    return grown


def dead_end_world(R, dev, cell=0.05):
    """The dead end of tests/plan_field_ref.py at size: lane r (x in [r - 0.5, r + 0.5), y in [-0.8, 0.8)) holds a U of
    shelving, a bar across y in [0.10, 0.15) for |x - r| < 0.2 and arms down to y = -0.30 at 0.15 <= |x - r| < 0.2; start
    (r, -0.45), goal (r, 0.50).  Returns (wall, CostMap of the wall inflated by one cell, starts, goals)."""
    W, H = 20 * R, 32
    x0, y0 = -0.5, -0.8
    xc = x0 + (np.arange(W) + 0.5) * cell
    yc = y0 + (np.arange(H) + 0.5) * cell
    dx = xc - np.floor(xc - x0) - x0 - 0.5
    bar = (np.abs(dx) < 0.2)[None, :] & ((yc >= 0.10) & (yc < 0.15))[:, None]
    arms = ((np.abs(dx) >= 0.15) & (np.abs(dx) < 0.2))[None, :] & ((yc >= -0.30) & (yc < 0.15))[:, None]
    wall = bar | arms
    cm = CostMap(torch.from_numpy(inflate(wall).astype(np.float32)).to(dev), (x0, y0), cell)
    starts = np.stack([np.arange(R, dtype=np.float64), np.full(R, -0.45)], axis=1).astype(np.float32)
    goals = np.stack([np.arange(R, dtype=np.float64), np.full(R, 0.50)], axis=1).astype(np.float32)
    return wall, cm, starts, goals


def field_play(a, dev, world, steps, iters, elite):
    """A scenario at size under argmin and CEM, with the map, with and without each robot's lane field (w_pos 0, w_goal 1,
    w_field 10 with it; w_pos 1, w_goal 10 without): the share of robots within 0.1 m of the goal after `steps` steps."""
    R, n_seg, seg_len, P = a.R, a.n_seg, a.seg_len, 25
    wall, cm, starts, goals = world(R, dev)
    ref = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(goals, (n_seg, R, 2)))).to(dev)
    aos = np.zeros((R, layout.VS_WORDS), dtype=np.uint32)
    aos[:, layout.VS_POS_X], aos[:, layout.VS_POS_Y] = starts[:, 0].view(np.uint32), starts[:, 1].view(np.uint32)
    offs = np.stack([np.arange(R) * 20, np.zeros(R, np.int64)], axis=1).astype(np.int32)
    ctg = cm.cost_to_go(goals, size=(cm.height, 20), offsets=offs, lethal=1.0, field_of=torch.arange(R, dtype=torch.int32, device=dev))
    out = {"robots": R, "steps": steps, "check_period": P, "w_map": 1e4, "field_bytes": ctg.field.numel() * 4, "build_rounds": ctg.rounds}
    for mode in ("argmin", "cem"):
        for use_field in (False, True):
            S = a.S if mode == "argmin" else a.S // iters
            pl = VehiclePlanner(R, S, n_seg, seg_len, dev, sigma=(250.0, 250.0, 0.2), seed=0xA11)
            vb = VehicleBatch(R, dev)
            vb.load_state_soa(layout.aos_to_soa(aos))
            w = (0.0, 1.0, 1e-9) if use_field else (1.0, 10.0, 1e-9)
            kw = dict(check_period=P, costmap=cm, w_map=1e4, field=ctg if use_field else None, w_field=10.0)
            for it in range(steps):
                if mode == "argmin":
                    pl.plan(vb, ref, *w, lam=0.0, shift=0, seed=0xA11 + it, **kw)
                else:
                    pl.plan_cem(vb, ref, *w, iters, elite, 0.0, (40.0, 40.0, 0.05), shift=0, seed=0xA11 + it, **kw)
                vb.rollout(seg_len, sensor_mode=_cabi.RK_SENSOR_PLANT, cmd=pl.first_command(), seg_len=seg_len)
            st = layout.soa_to_aos(vb.state.cpu().numpy().view(np.uint32), R, layout.VS_WORDS)
            pos = st[:, [layout.VS_POS_X, layout.VS_POS_Y]].view(np.float32)
            d = np.hypot(pos[:, 0] - goals[:, 0], pos[:, 1] - goals[:, 1])
            out[f"{mode}_{'field' if use_field else 'no_field'}"] = {
                "S": S, "goal_dist_median_m": float(np.median(d)), "goal_dist_p90_m": float(np.quantile(d, 0.9)),
                "within_0.1m_share": float((d < 0.1).mean())}
    return out


def field_bench(a, dev, pl, src, goal, cells_n, G, parent, iters, elite):
    """--field: the builder's time and rounds, rk_plan_rollout_field against rk_plan_rollout_map (and the parent's map
    rollout), and the two scenarios at size."""
    R, S, n_seg, seg_len = a.R, a.S, a.n_seg, a.seg_len
    n, K = R * S, n_seg * seg_len
    rng = np.random.default_rng(21)
    half = cells_n * 0.05 / 2
    g = random_walls(cells_n, rng)
    cm = CostMap(torch.from_numpy(g).to(dev), (-half, -half), 0.05)
    free = np.argwhere(g == 0)
    pick = free[rng.choice(len(free), G, replace=False)]
    goals = np.stack([-half + (pick[:, 1] + 0.5) * 0.05, -half + (pick[:, 0] + 0.5) * 0.05], axis=1).astype(np.float32)
    maze = CostMap(torch.from_numpy(serpentine(cells_n)).to(dev), (-half, -half), 0.05)
    corner = np.array([[-half + 0.025, -half + 0.025]], np.float32)
    out = {"cells": cells_n, "G": G, "builder": {}}
    for name, m, gl in (("random_walls", cm, goals), ("maze", maze, corner)):
        ms, rounds = [], None
        for _ in range(3 if name == "maze" else a.reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            ctg = m.cost_to_go(gl, lethal=1.0)  # synchronises the stream
            ms.append((time.perf_counter() - t0) * 1e3)
            rounds = ctg.rounds
        out["builder"][name] = {"fields": len(gl), "ms_median": round(float(np.median(ms)), 3), "ms_min": round(float(np.min(ms)), 3),
                                "rounds": rounds, "reachable_fraction": float(torch.isfinite(ctg.field).float().mean())}
    field = cm.cost_to_go(goals, lethal=1.0, field_of=(torch.arange(R, dtype=torch.int32, device=dev) % G).contiguous())
    # the robots spread over the world as for --map, each heading for its field's goal
    aos = layout.soa_to_aos(src.state.cpu().numpy().view(np.uint32), R, layout.VS_WORDS)
    pos1 = rng.uniform(-half + 1.0, half - 1.0, (R, 2)).astype(np.float32)
    aos[:, layout.VS_POS_X], aos[:, layout.VS_POS_Y] = pos1[:, 0].view(np.uint32), pos1[:, 1].view(np.uint32)
    src_f = VehicleBatch(R, dev)
    src_f.load_state_soa(layout.aos_to_soa(aos))
    ref_f = (torch.from_numpy(pos1).to(dev) + goal).unsqueeze(0).expand(n_seg, R, 2).contiguous()
    path = torch.empty((K // 5, n, 2), dtype=torch.float32, device=dev)
    par_cost = torch.empty(n, dtype=torch.float32, device=dev)

    def roll(P, use_field):
        pl.rollout(src_f, ref_f, 1.0, 10.0, 1e-9, check_period=P, path=path[: K // P], costmap=cm, w_map=1.0,
                   field=field if use_field else None, w_field=10.0)

    def parent_map(P, lib):
        c = _cabi.PlanCost()
        c.d_ref, c.w_pos, c.w_goal, c.w_cur = ref_f.data_ptr(), 1.0, 10.0, 1e-9
        o = _cabi.PlanObstacles()
        o.check_period = P
        mp = cm.struct(1.0)
        out_c = pl.cost if lib is pl.lib else par_cost
        _cabi.check(lib.rk_plan_rollout_map(C.byref(pl.params), src_f.state.data_ptr(), R, S, pl.candidates.data_ptr(), n_seg, seg_len,
                                            C.byref(c), C.byref(o), C.byref(mp), path[: K // P].data_ptr(), out_c.data_ptr(),
                                            C.c_void_p(torch.cuda.current_stream().cuda_stream)))

    rows, prow = [], []
    for P in (125, 25, 5):
        roll(P, False), roll(P, True)
        tm, tf = [], []
        for _ in range(a.reps):
            tm.append(timed(lambda: roll(P, False)))
            tf.append(timed(lambda: roll(P, True)))
        roll(P, False)
        base = pl.cost.clone()
        roll(P, True)
        rows.append({"check_period": P, "ms_median_map": round(float(np.median(tm)), 4), "ms_median_field": round(float(np.median(tf)), 4),
                     "ms_min_max_field": [round(float(np.min(tf)), 4), round(float(np.max(tf)), 4)],
                     "field_over_map": float(np.median(tf) / np.median(tm)), "priced_fraction": (pl.cost != base).float().mean().item()})
        if parent is not None:
            parent_map(P, parent), parent_map(P, pl.lib)
            tp, tt = [], []
            for _ in range(a.reps):
                tp.append(timed(lambda: parent_map(P, parent)))
                tt.append(timed(lambda: parent_map(P, pl.lib)))
            torch.cuda.synchronize()
            prow.append({"check_period": P, "ms_median_parent": round(float(np.median(tp)), 4), "ms_median_this": round(float(np.median(tt)), 4),
                         "this_over_parent": float(np.median(tt) / np.median(tp)),
                         "same_bits": bool(torch.equal(par_cost.view(torch.int32), pl.cost.view(torch.int32)))})
    out["rollout"] = rows
    if parent is not None:
        out["parent_map"] = prow
    out["wall"] = field_play(a, dev, wall_world, a.map_steps, iters, elite)
    out["dead_end"] = field_play(a, dev, dead_end_world, a.field_steps, iters, elite)
    return out


# The narrow-gap scenario of tests/plan_inflate_ref.py: 0.15 m body; the inflated map is +inf within 0.225 m of a wall cell
# (body, 10 mm between checkpoints, 65 mm for the grid) with a thin soft tail out to 0.3 m
NARROW_BODY, NARROW_INSCRIBED, NARROW_RADIUS, NARROW_SCALING, NARROW_PEAK = 0.15, 0.225, 0.3, 20.0, 1e-4


def narrow_gap_walls(R, cell=0.05):
    """Raw walls bool [H, W] of R lanes x in [r - 0.5, r + 0.5), y in [-1, 1): a 0.1 m band across y = 0 with a 0.2 m gap on
    the lane's line and a 0.6 m gap centred on each lane boundary; origin (-0.5, -1.0)."""
    W, H = 20 * R, 40
    ix = np.arange(W) % 20
    gap = ((ix >= 8) & (ix < 12)) | (ix < 6) | (ix >= 14)
    yc = -1.0 + (np.arange(H) + 0.5) * cell
    return (np.abs(yc) < 0.05)[:, None] & ~gap[None, :]


def clearance_overlap(pos, wall_t, origin, body, cell=0.05):
    """bool [R]: whether some position float32 [T, R, 2] (device) lies closer than `body` to a wall cell's square (the
    cells within 4 of the position's own are searched: 0.2 m > body)."""
    H, W = wall_t.shape
    p = pos.double()
    ix = torch.floor((p[..., 0] - origin[0]) / cell).long()
    iy = torch.floor((p[..., 1] - origin[1]) / cell).long()
    hit = torch.zeros(pos.shape[1], dtype=torch.bool, device=pos.device)
    for dy in range(-4, 5):
        for dx in range(-4, 5):
            cx, cy = ix + dx, iy + dy
            ok = (cx >= 0) & (cx < W) & (cy >= 0) & (cy < H)
            isw = ok & wall_t[cy.clamp(0, H - 1), cx.clamp(0, W - 1)]
            lx, ly = origin[0] + cx * cell, origin[1] + cy * cell
            ddx = torch.clamp(torch.maximum(lx - p[..., 0], p[..., 0] - (lx + cell)), min=0.0)
            ddy = torch.clamp(torch.maximum(ly - p[..., 1], p[..., 1] - (ly + cell)), min=0.0)
            hit |= (isw & (torch.hypot(ddx, ddy) < body)).any(dim=0)
    return hit


def inflate_bench(a, dev, iters, elite):
    """--inflate: rk_plan_inflate's time on the random-wall world, and the narrow-gap scenario at size."""
    out = {"timing": []}
    rng = np.random.default_rng(31)
    grids = np.stack([random_walls(800, rng) for _ in range(16)])
    batch = 20  # calls per timed window: one call on one map takes microseconds
    for n_maps in (1, 16):
        cm = CostMap(torch.from_numpy(grids[:n_maps].copy()).to(dev), (-20.0, -20.0), 0.05)
        for rc in (4, 10, 40):
            table = inflation_table(0.05, 0.2, rc * 0.05 + 1e-9, scaling=3.0, device=dev)
            cm.inflate(table, lethal=1.0)
            torch.cuda.synchronize()
            ts = [timed(lambda: [cm.inflate(table, lethal=1.0) for _ in range(batch)]) / batch for _ in range(a.reps)]
            cells = n_maps * 800 * 800
            ms = float(np.median(ts))
            out["timing"].append({"maps": n_maps, "cells": cells, "radius_cells": rc, "n_table": table.numel(), "us_median": round(ms * 1e3, 2),
                                  "us_min_max": [round(float(np.min(ts)) * 1e3, 2), round(float(np.max(ts)) * 1e3, 2)],
                                  "model_bytes": 16 * cells, "model_GB_per_s": round(16 * cells / (ms * 1e-3) / 1e9, 1)})
    out["timing_note"] = ("model_bytes: 16 per cell (cells read twice, a 2-byte column distance written and read, the output written); "
                          "the 16 maps' 164 MB would take about 21 us at the 7.7 TB/s HBM data-sheet rate; the working set stays in L2 "
                          "across the repeated calls")
    R, n_seg, seg_len, P = a.R, a.n_seg, a.seg_len, 25
    wall = narrow_gap_walls(R)
    origin = (-0.5, -1.0)
    raw = CostMap(torch.from_numpy(wall.astype(np.float32)).to(dev), origin, 0.05)
    inflated = raw.inflate(inflation_table(0.05, NARROW_INSCRIBED, NARROW_RADIUS, NARROW_SCALING, NARROW_PEAK, device=dev), lethal=1.0)
    wall_t = torch.from_numpy(wall).to(dev)
    starts = np.stack([np.arange(R, dtype=np.float64), np.full(R, -0.40)], axis=1).astype(np.float32)
    goals = np.stack([np.arange(R, dtype=np.float64), np.full(R, 0.40)], axis=1).astype(np.float32)
    ref = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(goals, (n_seg, R, 2)))).to(dev)
    aos = np.zeros((R, layout.VS_WORDS), dtype=np.uint32)
    aos[:, layout.VS_POS_X], aos[:, layout.VS_POS_Y] = starts[:, 0].view(np.uint32), starts[:, 1].view(np.uint32)
    offs = np.stack([np.arange(R) * 20, np.zeros(R, np.int64)], axis=1).astype(np.int32)
    sc = {"robots": R, "steps": a.inflate_steps, "check_period": P, "w_map": 1e4, "w_field": 10.0, "body_m": NARROW_BODY,
          "inscribed_m": NARROW_INSCRIBED, "radius_m": NARROW_RADIUS, "scaling": NARROW_SCALING, "peak": NARROW_PEAK}
    for use in (False, True):
        cm = inflated if use else raw
        ctg = cm.cost_to_go(goals, size=(cm.height, 20), offsets=offs, lethal=1.0, field_of=torch.arange(R, dtype=torch.int32, device=dev))
        for mode in ("argmin", "cem"):
            S = a.S if mode == "argmin" else a.S // iters
            pl = VehiclePlanner(R, S, n_seg, seg_len, dev, sigma=(250.0, 250.0, 0.2), seed=0xA11)
            vb = VehicleBatch(R, dev)
            vb.load_state_soa(layout.aos_to_soa(aos))
            tr = torch.empty((seg_len, _cabi.RK_VDT_TRACE_WORDS, R), dtype=torch.int32, device=dev)
            hit = torch.zeros(R, dtype=torch.bool, device=dev)
            kw = dict(check_period=P, costmap=cm, w_map=1e4, field=ctg, w_field=10.0)
            for it in range(a.inflate_steps):
                if mode == "argmin":
                    pl.plan(vb, ref, 0.0, 1.0, 1e-9, lam=0.0, shift=0, seed=0xA11 + it, **kw)
                else:
                    pl.plan_cem(vb, ref, 0.0, 1.0, 1e-9, iters, elite, 0.0, (40.0, 40.0, 0.05), shift=0, seed=0xA11 + it, **kw)
                vb.rollout(seg_len, sensor_mode=_cabi.RK_SENSOR_PLANT, cmd=pl.first_command(), seg_len=seg_len, trace=tr)
                hit |= clearance_overlap(tr[:, :2].view(torch.float32).permute(0, 2, 1), wall_t, origin, NARROW_BODY)
            st = layout.soa_to_aos(vb.state.cpu().numpy().view(np.uint32), R, layout.VS_WORDS)
            pos = st[:, [layout.VS_POS_X, layout.VS_POS_Y]].view(np.float32)
            d = np.hypot(pos[:, 0] - goals[:, 0], pos[:, 1] - goals[:, 1])
            sc[f"{mode}_{'inflated' if use else 'raw'}"] = {
                "S": S, "body_overlapped_wall_share": float(hit.float().mean()), "within_0.1m_share": float((d < 0.1).mean()),
                "goal_dist_median_m": float(np.median(d)), "goal_dist_p90_m": float(np.quantile(d, 0.9))}
    out["narrow_gap"] = sc
    return out


def wall_report(a, dev, iters, elite):
    """The wall scenario at size under argmin (S candidates) and CEM (iters rounds of S / iters), with and without the map:
    the share of robots that ever enter a wall cell and the distance to the goal after --map-steps steps."""
    R, n_seg, seg_len, P = a.R, a.n_seg, a.seg_len, 25
    wall, cm, starts, goals = wall_world(R, dev)
    ref = torch.from_numpy(np.ascontiguousarray(np.broadcast_to(goals, (n_seg, R, 2)))).to(dev)
    aos = np.zeros((R, layout.VS_WORDS), dtype=np.uint32)
    aos[:, layout.VS_POS_X], aos[:, layout.VS_POS_Y] = starts[:, 0].view(np.uint32), starts[:, 1].view(np.uint32)
    out = {"robots": R, "steps": a.map_steps, "check_period": P, "w_map": 1e4, "cell_m": 0.05, "inflation_cells": 1}
    for mode in ("argmin", "cem"):
        for use_map in (False, True):
            S = a.S if mode == "argmin" else a.S // iters
            pl = VehiclePlanner(R, S, n_seg, seg_len, dev, sigma=(250.0, 250.0, 0.2), seed=0xA11)
            vb = VehicleBatch(R, dev)
            vb.load_state_soa(layout.aos_to_soa(aos))
            tr = torch.empty((seg_len, _cabi.RK_VDT_TRACE_WORDS, R), dtype=torch.int32, device=dev)
            hit = np.zeros(R, dtype=bool)
            kw = dict(check_period=P, costmap=cm if use_map else None, w_map=1e4)
            for it in range(a.map_steps):
                if mode == "argmin":
                    pl.plan(vb, ref, 1.0, 10.0, 1e-9, lam=0.0, shift=0, seed=0xA11 + it, **kw)
                else:
                    pl.plan_cem(vb, ref, 1.0, 10.0, 1e-9, iters, elite, 0.0, (40.0, 40.0, 0.05), shift=0, seed=0xA11 + it, **kw)
                vb.rollout(seg_len, sensor_mode=_cabi.RK_SENSOR_PLANT, cmd=pl.first_command(), seg_len=seg_len, trace=tr)
                t = tr.cpu().numpy().view(np.uint32)
                u = ((t[:, 0].view(np.float32) - np.float32(-0.5)) * np.float32(20.0))
                v = ((t[:, 1].view(np.float32) - np.float32(-0.6)) * np.float32(20.0))
                ok = (u >= 0) & (u < wall.shape[1]) & (v >= 0) & (v < wall.shape[0])
                hit |= (ok & wall[np.where(ok, v, 0).astype(np.int64), np.where(ok, u, 0).astype(np.int64)]).any(axis=0)
            st = layout.soa_to_aos(vb.state.cpu().numpy().view(np.uint32), R, layout.VS_WORDS)
            pos = st[:, [layout.VS_POS_X, layout.VS_POS_Y]].view(np.float32)
            d = np.hypot(pos[:, 0] - goals[:, 0], pos[:, 1] - goals[:, 1])
            out[f"{mode}_{'map' if use_map else 'no_map'}"] = {
                "S": S, "entered_wall_share": float(hit.mean()), "goal_dist_median_m": float(np.median(d)),
                "goal_dist_p90_m": float(np.quantile(d, 0.9)), "within_0.1m_share": float((d < 0.1).mean()),
                "north_of_wall_share": float((pos[:, 1] > 0.05).mean())}
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
    ap.add_argument("--map", action="append", default=[], help="CELLS:P pairs (comma list or repeated): time cost maps")
    ap.add_argument("--map-steps", type=int, default=40, help="planning steps of the wall scenario")
    ap.add_argument("--parent-lib", default=None, help="another build's library: time its rk_plan_rollout_moving side by side")
    ap.add_argument("--field", default=None, help="CELLS:G: time cost-to-go fields and play the wall and dead-end scenarios")
    ap.add_argument("--field-steps", type=int, default=60, help="planning steps of the dead-end scenario")
    ap.add_argument("--inflate", action="store_true", help="time rk_plan_inflate and play the narrow-gap scenario")
    ap.add_argument("--inflate-steps", type=int, default=60, help="planning steps of the narrow-gap scenario")
    a = ap.parse_args()
    moving = [tuple(int(v) for v in x.split(":")) for arg in a.moving for x in arg.split(",") if x]
    maps = [tuple(int(v) for v in x.split(":")) for arg in a.map for x in arg.split(",") if x]
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

    # cost maps: CELLS x CELLS cells of 5 cm centred on the origin, walls of 1 - 4 cells by 4 - 40 cells at random, one per
    # 160 cells of area, each cell of a wall costing 1.  The robots of these rollouts are the mid-move robots moved to
    # random places over the world (1 m from its edge), so that their cells are spread over the whole map as in a
    # building, not all in the few cells around the origin; discs around them as for --moving
    worlds, map_tabs = {}, {}
    if maps:
        aos = layout.soa_to_aos(src.state.cpu().numpy().view(np.uint32), R, layout.VS_WORDS)
        rng_w = np.random.default_rng(13)
        half = max(c for c, _ in maps) * 0.05 / 2
        pos1 = rng_w.uniform(-half + 1.0, half - 1.0, (R, 2)).astype(np.float32)
        aos[:, layout.VS_POS_X], aos[:, layout.VS_POS_Y] = pos1[:, 0].view(np.uint32), pos1[:, 1].view(np.uint32)
        src_map = VehicleBatch(R, dev)
        src_map.load_state_soa(layout.aos_to_soa(aos))
        map_path = torch.empty((K // min(P for _, P in maps), n, 2), dtype=torch.float32, device=dev)
        ref_map = (torch.from_numpy(pos1).to(dev) + goal).unsqueeze(0).expand(n_seg, R, 2).contiguous()
    for cells_n, P in maps:
        if cells_n not in worlds:
            half = cells_n * 0.05 / 2
            worlds[cells_n] = CostMap(torch.from_numpy(random_walls(cells_n, rng_w)).to(dev), (-half, -half), 0.05)
        n_ck = K // P
        for m in (0, 8):
            d = np.zeros((m, R, 4), dtype=np.float32)
            d[:, :, :2] = pos1[None] + rng_w.uniform(-0.15, 0.15, (m, R, 2))
            d[:, :, 2] = rng_w.uniform(0.02, 0.08, (m, R))
            t4 = np.repeat(d[None], n_ck, axis=0)
            t4[..., :2] += np.cumsum(rng_w.uniform(-0.02, 0.02, (n_ck, m, R, 2)), axis=0).astype(np.float32)
            map_tabs[(m, P)] = torch.from_numpy(t4).to(dev)

    def map_moving(cells_n, P, m, use_map):
        p = map_path[: K // P] if m == 0 else None  # m = 0 without a path would run rk_plan_rollout's kernel
        pl.rollout(src_map, ref_map, 1.0, 10.0, 1e-9, obstacles=map_tabs[(m, P)], w_obst=1e3, check_period=P, path=p,
                   costmap=worlds[cells_n] if use_map else None, w_map=1.0)

    parent = None
    if a.parent_lib:
        assert maps or a.field, "--parent-lib times the discs of --map or the map rollout of --field"
        parent = C.CDLL(os.path.abspath(a.parent_lib), mode=C.RTLD_LOCAL)
        parent.rk_plan_rollout_moving.argtypes = pl.lib.rk_plan_rollout_moving.argtypes
        parent.rk_plan_rollout_map.argtypes = pl.lib.rk_plan_rollout_map.argtypes
        par_cost = torch.empty(n, dtype=torch.float32, device=dev)
        par_P = sorted({P for _, P in maps} or {P for _, P in moving} or {seg_len})
        par_tabs = map_tabs if maps else {}

    def parent_moving(P, m, lib):
        c = _cabi.PlanCost()
        c.d_ref, c.w_pos, c.w_goal, c.w_cur = ref_map.data_ptr(), 1.0, 10.0, 1e-9
        o = _cabi.PlanObstacles()
        tab = par_tabs[(m, P)]
        o.d_obs, o.m, o.check_period, o.w_obst = tab.data_ptr(), m, P, 1e3
        out = pl.cost if lib is pl.lib else par_cost
        pth = map_path[: K // P].data_ptr() if m == 0 else None
        _cabi.check(lib.rk_plan_rollout_moving(C.byref(pl.params), src_map.state.data_ptr(), R, S, pl.candidates.data_ptr(), n_seg, seg_len,
                                               C.byref(c), C.byref(o), pth, out.data_ptr(), C.c_void_p(torch.cuda.current_stream().cuda_stream)))

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
    for cells_n, P in maps:
        for m in (0, 8):
            map_moving(cells_n, P, m, False), map_moving(cells_n, P, m, True)
    if parent is not None and maps:
        for P in par_P:
            for m in (0, 8):
                parent_moving(P, m, parent), parent_moving(P, m, pl.lib)
    torch.cuda.synchronize()
    src_before = src.state.clone()
    t = {"sample": [], "plan_rollout": [], "select": [], "plain_rollout": []}
    if a.cem:
        t.update(sample_sigma=[], refit=[])
    t_obst, t_mov, t_map, t_par = {}, {}, {}, {}
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
        for cells_n, P in maps:  # the moving rollout and the map rollout on the same discs, alternated
            for m in (0, 8):
                tm, tmap = t_map.setdefault((cells_n, P, m), ([], []))
                tm.append(timed(lambda: map_moving(cells_n, P, m, False)))
                tmap.append(timed(lambda: map_moving(cells_n, P, m, True)))
        if parent is not None and maps:  # the same rk_plan_rollout_moving call from the other build and from this one, alternated
            for P in par_P:
                for m in (0, 8):
                    tpar, tthis = t_par.setdefault((P, m), ([], []))
                    tpar.append(timed(lambda: parent_moving(P, m, parent)))
                    tthis.append(timed(lambda: parent_moving(P, m, pl.lib)))
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
    if maps:
        rows = []
        for (cells_n, P, m), (tm, tmap) in t_map.items():
            map_moving(cells_n, P, m, False)
            base = pl.cost.clone()
            map_moving(cells_n, P, m, True)
            rows.append({"cells": cells_n, "map_bytes": cells_n * cells_n * 4, "check_period": P, "m": m,
                         "ms_median_moving": round(float(np.median(tm)), 4), "ms_median_map": round(float(np.median(tmap)), 4),
                         "ms_min_map": round(float(np.min(tmap)), 4), "ms_max_map": round(float(np.max(tmap)), 4),
                         "map_over_moving": float(np.median(tmap) / np.median(tm)),
                         "priced_fraction": (pl.cost != base).float().mean().item()})
        res["map"] = rows
        res["wall"] = wall_report(a, dev, *((cem_iters, cem_elite) if a.cem else (4, 8)))
    if parent is not None and maps:
        rows = []
        for (P, m), (tpar, tthis) in t_par.items():
            parent_moving(P, m, parent)
            parent_moving(P, m, pl.lib)
            torch.cuda.synchronize()
            rows.append({"check_period": P, "m": m, "path": m == 0, "ms_median_parent": round(float(np.median(tpar)), 4),
                         "ms_median_this": round(float(np.median(tthis)), 4), "this_over_parent": float(np.median(tthis) / np.median(tpar)),
                         "ms_min_max_parent": [round(float(np.min(tpar)), 4), round(float(np.max(tpar)), 4)],
                         "ms_min_max_this": [round(float(np.min(tthis)), 4), round(float(np.max(tthis)), 4)],
                         "same_bits": bool(torch.equal(par_cost.view(torch.int32), pl.cost.view(torch.int32)))})
        res["parent_moving"] = rows
    if a.field:
        cells_n, G = (int(v) for v in a.field.split(":"))
        res["field"] = field_bench(a, dev, pl, src, goal, cells_n, G, parent, *((cem_iters, cem_elite) if a.cem else (4, 8)))
    if a.inflate:
        res["inflate"] = inflate_bench(a, dev, *((cem_iters, cem_elite) if a.cem else (4, 8)))
    if moving or a.fleet or maps or a.field or a.inflate:
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
