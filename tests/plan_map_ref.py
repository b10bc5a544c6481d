"""TEST INFRASTRUCTURE: cost maps (rk_plan_rollout_map) restated on the host with the plain-C port -- the cell lookup, the
per-checkpoint accumulation of discs and map into one O on the port's trace rows, and the closed planning loop on a
wall scenario under argmin and CEM.  Shared by test_plan_map_cpu.py and test_plan_map_gpu.py.
"""
from dataclasses import dataclass

import numpy as np

import oracle_lib as ol
import plan_cem_ref as pcr
import plan_fleet_ref as pfr
import plan_ref as pr
from roboken_fmskf_robot_controller_b200 import _cabi, streams

f32 = np.float32


@dataclass
class HostMap:
    """rk_plan_map_t on the host: cells float32 [n_maps, H, W], map_of int32 [R] or None, and the float32 scalars the
    device reads (inv_res already rounded, as planner.CostMap passes it)."""

    cells: np.ndarray
    map_of: object
    x0: float
    y0: float
    inv_res: float
    outside: float
    w_map: float


def lookup(x, y, cells, k, x0, y0, inv_res, outside):
    """c of the map term for positions x, y (float32 [n]) in map k (int [n], each in [0, n_maps)): the cell under the point,
    `outside` off the grid.  One float32 operation each, in the header's order."""
    _, H, W = cells.shape
    u = (x - f32(x0)) * f32(inv_res)
    v = (y - f32(y0)) * f32(inv_res)
    with np.errstate(invalid="ignore"):  # NaN positions compare false
        ok = (u >= f32(0)) & (u < f32(W)) & (v >= f32(0)) & (v < f32(H))
    iu = np.where(ok, u, f32(0)).astype(np.int64)  # truncation, as (int) on the device
    iv = np.where(ok, v, f32(0)).astype(np.int64)
    idx = (np.asarray(k, dtype=np.int64) * H + iv) * W + iu
    return np.where(ok, cells.reshape(-1)[np.where(ok, idx, 0)], f32(outside)).astype(np.float32)


def map_term(O, x, y, mp, kk):
    """O after the map term: kk int [n] the map of each candidate (any integer; outside [0, n_maps) adds nothing)."""
    have = (kk >= 0) & (kk < mp.cells.shape[0])
    c = lookup(x, y, mp.cells, np.where(have, kk, 0), mp.x0, mp.y0, mp.inv_res, mp.outside)
    with np.errstate(all="ignore"):  # w_map = inf times a 0 cell in the unselected lanes
        return np.where(have & (c > f32(0)), O + f32(mp.w_map) * c, O).astype(np.float32)


def candidate_maps(mp, R, S):
    """The map index of every candidate i = r*S + j: map_of[r], or 0 without map_of."""
    return np.zeros(R * S, dtype=np.int64) if mp.map_of is None else np.repeat(np.asarray(mp.map_of, dtype=np.int64), S)


def map_obstacle_cost(trace, obs, S, P, w_obst, mp):
    """O of rk_plan_rollout_map: trace uint32 [K, 16, R*S], obs float32 [n_ck, m, R, 4] (m may be 0), mp a HostMap or
    None (then plan_fleet_ref.moving_obstacle_cost).  At checkpoint c = 1 .. n_ck (trace row c*P - 1): discs k = 0 .. m-1
    of table c - 1, then the map term, into one accumulator."""
    if mp is None or mp.w_map == 0:
        return pfr.moving_obstacle_cost(trace, obs, S, P, w_obst)
    w = f32(w_obst)
    n = trace.shape[2]
    R = n // S
    kk = candidate_maps(mp, R, S)
    O = np.zeros(n, dtype=np.float32)
    assert obs.shape[0] == trace.shape[0] // P
    with np.errstate(all="ignore"):
        for c in range(1, obs.shape[0] + 1):
            row = trace[c * P - 1]
            x, y = row[0].view(np.float32), row[1].view(np.float32)
            for k in range(obs.shape[1]):
                d = np.repeat(np.asarray(obs[c - 1, k], dtype=np.float32), S, axis=0)
                dx, dy = x - d[:, 0], y - d[:, 1]
                pen = d[:, 2] * d[:, 2] - (dx * dx + dy * dy)
                O = np.where(pen > f32(0), O + w * pen, O).astype(np.float32)
            O = map_term(O, x, y, mp, kk)
    return O


def candidate_costs_map(state_soa, R, S, cand, seg_len, ref, w_pos, w_goal, w_cur, obs, P, w_obst, mp, params=None, nthreads=8, trace=None):
    """The port's rk_plan_rollout_map from one traced rollout of the forked block (or the given trace): (J + O, O, path
    float32 [n_ck, R*S, 2]); state_soa is not modified."""
    if trace is None:
        trace = port_trace(state_soa, R, S, cand, seg_len, params, nthreads)
    J = pr.stage_cost(trace, ref, S, seg_len, w_pos, w_goal, w_cur)
    O = map_obstacle_cost(trace, obs, S, P, w_obst, mp)
    return (J + O).astype(np.float32), O, pfr.paths(trace, P)


def port_trace(state_soa, R, S, cand, seg_len, params=None, nthreads=8):
    """The port's trace uint32 [K, 16, R*S] of every candidate from its robot's state."""
    st = pr.fork(state_soa, R, S)
    ro = ol.HostRollout(R * S, cand.shape[0] * seg_len, _cabi.RK_SENSOR_PLANT, np.ascontiguousarray(cand), seg_len, trace=True)
    ol.run_port(st, R * S, ro, params=params, nthreads=nthreads)
    return ro.trace


# ---- the wall scenario ------------------------------------------------------------------------------------------------
# R robots in lanes 1 m apart along x.  Lane r has a wall band 0.1 m thick across it (y in [-0.05, 0.05)) with a gap 0.3 m
# wide whose centre is 0.25 m to the side of the lane's line (east on even lanes, west on odd ones).  Each robot starts
# 0.35 m south of the band and has its goal 0.35 m north of it, so that the straight line runs into the wall.  Cells are
# 5 cm.  The cost grid the planner reads is the wall inflated by one cell (the robot is a point read every P ticks); the
# wall cells a test checks the executed ticks against are the band itself.
CELL = 0.05


def wall_world(R, inflate=1):
    """(wall bool [H, W], cost cells float32 [H, W], origin (x0, y0), starts float32 [R, 2], goals float32 [R, 2])."""
    W, H = 20 * R, 24  # lane r spans x in [r - 0.5, r + 0.5); y in [-0.6, 0.6)
    x0, y0 = -0.5, -0.6
    xc = x0 + (np.arange(W) + 0.5) * CELL  # cell centres
    yc = y0 + (np.arange(H) + 0.5) * CELL
    lane = np.floor(xc - x0).astype(np.int64)
    side = np.where(lane % 2 == 0, 1.0, -1.0)
    in_gap = np.abs(xc - (lane + 0.25 * side)) < 0.15
    band = np.abs(yc) < 0.05
    wall = band[:, None] & ~in_gap[None, :]
    grown = wall.copy()
    for _ in range(inflate):  # one cell in each of the 8 directions
        g = np.pad(grown, 1)
        grown = np.zeros_like(wall)
        for dy in (0, 1, 2):
            for dx in (0, 1, 2):
                grown |= g[dy:dy + H, dx:dx + W]
    starts = np.stack([np.arange(R, dtype=np.float64), np.full(R, -0.40)], axis=1).astype(np.float32)
    goals = np.stack([np.arange(R, dtype=np.float64), np.full(R, 0.40)], axis=1).astype(np.float32)
    return wall, grown.astype(np.float32), (x0, y0), starts, goals


def host_map(cells, origin, w_map, outside=np.inf, map_of=None):
    """The HostMap planner.CostMap(cells, origin, CELL, outside, map_of) passes: inv_res = float32(1 / CELL)."""
    c = np.ascontiguousarray(cells, dtype=np.float32)
    return HostMap(c if c.ndim == 3 else c[None], map_of, f32(origin[0]), f32(origin[1]), f32(1.0 / CELL), f32(outside), f32(w_map))


def in_wall(pos, wall, origin):
    """bool [...]: whether positions float32 [..., 2] lie in a wall cell (the same cell rule as the map lookup)."""
    H, W = wall.shape
    u = (pos[..., 0] - f32(origin[0])) * f32(1.0 / CELL)
    v = (pos[..., 1] - f32(origin[1])) * f32(1.0 / CELL)
    ok = (u >= 0) & (u < W) & (v >= 0) & (v < H)
    return ok & wall[np.where(ok, v, 0).astype(np.int64), np.where(ok, u, 0).astype(np.int64)]


# 4 robots, 96 candidates of 8 x 125-tick segments (the 0.4 m the 400 mm/s limit covers in the horizon), checkpoints every
# 25 ticks (10 mm at most between two, inside the one-cell inflation).  Plans keep shift = 0, so the segment executed is
# segment 0 of the candidate the map priced from the robot's state.
WALL = dict(R=4, S=96, n_seg=8, seg_len=125, P=25, steps=30, w_pos=1.0, w_goal=10.0, w_cur=1e-9, sigma=(250.0, 250.0, 0.2),
            seed=0xA11, w_map=1.0e4)
WALL_CEM = dict(iters=3, elite=8, alpha=0.0, sigma_min=(40.0, 40.0, 0.05), S=48)


def wall_loop(sc=WALL, use_map=True, cem=None, steps=None):
    """The planning loop of INTEGRATION.md §2 with a cost map on the port: per step plan with shift = 0 (argmin, or with
    cem a plan_cem step as plan_cem_ref restates it) with the map (use_map=False: m = 0 and no map), then execute segment 0.  Returns
    per step (costs of every round, best, executed state, executed positions float32 [seg_len, R, 2]), the goals, the wall
    and the origin."""
    R, n_seg, seg_len, P = sc["R"], sc["n_seg"], sc["seg_len"], sc["P"]
    wall, cells, origin, start, g = wall_world(R)
    mp = host_map(cells, origin, sc["w_map"]) if use_map else None
    ref = np.ascontiguousarray(np.broadcast_to(g, (n_seg, R, 2)))
    state = pfr.start_states(start)
    nominal = np.zeros((n_seg, R), dtype=pr.CMD_DT)
    discs = np.zeros((n_seg * seg_len // P, 0, R, 4), dtype=np.float32)
    w = (sc["w_pos"], sc["w_goal"], sc["w_cur"])
    out = []
    for it in range(sc["steps"] if steps is None else steps):
        seed = sc["seed"] + it
        costs = []
        if cem is None:
            S = sc["S"]
            cand = streams.plan_commands_v2(nominal, S, seed=seed, sigma=sc["sigma"])
            cost, _, _ = candidate_costs_map(state, R, S, cand, seg_len, ref, *w, discs, P, 0.0, mp)
            nominal, best, _ = pr.select_argmin(cost, cand, R, S, 0)
            costs.append(cost)
        else:
            S = cem["S"]
            sig = pcr.sigma_cells(sc["sigma"], n_seg, R)
            for i in range(cem["iters"]):
                cand = streams.plan_commands_v2(nominal, S, seed=(seed + i * pcr.GOLDEN) & 0xFFFFFFFF, sigma_table=sig)
                cost, _, _ = candidate_costs_map(state, R, S, cand, seg_len, ref, *w, discs, P, 0.0, mp)
                nominal, sig, best, _ = pcr.refit(cost, cand, sig, R, S, cem["elite"], cem["alpha"], cem["sigma_min"], 0)
                costs.append(cost)
        ro = ol.HostRollout(R, seg_len, _cabi.RK_SENSOR_PLANT, np.ascontiguousarray(nominal[:1]), seg_len, trace=True)
        ol.run_port(state, R, ro)
        pos = np.stack([ro.trace[:, 0].view(np.float32), ro.trace[:, 1].view(np.float32)], axis=2)
        out.append((costs, best, state.copy(), pos))
    return out, g, wall, origin
