"""TEST INFRASTRUCTURE: cost-to-go fields (rk_plan_cost_to_go, rk_plan_rollout_field) restated on the host -- the field as
a float32 Dijkstra (heapq) and as a vectorised float32 Bellman-Ford, the terminal lookup and its place in the cost on the
port's trace rows, and the closed planning loops of the wall and dead-end scenarios.  Shared by test_plan_field_cpu.py
and the GPU tests.
"""
import heapq
from dataclasses import dataclass

import numpy as np

import oracle_lib as ol
import plan_cem_ref as pcr
import plan_fleet_ref as pfr
import plan_map_ref as pmr
import plan_ref as pr
from roboken_fmskf_robot_controller_b200 import _cabi, streams

f32 = np.float32
INF = f32(np.inf)
EXACT = 1 << 24  # a window edge beyond +-2^24 cells is not exact in float32


@dataclass
class HostCtg:
    """rk_plan_ctg_t: the float32 steps, the traversal weight and the lethal threshold."""

    step_axial: float
    step_diag: float
    k_cost: float
    lethal: float


def spec_for(resolution, k_cost=0.0, lethal=np.inf):
    """The spec planner.CostMap.cost_to_go passes: float32(res), float32(res * sqrt 2)."""
    return HostCtg(f32(resolution), f32(resolution * 2.0 ** 0.5), f32(k_cost), f32(lethal))


def _exact(o, n):
    return -EXACT <= o <= EXACT - n


def window_cell(u, v, ox, oy, fw, fh):
    """The window cell under grid coordinates (u, v) (float32 scalars), or None: the comparisons of the header."""
    if not (_exact(ox, fw) and _exact(oy, fh)):
        return None
    with np.errstate(invalid="ignore"):
        if not (u >= f32(ox) and u < f32(ox + fw) and v >= f32(oy) and v < f32(oy + fh)):
            return None
    return int(np.floor(u)) - ox, int(np.floor(v)) - oy


def window_costs(mp, k, ox, oy, fw, fh):
    """c float32 [fh, fw] of a field's window: map k's cells, `outside` off the map."""
    _, H, W = mp.cells.shape
    iy = oy + np.arange(fh)[:, None]
    ix = ox + np.arange(fw)[None, :]
    on = (ix >= 0) & (ix < W) & (iy >= 0) & (iy < H)
    return np.where(on, mp.cells[k][np.clip(iy, 0, H - 1), np.clip(ix, 0, W - 1)], f32(mp.outside)).astype(np.float32)


def goal_cell(mp, goal, k, ox, oy, fw, fh):
    """The goal's window cell (ix, iy), or None when the field has no goal (+inf everywhere)."""
    if not 0 <= k < mp.cells.shape[0]:
        return None
    gu = (f32(goal[0]) - f32(mp.x0)) * f32(mp.inv_res)
    gv = (f32(goal[1]) - f32(mp.y0)) * f32(mp.inv_res)
    return window_cell(gu, gv, ox, oy, fw, fh)


def _weights(c, spec):
    """(free bool [fh, fw], w_axial, w_diag float32 [fh, fw]): the step weights into each cell."""
    with np.errstate(invalid="ignore", over="ignore"):
        free = ~(c >= f32(spec.lethal))
        t = np.where(c > f32(0), f32(1) + f32(spec.k_cost) * c, f32(1)).astype(np.float32)
        return free, (f32(spec.step_axial) * t).astype(np.float32), (f32(spec.step_diag) * t).astype(np.float32)


DIRS = [(dx, dy) for dy in (-1, 0, 1) for dx in (-1, 0, 1) if (dx, dy) != (0, 0)]


def dijkstra(c, spec, goal):
    """The field float32 [fh, fw] of window costs c from goal cell (ix, iy) (None: +inf everywhere), heapq Dijkstra in
    float32: fl(a + w) is monotone in a and w >= 0, so the first time a cell is popped its value is final."""
    fh, fw = c.shape
    D = np.full((fh, fw), INF, dtype=np.float32)
    if goal is None:
        return D
    free, wa, wd = _weights(c, spec)
    gx, gy = goal
    D[gy, gx] = f32(0)
    heap = [(0.0, gx, gy)]
    done = np.zeros((fh, fw), dtype=bool)
    while heap:
        _, x, y = heapq.heappop(heap)
        if done[y, x]:
            continue
        done[y, x] = True
        d = D[y, x]
        for dx, dy in DIRS:
            qx, qy = x + dx, y + dy
            if not (0 <= qx < fw and 0 <= qy < fh) or not free[qy, qx]:
                continue
            if dx and dy and not (free[y, qx] and free[qy, x]):  # no corner cutting
                continue
            nd = f32(d + (wd if dx and dy else wa)[qy, qx])
            if nd < D[qy, qx]:
                D[qy, qx] = nd
                heapq.heappush(heap, (float(nd), qx, qy))
    return D


def bellman_ford(c, spec, goal):
    """The same field by synchronous Bellman-Ford sweeps over whole arrays until nothing changes."""
    fh, fw = c.shape
    D = np.full((fh, fw), INF, dtype=np.float32)
    if goal is None:
        return D
    free, wa, wd = _weights(c, spec)
    D[goal[1], goal[0]] = f32(0)
    pad = lambda a, v: np.pad(a, 1, constant_values=v)  # noqa: E731
    fp = pad(free, False)
    while True:
        Dp = pad(D, INF)
        best = np.full((fh, fw), INF, dtype=np.float32)
        for dx, dy in DIRS:
            src = Dp[1 - dy:1 - dy + fh, 1 - dx:1 - dx + fw]  # D(q - (dx, dy)): the predecessor p of q
            ok = free.copy()
            w = wa
            if dx and dy:
                ok &= fp[1:1 + fh, 1 - dx:1 - dx + fw] & fp[1 - dy:1 - dy + fh, 1:1 + fw]
                w = wd
            with np.errstate(invalid="ignore", over="ignore"):
                cand = np.where(ok, src + w, INF).astype(np.float32)
            best = np.minimum(best, cand)
        new = np.minimum(D, best)
        if np.array_equal(new, D):
            return D
        D = new


def build(mp, spec, goals, fw, fh, offsets=None, field_map=None, method=dijkstra):
    """rk_plan_cost_to_go on the host: float32 [n_fields, fh, fw]."""
    n = len(goals)
    out = np.empty((n, fh, fw), dtype=np.float32)
    for f in range(n):
        ox, oy = (0, 0) if offsets is None else (int(offsets[f][0]), int(offsets[f][1]))
        k = 0 if field_map is None else int(field_map[f])
        g = goal_cell(mp, goals[f], k, ox, oy, fw, fh)
        c = window_costs(mp, k, ox, oy, fw, fh) if 0 <= k < mp.cells.shape[0] and _exact(ox, fw) and _exact(oy, fh) else np.zeros((fh, fw), np.float32)
        out[f] = method(c, spec, g)
    return out


@dataclass
class HostField:
    """rk_plan_field_t on the host: field float32 [n_fields, fh, fw], offsets int [n_fields, 2] or None, field_of int [R]
    or None, and the float32 scalars the device reads."""

    field: np.ndarray
    offsets: object
    field_of: object
    x0: float
    y0: float
    inv_res: float
    outside: float
    w_field: float


def field_term(O, x, y, hf, ff):
    """O after the terminal term: x, y float32 [n] end positions, ff int [n] the field of each candidate."""
    n_f, fh, fw = hf.field.shape
    out = O.copy()
    for i in range(len(O)):
        f = int(ff[i])
        if not 0 <= f < n_f:
            continue
        ox, oy = (0, 0) if hf.offsets is None else (int(hf.offsets[f][0]), int(hf.offsets[f][1]))
        u = (f32(x[i]) - f32(hf.x0)) * f32(hf.inv_res)
        v = (f32(y[i]) - f32(hf.y0)) * f32(hf.inv_res)
        cell = window_cell(u, v, ox, oy, fw, fh)
        c = f32(hf.outside) if cell is None else hf.field[f, cell[1], cell[0]]
        if c > f32(0):
            with np.errstate(over="ignore"):
                out[i] = f32(out[i] + f32(hf.w_field) * c)
    return out


def candidate_costs_field(state_soa, R, S, cand, seg_len, ref, w_pos, w_goal, w_cur, obs, P, w_obst, mp, hf, params=None, trace=None):
    """The port's rk_plan_rollout_field: (J + O, O, path) -- plan_map_ref.candidate_costs_map plus the terminal term on the
    last trace row (mp may be None: no map term; hf None or w_field 0: the map rollout)."""
    if trace is None:
        trace = pmr.port_trace(state_soa, R, S, cand, seg_len, params)
    J = pr.stage_cost(trace, ref, S, seg_len, w_pos, w_goal, w_cur)
    O = pmr.map_obstacle_cost(trace, obs, S, P, w_obst, mp)
    if hf is not None and hf.w_field != 0:
        row = trace[-1]
        ff = np.zeros(R * S, dtype=np.int64) if hf.field_of is None else np.repeat(np.asarray(hf.field_of, dtype=np.int64), S)
        O = field_term(O, row[0].view(np.float32), row[1].view(np.float32), hf, ff)
    with np.errstate(over="ignore", invalid="ignore"):
        return (J + O).astype(np.float32), O, pfr.paths(trace, P)


# ---- scenarios ----------------------------------------------------------------------------------------------------------
# Each robot has its own lane, 1 m wide along x, and its own field: the lane's window of the inflated map (lethal = 1, so
# the inflated wall blocks) with its goal.  Positions are points; the field prices where a candidate ends after the
# horizon, so the planner needs no straight-line pull: w_pos = 0 and a small w_goal for the last centimetres inside the
# goal cell.
CELL = pmr.CELL


def dead_end_world(R, inflate=1):
    """A U of shelving that opens toward the robot: lane r has a bar 0.05 m thick across y in [0.10, 0.15) for x in
    [r - 0.2, r + 0.2) and two arms down to y = -0.30 along its ends.  The robot starts at (r, -0.45), south of the
    opening, and its goal is (r, 0.50), straight behind the bar.  (wall, cells, origin, starts, goals), as
    plan_map_ref.wall_world."""
    W, H = 20 * R, 32  # y in [-0.8, 0.8)
    x0, y0 = -0.5, -0.8
    xc = x0 + (np.arange(W) + 0.5) * CELL
    yc = y0 + (np.arange(H) + 0.5) * CELL
    dx = xc - np.floor(xc - x0) - x0 - 0.5  # x relative to the lane centre
    bar = (np.abs(dx) < 0.2)[None, :] & ((yc >= 0.10) & (yc < 0.15))[:, None]
    arms = ((np.abs(dx) >= 0.15) & (np.abs(dx) < 0.2))[None, :] & ((yc >= -0.30) & (yc < 0.15))[:, None]
    wall = bar | arms
    grown = _inflate(wall, inflate)
    starts = np.stack([np.arange(R, dtype=np.float64), np.full(R, -0.45)], axis=1).astype(np.float32)
    goals = np.stack([np.arange(R, dtype=np.float64), np.full(R, 0.50)], axis=1).astype(np.float32)
    return wall, grown.astype(np.float32), (x0, y0), starts, goals


def _inflate(wall, n):
    """wall grown by n cells in each of the 8 directions (as plan_map_ref.wall_world grows its wall)."""
    H, W = wall.shape
    grown = wall.copy()
    for _ in range(n):
        g = np.pad(grown, 1)
        grown = np.zeros_like(wall)
        for dy in (0, 1, 2):
            for dx in (0, 1, 2):
                grown |= g[dy:dy + H, dx:dx + W]
    return grown


def lane_fields(cells, origin, goals, R, lane_cells=20, k_cost=0.0):
    """(HostMap with w_map 0, spec, offsets int32 [R, 2], the fields float32 [R, H, lane_cells]): one window per lane."""
    mp = pmr.host_map(cells, origin, 0.0)
    spec = spec_for(CELL, k_cost, lethal=1.0)
    H = mp.cells.shape[1]
    offsets = np.stack([np.arange(R) * lane_cells, np.zeros(R, np.int64)], axis=1).astype(np.int32)
    return mp, spec, offsets, build(mp, spec, goals, lane_cells, H, offsets)


def host_field(fields, offsets, mp, w_field, field_of=None, outside=np.inf):
    return HostField(fields, offsets, field_of, f32(mp.x0), f32(mp.y0), f32(mp.inv_res), f32(outside), f32(w_field))


WALL_FIELD = dict(pmr.WALL, w_pos=0.0, w_goal=1.0, w_field=10.0)
DEAD_END = dict(WALL_FIELD, steps=60)


def field_loop(sc, world, use_field=True, use_map=True, cem=None, steps=None):
    """plan_map_ref.wall_loop with each robot's cost-to-go field as the terminal term (use_field) and with or without
    the cost map; world is wall_world or dead_end_world.  Returns (per step (costs, best, state, positions), goals, wall,
    origin, host field or None)."""
    R, n_seg, seg_len, P = sc["R"], sc["n_seg"], sc["seg_len"], sc["P"]
    wall, cells, origin, start, g = world(R)
    mp = pmr.host_map(cells, origin, sc["w_map"]) if use_map else None
    hf = None
    if use_field:
        mp0, _, offsets, fields = lane_fields(cells, origin, g, R)
        hf = host_field(fields, offsets, mp0, sc["w_field"], field_of=np.arange(R, dtype=np.int32))
    ref = np.ascontiguousarray(np.broadcast_to(g, (n_seg, R, 2)))
    state = pfr.start_states(start)
    nominal = np.zeros((n_seg, R), dtype=pr.CMD_DT)
    discs = np.zeros((n_seg * seg_len // P, 0, R, 4), dtype=np.float32)
    w = (sc["w_pos"], sc["w_goal"], sc["w_cur"]) if use_field else (pmr.WALL["w_pos"], pmr.WALL["w_goal"], pmr.WALL["w_cur"])
    out = []
    for it in range(sc["steps"] if steps is None else steps):
        seed = sc["seed"] + it
        costs = []
        rounds = [(sc["S"], None)] if cem is None else [(cem["S"], i) for i in range(cem["iters"])]
        sig = pcr.sigma_cells(sc["sigma"], n_seg, R)
        for S, i in rounds:
            if i is None:
                cand = streams.plan_commands_v2(nominal, S, seed=seed, sigma=sc["sigma"])
            else:
                cand = streams.plan_commands_v2(nominal, S, seed=(seed + i * pcr.GOLDEN) & 0xFFFFFFFF, sigma_table=sig)
            cost, _, _ = candidate_costs_field(state, R, S, cand, seg_len, ref, *w, discs, P, 0.0, mp, hf)
            if i is None:
                nominal, best, _ = pr.select_argmin(cost, cand, R, S, 0)
            else:
                nominal, sig, best, _ = pcr.refit(cost, cand, sig, R, S, cem["elite"], cem["alpha"], cem["sigma_min"], 0)
            costs.append(cost)
        ro = ol.HostRollout(R, seg_len, _cabi.RK_SENSOR_PLANT, np.ascontiguousarray(nominal[:1]), seg_len, trace=True)
        ol.run_port(state, R, ro)
        pos = np.stack([ro.trace[:, 0].view(np.float32), ro.trace[:, 1].view(np.float32)], axis=2)
        out.append((costs, best, state.copy(), pos))
    return out, g, wall, origin, hf


# ---- builder cases ------------------------------------------------------------------------------------------------------
def _grid(rng, shape, lethal_frac=0.2, nan=0.05, neg=0.1, inf=0.03):
    """Cells uniform in [0, 1) with some NaN, negative and +inf cells and a share at or above 1 (lethal at 1)."""
    c = rng.uniform(0.0, 1.0, shape).astype(np.float32)
    c[rng.random(shape) < lethal_frac] = f32(1.5)
    c[rng.random(shape) < neg] = f32(-2.0)
    c[rng.random(shape) < nan] = np.nan
    c[rng.random(shape) < inf] = np.inf
    return c


def builder_cases():
    """name -> (HostMap, HostCtg, goals float32 [n, 2], fw, fh, offsets int32 [n, 2] or None, field_map int32 [n] or None):
    every edge case of the header's definition.  Cells are 5 cm, origin (-0.3, -0.2)."""
    rng = np.random.default_rng(0xC7)
    cases = {}

    def mp_of(cells, outside=np.inf):
        return pmr.host_map(cells, (-0.3, -0.2), 0.0, outside=outside)

    def centre(m, ix, iy):  # the point at the centre of map cell (ix, iy)
        return [f32(m.x0) + (ix + 0.5) * CELL, f32(m.y0) + (iy + 0.5) * CELL]

    m = mp_of(_grid(rng, (37, 45)))
    blocked_goal = np.argwhere(m.cells[0] >= 1.0)[0]
    goals = [centre(m, 3, 4), centre(m, 40, 30), centre(m, blocked_goal[1], blocked_goal[0]), [np.nan, 0.0], centre(m, 60, 5)]
    cases["lethal 1, k_cost 0.5, blocked, NaN and off-window goals"] = (m, spec_for(CELL, 0.5, 1.0), goals, 45, 37, None, None)
    cases["lethal inf, k_cost 0"] = (m, spec_for(CELL), goals[:2], 45, 37, None, None)
    cases["k_cost 3, lethal 0.75"] = (m, spec_for(CELL, 3.0, 0.75), goals[:2], 45, 37, None, None)
    for outside in (0.0, np.inf):
        mo = mp_of(m.cells[0], outside)
        offs = np.array([[-5, -7], [30, 20], [-40, 0]], np.int32)  # hanging off the low corner, the high corner, all off
        g = [centre(mo, -3, -6), centre(mo, 50, 40), centre(mo, -30, 10)]
        cases[f"windows off the map, outside {outside}"] = (mo, spec_for(CELL, 0.5, 1.0), g, 24, 20, offs, None)
    mm = mp_of(np.stack([_grid(rng, (33, 40)) for _ in range(3)]))
    fm = np.array([0, 1, 2, -1, 3, 2], np.int32)
    g = [centre(mm, int(rng.integers(0, 40)), int(rng.integers(0, 33))) for _ in fm]
    cases["three maps through field_map, two out of range"] = (mm, spec_for(CELL, 0.25, 1.0), g, 40, 33, None, fm)
    cases["window 1 x 1"] = (m, spec_for(CELL, 0.5, 1.0), [centre(m, 7, 9), centre(m, 8, 9)], 1, 1, np.array([[7, 9], [7, 9]], np.int32), None)
    cases["window 1 x N"] = (m, spec_for(CELL, 0.5, 1.0), [centre(m, 5, 30)], 1, 37, np.array([[5, 0]], np.int32), None)
    cases["window N x 1"] = (m, spec_for(CELL, 0.5, 1.0), [centre(m, 44, 3)], 45, 1, np.array([[0, 3]], np.int32), None)
    big = np.array([[EXACT, 0], [0, -EXACT - 1], [EXACT - 45, 0]], np.int32)
    cases["offsets beyond 2^24"] = (m, spec_for(CELL), [[0.0, 0.0]] * 3, 45, 37, big, None)
    # a diagonal wall of single cells: without corner cutting the two sides do not connect
    c = np.zeros((16, 16), np.float32)
    for i in range(16):
        c[i, i] = np.inf
    cases["no corner cutting through a diagonal wall"] = (mp_of(c), spec_for(CELL), [centre(mp_of(c), 12, 2), centre(mp_of(c), 2, 12)], 16, 16, None, None)
    return cases


def serpentine(n_cells, corridor=1):
    """A serpentine maze of n_cells x n_cells: walls (+inf) on every other row pair, with a gap at alternating ends, so the
    one path from the corner crosses the whole grid back and forth.  Returns cells float32 [n, n]."""
    c = np.zeros((n_cells, n_cells), np.float32)
    step = corridor + 1
    for k, y in enumerate(range(corridor, n_cells, step)):
        c[y, :] = np.inf
        c[y, -1 if k % 2 == 0 else 0] = 0.0
    return c
