"""TEST INFRASTRUCTURE: cost-map inflation (rk_plan_inflate) restated on the host -- the squared distance to the nearest
obstacle twice, by brute force over every obstacle and through scipy's exact Euclidean distance transform, with the one
output rule both share -- the edge cases of the definition, and the narrow-gap scenario for plan_field_ref.field_loop.
Shared by test_plan_inflate_cpu.py and test_plan_inflate_gpu.py.
"""
import numpy as np
from scipy import ndimage

import plan_map_ref as pmr

f32 = np.float32
NONE = 1 << 62  # d2 without an obstacle: beyond every table


def obstacles(cells, lethal):
    """bool [n_maps, H, W]: c >= lethal (NaN never)."""
    with np.errstate(invalid="ignore"):
        return np.asarray(cells, np.float32) >= f32(lethal)


def _ring(obst, edge):
    """The maps padded with a one-cell ring of obstacles when the cells off the grid are obstacles (the nearest off-grid
    obstacle is always in the ring), else returned as they are; and the pad width."""
    if not edge:
        return obst, 0
    return np.pad(obst, ((0, 0), (1, 1), (1, 1)), constant_values=True), 1


def d2_brute(cells, outside, lethal):
    """int64 [n_maps, H, W]: the least (qx - ox)^2 + (qy - oy)^2 over every obstacle o of the cell's map, NONE without one."""
    obst, p = _ring(obstacles(cells, lethal), f32(outside) >= f32(lethal))
    n, H, W = np.shape(cells)
    yy, xx = np.mgrid[0:H, 0:W]
    out = np.full((n, H, W), NONE, np.int64)
    for k in range(n):
        oy, ox = np.nonzero(obst[k])
        if len(oy):
            d2 = (yy[..., None] + p - oy) ** 2 + (xx[..., None] + p - ox) ** 2
            out[k] = d2.min(axis=-1)
    return out


def d2_edt(cells, outside, lethal):
    """The same d2 from scipy.ndimage.distance_transform_edt's nearest-obstacle indices, squared in integers."""
    obst, p = _ring(obstacles(cells, lethal), f32(outside) >= f32(lethal))
    n, H, W = np.shape(cells)
    out = np.full((n, H, W), NONE, np.int64)
    yy, xx = np.mgrid[0:H + 2 * p, 0:W + 2 * p]
    for k in range(n):
        if not obst[k].any():
            continue
        iy, ix = ndimage.distance_transform_edt(~obst[k], return_distances=False, return_indices=True)
        d2 = (iy.astype(np.int64) - yy) ** 2 + (ix.astype(np.int64) - xx) ** 2
        out[k] = d2[p:p + H, p:p + W]
    return out


def apply(cells, d2, table):
    """The output rule: v = table[d2] where d2 < n_table, out = (v > c || c != c) ? v : c; out = c elsewhere."""
    c = np.asarray(cells, np.float32)
    table = np.asarray(table, np.float32)
    have = d2 < len(table)
    v = table[np.where(have, d2, 0)]
    with np.errstate(invalid="ignore"):
        take = have & ((v > c) | np.isnan(c))
    return np.where(take, v, c).astype(np.float32)


def inflate(cells, outside, lethal, table, d2=d2_edt):
    """rk_plan_inflate on the host: float32 [n_maps, H, W] (cells [H, W] or [n_maps, H, W])."""
    c = np.asarray(cells, np.float32)
    c = c if c.ndim == 3 else c[None]
    return apply(c, d2(c, outside, lethal), table)


# ---- edge cases -----------------------------------------------------------------------------------------------------------
def _random(rng, shape, obst=0.05):
    c = rng.uniform(-0.5, 1.0, shape).astype(np.float32)
    c[rng.random(shape) < obst] = f32(2.0)
    return c


def cases():
    """name -> (cells float32 [n_maps, H, W], outside, lethal, table float32 [n]): every edge case of the header's
    definition.  The tables rise with d2 where that matters, so that a wrong distance shows in the output."""
    rng = np.random.default_rng(0x1F)
    ramp = lambda n, top=3.0: np.linspace(top, 0.25, n).astype(np.float32)  # noqa: E731
    out = {}
    base = _random(rng, (1, 23, 37))
    out["random, outside below lethal"] = (base, 0.0, 1.0, ramp(50))
    out["random, outside at lethal"] = (base, 1.0, 1.0, ramp(50))
    out["random, outside +inf"] = (base, np.inf, 1.0, ramp(50))
    out["no obstacle"] = (rng.uniform(0.0, 0.9, (1, 9, 11)).astype(np.float32), 0.5, 1.0, ramp(20))
    out["no obstacle but the edge"] = (rng.uniform(0.0, 0.9, (1, 9, 11)).astype(np.float32), 1.5, 1.0, ramp(20))
    out["all obstacles"] = (np.full((1, 6, 7), 4.0, np.float32), 0.0, 1.0, ramp(9))
    sp = _random(rng, (1, 19, 21), obst=0.03)
    for i, v in enumerate((np.nan, -np.inf, np.inf, -3.0, np.nan, np.inf)):
        sp[0, 3 * i + 1, 2 * i + 5] = v
    out["NaN, -inf, +inf and negative cells"] = (sp, 0.0, 1.0, ramp(40))
    out["lethal +inf: only +inf cells and an +inf edge"] = (sp, np.inf, np.inf, ramp(40))
    out["lethal +inf, finite outside"] = (sp, 1e30, np.inf, ramp(40))
    out["n_table 1"] = (base, 0.0, 1.0, np.array([5.0], np.float32))
    for n in (10, 17, 26):  # d2 = n - 1 = rmax^2 is in the table, d2 = n (rmax^2 + 1) is not
        one = np.zeros((1, 15, 15), np.float32)
        one[0, 7, 7] = 1.0
        out[f"one obstacle, n_table {n}"] = (one, 0.0, 1.0, ramp(n))
    out["1 x N"] = (_random(rng, (1, 1, 40), obst=0.1), 0.0, 1.0, ramp(30))
    out["N x 1"] = (_random(rng, (1, 40, 1), obst=0.1), 0.0, 1.0, ramp(30))
    out["1 x N, edge"] = (_random(rng, (1, 1, 40), obst=0.0), np.inf, 1.0, ramp(30))
    out["N x 1, edge"] = (_random(rng, (1, 40, 1), obst=0.0), np.inf, 1.0, ramp(30))
    out["1 x 1"] = (np.array([[[0.5]]], np.float32), np.inf, 1.0, ramp(3))
    several = np.stack([_random(rng, (17, 29), obst=o) for o in (0.0, 0.02, 0.2)])
    out["three maps, one without obstacles"] = (several, 0.0, 1.0, ramp(65))
    out["three maps, edge"] = (several, np.inf, 1.0, ramp(65))
    z = np.zeros((1, 8, 9), np.float32)
    z[0, ::2, ::3] = -0.0
    z[0, 4, 4] = 1.0
    z[0, 1, 1] = np.nan
    out["signed zeros, table +0"] = (z, 0.0, 1.0, np.zeros(10, np.float32))
    out["signed zeros, table -0"] = (z, 0.0, 1.0, np.full(10, -0.0, np.float32))
    t = ramp(12)
    t[[0, 2, 5]] = np.nan
    out["NaN table entries"] = (z, 0.0, 1.0, t)
    tn = ramp(12)
    tn[[1, 4]] = -np.inf
    out["-inf table entries"] = (sp, 0.0, 1.0, tn)
    return out


# ---- the narrow-gap scenario --------------------------------------------------------------------------------------------
# Lane r spans x in [r - 0.5, r + 0.5) (20 cells, as plan_field_ref.lane_fields windows it) and y in [-1, 1).  A wall band
# 0.1 m thick across y = 0 has a narrow gap 0.2 m wide straight ahead on the lane's line x = r, narrower than the 0.3 m
# body, and a wide gap 0.6 m wide centred on each lane boundary x = r +- 0.5, which the neighbouring lanes share.  Each
# robot starts at (r, -0.4) with its goal at (r, 0.4).  The raw walls are cost-1 cells.  The inflated map prices a cell
# +inf within INSCRIBED of a raw wall cell (and of the map's edge, outside = +inf): the body radius, 10 mm for the
# distance covered between two checkpoints (P = 25 ticks at 0.4 mm per tick) and 65 mm for the grid, since the distance
# is between cell centres while the check below is from the robot's point to a wall cell's square.  A thin soft tail
# beyond keeps the map term small next to the field.
BODY_M = 0.15
INSCRIBED = BODY_M + 0.010 + 0.065
RADIUS, SCALING, PEAK = 0.3, 20.0, 1e-4


def narrow_gap_walls(R):
    """(wall bool [H, W], origin): the raw walls of R lanes."""
    W, H = 20 * R, 40
    x0, y0 = -0.5, -1.0
    ix = np.arange(W) % 20  # the cell within its lane; the lane's line x = r lies between cells 9 and 10
    gap = ((ix >= 8) & (ix < 12)) | (ix < 6) | (ix >= 14)
    yc = y0 + (np.arange(H) + 0.5) * pmr.CELL
    return (np.abs(yc) < 0.05)[:, None] & ~gap[None, :], (x0, y0)


def table(resolution=pmr.CELL):
    """The scenario's inflation profile: planner.inflation_table(resolution, INSCRIBED, RADIUS, SCALING, PEAK), on the host."""
    d = np.sqrt(np.arange(65537, dtype=np.float64)) * resolution
    d = d[: int(np.count_nonzero(d <= RADIUS))]
    return np.where(d <= INSCRIBED, np.inf, PEAK * np.exp(-SCALING * (d - INSCRIBED))).astype(np.float32)


def narrow_gap_world(R, inflated=True):
    """(wall, cells float32 [H, W], origin, starts, goals) for plan_field_ref.field_loop: the raw cost-1 walls, inflated
    (lethal 1, outside +inf) by table() when `inflated`."""
    wall, origin = narrow_gap_walls(R)
    cells = wall.astype(np.float32)
    if inflated:
        cells = inflate(cells, np.inf, 1.0, table())[0]
    starts = np.stack([np.arange(R, dtype=np.float64), np.full(R, -0.40)], axis=1).astype(np.float32)
    goals = np.stack([np.arange(R, dtype=np.float64), np.full(R, 0.40)], axis=1).astype(np.float32)
    return wall, cells, origin, starts, goals


def point_robot_world(R):
    return narrow_gap_world(R, inflated=False)


def wall_clearance(pos, wall, origin):
    """float64 [...]: the distance in metres from each position float32 [..., 2] to the nearest raw wall cell, taken as a
    square."""
    iy, ix = np.nonzero(wall)
    lo_x = origin[0] + ix * pmr.CELL
    lo_y = origin[1] + iy * pmr.CELL
    p = np.asarray(pos, np.float64).reshape(-1, 1, 2)
    best = np.full(p.shape[0], np.inf)
    for s in range(0, len(ix), 256):
        dx = np.maximum(np.maximum(lo_x[s:s + 256] - p[..., 0], 0.0), p[..., 0] - (lo_x[s:s + 256] + pmr.CELL))
        dy = np.maximum(np.maximum(lo_y[s:s + 256] - p[..., 1], 0.0), p[..., 1] - (lo_y[s:s + 256] + pmr.CELL))
        best = np.minimum(best, np.hypot(dx, dy).min(axis=1))
    return best.reshape(np.shape(pos)[:-1])
