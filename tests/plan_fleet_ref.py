"""TEST INFRASTRUCTURE: moving keep-out discs and predicted paths (rk_plan_rollout_moving, rk_plan_peer_discs) restated
on the host with the plain-C port -- the per-checkpoint disc cost on the port's trace rows, the candidates' paths, the
peer discs in numpy, and the closed fleet loop (predict -> peer discs -> plan -> execute) under argmin and CEM, on the
circle-swap scenario.  Shared by test_plan_fleet_cpu.py and test_plan_fleet_gpu.py.
"""
import numpy as np

import oracle_lib as ol
import plan_cem_ref as pcr
import plan_ref as pr
from roboken_fmskf_robot_controller_b200 import _cabi, layout, streams

NAN_DISC = np.array([0.0, 0.0, np.nan, 0.0], dtype=np.float32)  # what rk_plan_peer_discs writes for a missing peer


def moving_obstacle_cost(trace, obs, S, P, w):
    """O of rk_plan_rollout_moving: trace uint32 [K, 16, R*S] (K % P == 0), obs float32 [n_ck, m, R, 4] (n_ck = K/P) ->
    O float32 [R*S].  plan_obst_ref.obstacle_cost with checkpoint c = 1 .. n_ck (trace row c*P - 1) reading table c - 1."""
    f32 = np.float32
    w = f32(w)
    O = np.zeros(trace.shape[2], dtype=np.float32)
    assert obs.shape[0] == trace.shape[0] // P
    with np.errstate(all="ignore"):  # NaN discs and w = inf: the unselected lanes of np.where
        for c in range(1, obs.shape[0] + 1):
            row = trace[c * P - 1]
            x, y = row[0].view(np.float32), row[1].view(np.float32)
            for k in range(obs.shape[1]):
                d = np.repeat(np.asarray(obs[c - 1, k], dtype=np.float32), S, axis=0)
                dx, dy = x - d[:, 0], y - d[:, 1]
                pen = d[:, 2] * d[:, 2] - (dx * dx + dy * dy)
                O = np.where(pen > f32(0), O + w * pen, O).astype(np.float32)
    return O


def paths(trace, P):
    """d_path of rk_plan_rollout_moving: float32 [n_ck, n, 2], the position words of trace rows c*P - 1, c = 1 .. n_ck."""
    rows = trace[P - 1 :: P]
    return np.stack([rows[:, 0].view(np.float32), rows[:, 1].view(np.float32)], axis=2)


def candidate_costs_moving(state_soa, R, S, cand, seg_len, ref, w_pos, w_goal, w_cur, obs, P, w_obst, params=None, nthreads=8):
    """The port's rk_plan_rollout_moving from one traced rollout of the forked block: (J + O, O, path float32
    [n_ck, R*S, 2]); state_soa is not modified.  obs float32 [n_ck, m, R, 4] (m may be 0)."""
    n_seg = cand.shape[0]
    st = pr.fork(state_soa, R, S)
    ro = ol.HostRollout(R * S, n_seg * seg_len, _cabi.RK_SENSOR_PLANT, np.ascontiguousarray(cand), seg_len, trace=True)
    ol.run_port(st, R * S, ro, params=params, nthreads=nthreads)
    J = pr.stage_cost(ro.trace, ref, S, seg_len, w_pos, w_goal, w_cur)
    O = moving_obstacle_cost(ro.trace, obs, S, P, w_obst)
    return (J + O).astype(np.float32), O, paths(ro.trace, P)


def predict(state_soa, R, nominal, seg_len, P, params=None):
    """VehiclePlanner.predict: where each robot's nominal [n_seg, R] records takes it, float32 [n_ck, R, 2]."""
    ro = ol.HostRollout(R, nominal.shape[0] * seg_len, _cabi.RK_SENSOR_PLANT, np.ascontiguousarray(nominal), seg_len, trace=True)
    ol.run_port(pr.fork(state_soa, R, 1), R, ro, params=params)
    return paths(ro.trace, P)


def peer_discs(path, peers, radius, out=None, k0=0):
    """rk_plan_peer_discs: path float32 [n_ck, R, 2], peers int32 [m, R] -> out float32 [n_ck, M, R, 4] (default a new
    [n_ck, m, R, 4]); slots k0 .. k0+m-1 written, the others untouched."""
    n_ck, R = path.shape[0], path.shape[1]
    m = peers.shape[0]
    if out is None:
        out = np.zeros((n_ck, m, R, 4), dtype=np.float32)
    for k in range(m):
        for r in range(R):
            q = int(peers[k, r])
            if 0 <= q < R and q != r:
                out[:, k0 + k, r] = np.stack([path[:, q, 0], path[:, q, 1], np.full(n_ck, radius, np.float32), np.zeros(n_ck, np.float32)], 1)
            else:
                out[:, k0 + k, r] = NAN_DISC
    return out


def fleet_peers(R, G):
    """planner.fleet_peers in numpy: int32 [G-1, R], the other robots of r's group r // G in ascending order, -1 past R."""
    out = np.full((G - 1, R), -1, dtype=np.int32)
    for r in range(R):
        others = [q for q in range(r - r % G, r - r % G + G) if q != r]
        for k, q in enumerate(others):
            out[k, r] = q if q < R else -1
    return out


# The circle swap: groups of G robots start evenly spaced on a circle of radius `circle` around their group's centre,
# each with the antipodal point as its goal, so that every straight path crosses the centre at about the same time.
# Groups sit `spacing` apart along x and never see each other.
def circle_swap(n_groups, G, circle, spacing):
    """(start positions, goals), float32 [R, 2] each, R = n_groups * G, metres."""
    g = np.repeat(np.arange(n_groups), G)
    a = 2.0 * np.pi * (np.arange(n_groups * G) % G) / G + 0.3 * g  # each group turned a little
    centre = np.stack([g * spacing, np.zeros_like(g, dtype=np.float64)], axis=1)
    u = np.stack([np.cos(a), np.sin(a)], axis=1)
    return (centre + circle * u).astype(np.float32), (centre - circle * u).astype(np.float32)


def start_states(start):
    """Power-on states (plane layout) with the position words set to start float32 [R, 2]."""
    aos = np.zeros((start.shape[0], layout.VS_WORDS), dtype=np.uint32)
    aos[:, layout.VS_POS_X], aos[:, layout.VS_POS_Y] = start[:, 0].view(np.uint32), start[:, 1].view(np.uint32)
    return layout.aos_to_soa(aos)


def fleet_loop(sc, avoid=True, cem=None, steps=None):
    """The fleet loop of INTEGRATION.md §2 on the port: per step predict (P ticks) -> peer discs (fleet_peers, radius
    sc["disc"]) -> plan with shift = 0 (argmin, or with cem a plan_cem step as plan_cem_ref restates it) ->
    execute segment 0.  avoid=False plans the same way with no discs (m = 0).  Returns per step (costs of every round,
    best, executed state, executed positions float32 [seg_len, R, 2]) and the goals."""
    n_grp, G, S, n_seg, seg_len, P = sc["groups"], sc["G"], sc["S"], sc["n_seg"], sc["seg_len"], sc["P"]
    R = n_grp * G
    start, g = circle_swap(n_grp, G, sc["circle"], sc["spacing"])
    ref = np.ascontiguousarray(np.broadcast_to(g, (n_seg, R, 2)))
    state = start_states(start)
    nominal = np.zeros((n_seg, R), dtype=pr.CMD_DT)
    peers = fleet_peers(R, G)
    w = (sc["w_pos"], sc["w_goal"], sc["w_cur"])
    out = []
    for it in range(sc["steps"] if steps is None else steps):
        if avoid:
            discs = peer_discs(predict(state, R, nominal, seg_len, P), peers, sc["disc"])
        else:
            discs = np.zeros((n_seg * seg_len // P, 0, R, 4), dtype=np.float32)
        seed = sc["seed"] + it
        costs = []
        if cem is None:
            cand = streams.plan_commands_v2(nominal, S, seed=seed, sigma=sc["sigma"])
            cost, _, _ = candidate_costs_moving(state, R, S, cand, seg_len, ref, *w, discs, P, sc["w_obst"])
            nominal, best, _ = pr.select_argmin(cost, cand, R, S, 0)
            costs.append(cost)
        else:
            sig = pcr.sigma_cells(sc["sigma"], n_seg, R)
            for i in range(cem["iters"]):
                cand = streams.plan_commands_v2(nominal, cem["S"], seed=(seed + i * pcr.GOLDEN) & 0xFFFFFFFF, sigma_table=sig)
                cost, _, _ = candidate_costs_moving(state, R, cem["S"], cand, seg_len, ref, *w, discs, P, sc["w_obst"])
                nominal, sig, best, _ = pcr.refit(cost, cand, sig, R, cem["S"], cem["elite"], cem["alpha"], cem["sigma_min"], 0)
                costs.append(cost)
        ro = ol.HostRollout(R, seg_len, _cabi.RK_SENSOR_PLANT, np.ascontiguousarray(nominal[:1]), seg_len, trace=True)
        ol.run_port(state, R, ro)
        pos = np.stack([ro.trace[:, 0].view(np.float32), ro.trace[:, 1].view(np.float32)], axis=2)
        out.append((costs, best, state.copy(), pos))
    return out, g


def least_pair_distance(pos, G):
    """Per group, the least distance between two of its robots over every executed tick: pos float32 [ticks, R, 2] ->
    float64 [R // G]."""
    p = pos.astype(np.float64).reshape(pos.shape[0], -1, G, 2)
    d = np.hypot(p[:, :, :, None, 0] - p[:, :, None, :, 0], p[:, :, :, None, 1] - p[:, :, None, :, 1])
    d[:, :, np.arange(G), np.arange(G)] = np.inf
    return d.min(axis=(0, 2, 3))
