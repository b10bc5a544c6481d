"""TEST INFRASTRUCTURE: rk_plan_rollout_obstacles restated on the host -- the keep-out cost O on the port's trace rows at
every checkpoint, on top of plan_ref's stage cost, and the lambda = 0 planning loop of plan_ref.plan_loop with discs.
Shared by test_plan_obst_cpu.py and test_plan_obst_gpu.py.
"""
import numpy as np

import oracle_lib as ol
import plan_ref as pr
from roboken_fmskf_robot_controller_b200 import _cabi, layout, streams


def obstacle_cost(trace, obs, S, P, w):
    """O of rk_plan_obstacles_t: trace uint32 [K, 16, R*S] (K % P == 0), obs float32 [m, R, 4] -> O float32 [R*S].
    Checkpoint c = 1 .. K/P is trace row c*P - 1; discs in order k = 0 .. m-1; float32 operations in the defined order."""
    f32 = np.float32
    w = f32(w)
    O = np.zeros(trace.shape[2], dtype=np.float32)
    with np.errstate(all="ignore"):  # NaN discs and w = inf: the unselected lanes of np.where
        for c in range(1, trace.shape[0] // P + 1):
            row = trace[c * P - 1]
            x, y = row[0].view(np.float32), row[1].view(np.float32)
            for k in range(obs.shape[0]):
                d = np.repeat(np.asarray(obs[k], dtype=np.float32), S, axis=0)
                dx, dy = x - d[:, 0], y - d[:, 1]
                pen = d[:, 2] * d[:, 2] - (dx * dx + dy * dy)
                O = np.where(pen > f32(0), O + w * pen, O).astype(np.float32)
    return O


def candidate_costs_obst(state_soa, R, S, cand, seg_len, ref, w_pos, w_goal, w_cur, obs, P, w_obst, params=None, nthreads=8):
    """The port's rk_plan_rollout_obstacles from one traced rollout of the forked block: (J + O, O), float32 [R*S] each;
    state_soa is not modified."""
    n_seg = cand.shape[0]
    st = pr.fork(state_soa, R, S)
    ro = ol.HostRollout(R * S, n_seg * seg_len, _cabi.RK_SENSOR_PLANT, np.ascontiguousarray(cand), seg_len, trace=True)
    ol.run_port(st, R * S, ro, params=params, nthreads=nthreads)
    J = pr.stage_cost(ro.trace, ref, S, seg_len, w_pos, w_goal, w_cur)
    O = obstacle_cost(ro.trace, obs, S, P, w_obst)
    return (J + O).astype(np.float32), O


def discs_near_the_path(g, radius, offset):
    """One disc per robot, float32 [1, R, 4]: centred halfway from the origin to the goal g [R, 2], moved `offset` metres
    sideways (to the left of the path) so that neither way round is the obvious one."""
    g = np.asarray(g, dtype=np.float64)
    u = g / np.hypot(g[:, 0], g[:, 1])[:, None]
    c = 0.5 * g + offset * np.stack([-u[:, 1], u[:, 0]], axis=1)
    obs = np.zeros((1, g.shape[0], 4), dtype=np.float32)
    obs[0, :, 0], obs[0, :, 1], obs[0, :, 2] = c[:, 0], c[:, 1], radius
    return obs


def plan_loop_obst(obs, w_obst, P, sc=pr.SCENARIO, steps=None, shift=0):
    """plan_ref.plan_loop with the keep-out discs obs float32 [m, R, 4] in the cost.  Returns per step (cost, best,
    executed state, executed positions float32 [seg_len, R, 2] of every tick of the segment) and the goals.

    shift = 0: the robots execute segment 0 of the chosen candidate, the very segment whose checkpoints the cost saw
    (with shift = 1 they would execute its segment 1 from the state its segment 0 started from)."""
    R, S, n_seg, seg_len = sc["R"], sc["S"], sc["n_seg"], sc["seg_len"]
    g = pr.goals(R)
    ref = np.ascontiguousarray(np.broadcast_to(g, (n_seg, R, 2)))
    state = np.zeros(layout.VS_WORDS * R, dtype=np.uint32)
    nominal = np.zeros((n_seg, R), dtype=pr.CMD_DT)
    out = []
    for it in range(sc["steps"] if steps is None else steps):
        cand = streams.plan_commands_v2(nominal, S, seed=sc["seed"] + it, sigma=sc["sigma"])
        cost, _ = candidate_costs_obst(state, R, S, cand, seg_len, ref, sc["w_pos"], sc["w_goal"], sc["w_cur"], obs, P, w_obst)
        nominal, best, _ = pr.select_argmin(cost, cand, R, S, shift)
        ro = ol.HostRollout(R, seg_len, _cabi.RK_SENSOR_PLANT, np.ascontiguousarray(nominal[:1]), seg_len, trace=True)
        ol.run_port(state, R, ro)
        pos = np.stack([ro.trace[:, 0].view(np.float32), ro.trace[:, 1].view(np.float32)], axis=2)
        out.append((cost, best, state.copy(), pos))
    return out, g


def min_clearance(out, obs):
    """Per robot, the least distance of any executed tick's position to any disc's centre minus its radius (metres)."""
    pos = np.concatenate([o[3] for o in out], axis=0).astype(np.float64)  # [ticks, R, 2]
    c = obs.astype(np.float64)
    d = np.hypot(pos[:, None, :, 0] - c[None, :, :, 0], pos[:, None, :, 1] - c[None, :, :, 1]) - c[None, :, :, 2]
    return d.min(axis=(0, 1))
