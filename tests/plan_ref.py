"""TEST INFRASTRUCTURE: the vehicle sampling planner (rk_plan_*) restated on the host with the plain-C port.

Candidates come from streams.plan_commands_v2, rollouts from the port on the S-fold forked state block (traces on), the
stage cost from the trace rows at the segment ends, the choice by argmin -- the planning loop with lambda = 0, word for
word what the device computes.  Shared by test_plan_cpu.py and test_plan_gpu.py.
"""
import numpy as np

import oracle_lib as ol
from roboken_fmskf_robot_controller_b200 import _cabi, layout, streams

CMD_DT = np.dtype([("vx", "<f4"), ("vy", "<f4"), ("vth", "<f4"), ("kind", "<i4")])

# the closed-loop scenario both test files plan: 8 robots from power-on, goals 0.2 - 0.3 m away, 128 candidates of
# 8 x 50-tick segments, 30 planning steps of which each executes one segment
SCENARIO = dict(R=8, S=128, n_seg=8, seg_len=50, steps=30, w_pos=1.0, w_goal=10.0, w_cur=1e-9, sigma=(100.0, 100.0, 0.2),
                seed=0xC0FFEE)


def fork(state_soa, R, S):
    """The S-fold copy of an R-robot block: instance r*S + j holds robot r's state (plane layout, pitch R*S)."""
    aos = layout.soa_to_aos(np.asarray(state_soa, dtype=np.uint32), R, layout.VS_WORDS)
    return layout.aos_to_soa(np.ascontiguousarray(np.repeat(aos, S, axis=0)))


def stage_cost(trace, ref, S, seg_len, w_pos, w_goal, w_cur):
    """rk_plan_cost_t on the port's trace rows: trace uint32 [n_seg*seg_len, 16, R*S], ref float32 [n_seg, R, 2] -> J float32 [R*S]."""
    f32 = np.float32
    n_seg = ref.shape[0]
    J = np.zeros(trace.shape[2], dtype=np.float32)
    for s in range(n_seg):
        row = trace[(s + 1) * seg_len - 1]
        x, y = row[0].view(np.float32), row[1].view(np.float32)
        c = [row[9 + k].view(np.int32).astype(np.float32) for k in range(4)]
        g = np.repeat(ref[s], S, axis=0)
        dx, dy = x - g[:, 0], y - g[:, 1]
        e = dx * dx + dy * dy
        q = ((c[0] * c[0] + c[1] * c[1]) + c[2] * c[2]) + c[3] * c[3]
        w = f32(w_pos if s < n_seg - 1 else w_goal)
        J = ((J + w * e) + f32(w_cur) * q).astype(np.float32)
    return J


def candidate_costs(state_soa, R, S, cand, seg_len, ref, w_pos, w_goal, w_cur, params=None, nthreads=8):
    """The port's rk_plan_rollout: cand [n_seg, R*S] records -> cost float32 [R*S]; state_soa is not modified."""
    n_seg = cand.shape[0]
    st = fork(state_soa, R, S)
    ro = ol.HostRollout(R * S, n_seg * seg_len, _cabi.RK_SENSOR_PLANT, np.ascontiguousarray(cand), seg_len, trace=True)
    ol.run_port(st, R * S, ro, params=params, nthreads=nthreads)
    return stage_cost(ro.trace, ref, S, seg_len, w_pos, w_goal, w_cur)


def select_argmin(cost, cand, R, S, shift=1):
    """rk_plan_select with lambda = 0: (new nominal [n_seg, R] records, best int32 [R], best_cost float32 [R])."""
    n_seg = cand.shape[0]
    key = np.where(np.isnan(cost), np.float32(np.inf), cost).reshape(R, S)
    best = np.argmin(key, axis=1).astype(np.int32)  # first occurrence: ties to the lowest j, all-NaN -> 0
    cols = np.arange(R) * S + best
    ss = np.minimum(np.arange(n_seg) + shift, n_seg - 1)
    return np.ascontiguousarray(cand[ss][:, cols]), best, cost.reshape(R, S)[np.arange(R), best]


def execute(state_soa, R, nominal, seg_len, params=None):
    """The robots run the first segment of the plan (rk_vdt_rollout of seg_len ticks); state_soa is advanced in place."""
    ro = ol.HostRollout(R, seg_len, _cabi.RK_SENSOR_PLANT, np.ascontiguousarray(nominal[:1]), seg_len)
    ol.run_port(state_soa, R, ro, params=params)


def goals(R, seed=5):
    """Goals 0.2 - 0.3 m from the origin in every direction, float32 [R, 2] metres."""
    rng = np.random.default_rng(seed)
    d, a = rng.uniform(0.2, 0.3, R), rng.uniform(-np.pi, np.pi, R)
    return np.stack([d * np.cos(a), d * np.sin(a)], axis=1).astype(np.float32)


def plan_loop(sc=SCENARIO, steps=None):
    """The whole planning loop with lambda = 0 from power-on.  Returns per step (cost, best, executed state) and the goals."""
    R, S, n_seg, seg_len = sc["R"], sc["S"], sc["n_seg"], sc["seg_len"]
    g = goals(R)
    ref = np.ascontiguousarray(np.broadcast_to(g, (n_seg, R, 2)))
    state = np.zeros(layout.VS_WORDS * R, dtype=np.uint32)
    nominal = np.zeros((n_seg, R), dtype=CMD_DT)
    out = []
    for it in range(sc["steps"] if steps is None else steps):
        cand = streams.plan_commands_v2(nominal, S, seed=sc["seed"] + it, sigma=sc["sigma"])
        cost = candidate_costs(state, R, S, cand, seg_len, ref, sc["w_pos"], sc["w_goal"], sc["w_cur"])
        nominal, best, _ = select_argmin(cost, cand, R, S)
        execute(state, R, nominal, seg_len)
        out.append((cost, best, state.copy()))
    return out, g


def distances(state_soa, R, g):
    aos = layout.soa_to_aos(state_soa, R, layout.VS_WORDS)
    pos = aos[:, [layout.VS_POS_X, layout.VS_POS_Y]].view(np.float32)
    return np.hypot(pos[:, 0] - g[:, 0], pos[:, 1] - g[:, 1])
