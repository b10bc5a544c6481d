"""TEST INFRASTRUCTURE: the cross-entropy refit (rk_plan_refit) restated in numpy from its definition in
include/robotick.h, and the CEM planning loop of VehiclePlanner.plan_cem restated on the host with the plain-C port
(plan_ref / plan_obst_ref).  Shared by test_plan_cem_cpu.py and test_plan_cem_gpu.py.
"""
import numpy as np

import plan_obst_ref as por
import plan_ref as pr
from roboken_fmskf_robot_controller_b200 import _cabi, layout, streams

# the CEM loop both test files plan: plan_ref.SCENARIO's robots, goals and segments, 3 rounds of 64 candidates a step
# (192 rollouts, against plan_ref's 128), refitted to the 8 best
CEM = dict(iters=3, S=64, elite=8, alpha=0.3, sigma_min=(5.0, 5.0, 0.01))
GOLDEN = 0x9E3779B9  # round i of a step draws with seed + i * GOLDEN (mod 2^32)


def elites(cost, R, S, k):
    """Per robot, its elite candidates in ascending j: the first min(k, #finite) in the (cost, j) order, costs compared as
    floats (-0 equals +0), ties to the lower j; NaN and +-inf never elites."""
    c = np.asarray(cost, dtype=np.float32).reshape(R, S)
    out = []
    for r in range(R):
        fin = np.flatnonzero(np.isfinite(c[r]))
        key = c[r, fin] + np.float32(0.0)  # -0 + 0 = +0: one key for both zeros
        order = fin[np.argsort(key, kind="stable")]  # stable: ties keep ascending j
        out.append(np.sort(order[: min(k, fin.size)]))
    return out


def refit(cost, cand, sigma_in, R, S, k, alpha=0.0, sigma_min=(0.0, 0.0, 0.0), shift=1):
    """rk_plan_refit: cost float32 [R*S], cand [n_seg, R*S] records, sigma_in float32 [n_seg, R, 4] -> (nominal_out [n_seg, R]
    records, sigma_out float32 [n_seg, R, 4], best int32 [R], best_cost float32 [R]).  float32, one rounding per operation,
    in the header's order."""
    f32 = np.float32
    n_seg = cand.shape[0]
    _, best, best_cost = pr.select_argmin(cost, cand, R, S, shift)
    ss = np.minimum(np.arange(n_seg) + shift, n_seg - 1)
    cc = cand[ss].reshape(n_seg, R, S)
    v = np.stack([cc["vx"], cc["vy"], cc["vth"]], axis=-1).astype(np.float32)  # [n_seg, R, S, 3]
    sig_in = np.asarray(sigma_in, dtype=np.float32)[ss]  # [n_seg, R, 4]
    el = elites(cost, R, S, k)
    k_eff = np.array([e.size for e in el])
    kmax = max(1, int(k_eff.max()))
    idx = np.zeros((R, kmax), dtype=np.int64)
    for r, e in enumerate(el):
        idx[r, : e.size] = e
    valid = np.arange(kmax)[None, :] < k_eff[:, None]  # [R, kmax]
    ve = v[:, np.arange(R)[:, None], idx, :]  # [n_seg, R, kmax, 3]: the elites in ascending j
    kf = np.maximum(k_eff, 1).astype(np.float32)[None, :, None]
    with np.errstate(all="ignore"):  # robots without elites compute garbage here and are replaced below
        acc = ve[:, :, 0].copy()  # the sum starts from the first elite
        for i in range(1, kmax):
            acc = np.where(valid[None, :, i, None], acc + ve[:, :, i], acc).astype(np.float32)
        m = (acc / kf).astype(np.float32)
        q = np.zeros_like(m)
        for i in range(kmax):
            d = (ve[:, :, i] - m).astype(np.float32)
            q = np.where(valid[None, :, i, None], q + d * d, q).astype(np.float32)
        sd = np.sqrt(q / kf, dtype=np.float32)
        a = f32(alpha)
        if a > 0:
            b = f32(1.0) - a
            mean = (a * v[:, :, 0, :] + b * m).astype(np.float32)
            sig = (a * sig_in[:, :, :3] + b * sd).astype(np.float32)
        else:
            mean, sig = m, sd
    sigma_out = np.zeros((n_seg, R, 4), dtype=np.float32)
    sigma_out[:, :, :3] = np.fmax(sig, np.asarray(sigma_min, dtype=np.float32))
    nom = np.zeros((n_seg, R), dtype=pr.CMD_DT)
    nom["vx"], nom["vy"], nom["vth"], nom["kind"] = mean[..., 0], mean[..., 1], mean[..., 2], _cabi.RK_CMD_MOVE
    for r in np.flatnonzero(k_eff == 0):  # no finite cost: candidate best and the incoming sigma, bit for bit
        nom[:, r] = cc[:, r, best[r]]
        sigma_out[:, r] = sig_in[:, r]
    return nom, sigma_out, best, best_cost


def sigma_cells(sigma, n_seg, R):
    """The sigma table every cell of which is {sigma, 0}: what plan_cem resets the table to at the start of a step."""
    return np.ascontiguousarray(np.broadcast_to(np.array(tuple(sigma) + (0.0,), dtype=np.float32), (n_seg, R, 4)))


def plan_cem_loop(sc=pr.SCENARIO, cem=CEM, steps=None, shift=1, obs=None, w_obst=0.0, P=None):
    """VehiclePlanner.plan_cem in a closed loop from power-on, each step followed by the first segment of the new nominal.
    With obs (float32 [m, R, 4]) the rollouts price the keep-out discs (plan_obst_ref) with w_obst every P ticks.
    Returns per step (costs of every round, best, executed state) and the goals."""
    R, n_seg, seg_len, S = sc["R"], sc["n_seg"], sc["seg_len"], cem["S"]
    g = pr.goals(R)
    ref = np.ascontiguousarray(np.broadcast_to(g, (n_seg, R, 2)))
    state = np.zeros(layout.VS_WORDS * R, dtype=np.uint32)
    nominal = np.zeros((n_seg, R), dtype=pr.CMD_DT)
    out = []
    for it in range(sc["steps"] if steps is None else steps):
        seed = sc["seed"] + it
        sig = sigma_cells(sc["sigma"], n_seg, R)
        costs = []
        for i in range(cem["iters"]):
            cand = streams.plan_commands_v2(nominal, S, seed=(seed + i * GOLDEN) & 0xFFFFFFFF, sigma_table=sig)
            w = (sc["w_pos"], sc["w_goal"], sc["w_cur"])
            if obs is None:
                cost = pr.candidate_costs(state, R, S, cand, seg_len, ref, *w)
            else:
                cost, _ = por.candidate_costs_obst(state, R, S, cand, seg_len, ref, *w, obs, P, w_obst)
            last = i == cem["iters"] - 1
            nominal, sig, best, _ = refit(cost, cand, sig, R, S, cem["elite"], cem["alpha"], cem["sigma_min"], shift if last else 0)
            costs.append(cost)
        pr.execute(state, R, nominal, seg_len)
        out.append((costs, best, state.copy()))
    return out, g
