"""Sampling planner for the vehicle over the C-ABI (rk_plan_* in include/robotick.h), torch owning the buffers.

One planning step for R robots with S candidates each: sample candidate command tables around the nominal plan, roll
every candidate out from its robot's current state and rank it by a stage cost, then pick (argmin) or blend (MPPI) the
candidates into the next nominal plan.  Candidate j of robot r is column r*S + j of every table.  The cross-entropy
method (plan_cem) runs several sample -> rollout -> refit rounds per step, refitting a per-robot, per-segment mean and
sigma to each round's elite candidates.
"""
import ctypes as C

import torch

from . import _cabi
from .vehicle import _dev_index


class VehiclePlanner:
    """Owns the candidate table int32 [n_seg, R*S, 4] (rk_vdt_cmd_t records), the cost float32 [R*S], the nominal plan
    int32 [n_seg, R, 4], the sigma table float32 [n_seg, R, 4] {sx, sy, sth, 0} of the cross-entropy rounds, and best
    (int32 [R]) / best_cost (float32 [R]) of the last selection or refit.  Every call is asynchronous on the current torch
    stream of the planner's device.

    sigma: noise scale of vx, vy (mm/s) and vth (rad/s); seed / first: the counter hash of the noise (first = global index
    of robot 0, so that sharded planners draw what one planner over all robots would)."""

    def __init__(self, R, S, n_seg, seg_len, device="cuda:0", params=None, sigma=(100.0, 100.0, 1.0), seed=0x5EED, first=0):
        self.lib = _cabi.load()
        self.R, self.S, self.n_seg, self.seg_len = int(R), int(S), int(n_seg), int(seg_len)
        self.device = torch.device(device)
        self.dev_index = _dev_index(device)
        self.params = params or _cabi.default_params()
        self.sigma, self.seed, self.first = tuple(float(x) for x in sigma), int(seed), int(first)
        with torch.cuda.device(self.dev_index):
            kw = dict(device=self.device)
            self.candidates = torch.zeros((self.n_seg, self.R * self.S, 4), dtype=torch.int32, **kw)
            self.cost = torch.zeros(self.R * self.S, dtype=torch.float32, **kw)
            self.nominal = torch.zeros((self.n_seg, self.R, 4), dtype=torch.int32, **kw)
            self.best = torch.zeros(self.R, dtype=torch.int32, **kw)
            self.best_cost = torch.zeros(self.R, dtype=torch.float32, **kw)
            self._sigma_cell = torch.tensor(self.sigma + (0.0,), dtype=torch.float32, **kw)
            self.sigma_table = self._sigma_cell.expand(self.n_seg, self.R, 4).contiguous()
            self._sigma_next = torch.empty_like(self.sigma_table)  # the refit's output when it shifts the plan
        self._keep = None

    def _stream(self):
        _cabi.check(self.lib.rk_set_device(self.dev_index))
        return C.c_void_p(torch.cuda.current_stream(self.dev_index).cuda_stream)

    def _table(self, t, shape, what):
        assert t.is_cuda and t.is_contiguous() and t.element_size() == 4 and tuple(t.shape) == shape, f"{what}: {tuple(shape)} 32-bit device tensor"
        return t.data_ptr()

    def sample(self, nominal=None, seed=None, sigma_table=None):
        """rk_plan_sample_commands: candidates around `nominal` (int32/float32 [n_seg, R, 4]; default the planner's own).
        With sigma_table (float32 [n_seg, R, 4], e.g. the planner's own) rk_plan_sample_commands_sigma: the noise scale of
        segment s of robot r is cell [s, r] instead of the planner's sigma."""
        nom = self._table(self.nominal if nominal is None else nominal, (self.n_seg, self.R, 4), "nominal")
        s = _cabi.PlanSample()
        s.first, s.seed = self.first, (self.seed if seed is None else int(seed)) & 0xFFFFFFFF
        s.sigma[:] = self.sigma
        tail = (self.R, self.S, self.n_seg, self.candidates.data_ptr(), self._stream())
        if sigma_table is None:
            _cabi.check(self.lib.rk_plan_sample_commands(C.byref(self.params), C.byref(s), nom, *tail))
        else:
            assert sigma_table.dtype == torch.float32, "sigma_table: float32"
            sig = self._table(sigma_table, (self.n_seg, self.R, 4), "sigma_table")
            _cabi.check(self.lib.rk_plan_sample_commands_sigma(C.byref(self.params), C.byref(s), nom, sig, *tail))
        return self.candidates

    def rollout(self, src, ref, w_pos, w_goal, w_cur, obstacles=None, w_obst=0.0, check_period=None):
        """rk_plan_rollout: every candidate from its robot's state in `src` (a VehicleBatch of R robots, left untouched),
        ranked against ref (float32 [n_seg, R, 2], metres: where each robot should be when each segment ends).

        obstacles: keep-out discs, float32 [m, R, 4] = {cx, cy, radius, unused} in metres per robot (one world shared by
        all robots: t.expand(m, R, 4).contiguous()).  Then rk_plan_rollout_obstacles adds w_obst * (radius^2 - d^2) for
        every disc a candidate is inside of, every check_period ticks (default seg_len; it must divide seg_len);
        w_obst = inf makes any penetrating candidate cost +inf."""
        assert src.n == self.R, "the source batch must hold the planner's R robots"
        assert ref.is_cuda and ref.is_contiguous() and ref.dtype == torch.float32 and tuple(ref.shape) == (self.n_seg, self.R, 2)
        c = _cabi.PlanCost()
        c.d_ref, c.w_pos, c.w_goal, c.w_cur = ref.data_ptr(), float(w_pos), float(w_goal), float(w_cur)
        args = (C.byref(self.params), src.state.data_ptr(), self.R, self.S, self.candidates.data_ptr(), self.n_seg, self.seg_len, C.byref(c))
        if obstacles is None:
            self._keep = ref
            _cabi.check(self.lib.rk_plan_rollout(*args, self.cost.data_ptr(), self._stream()))
            return self.cost
        assert (obstacles.is_cuda and obstacles.is_contiguous() and obstacles.dtype == torch.float32 and obstacles.dim() == 3
                and tuple(obstacles.shape[1:]) == (self.R, 4)), "obstacles: float32 [m, R, 4] contiguous device tensor"
        o = _cabi.PlanObstacles()
        o.d_obs, o.m = obstacles.data_ptr(), obstacles.shape[0]
        o.check_period = self.seg_len if check_period is None else int(check_period)
        o.w_obst = float(w_obst)
        self._keep = (ref, obstacles)
        _cabi.check(self.lib.rk_plan_rollout_obstacles(*args, C.byref(o), self.cost.data_ptr(), self._stream()))
        return self.cost

    def select(self, lam, shift=1):
        """rk_plan_select into the planner's nominal: lam == 0 takes the best candidate, lam > 0 the MPPI-weighted mean;
        shift = 1 moves the plan on by the segment about to be executed (the last segment is repeated)."""
        _cabi.check(self.lib.rk_plan_select(self.cost.data_ptr(), self.candidates.data_ptr(), self.R, self.S, self.n_seg, float(lam),
                                            int(shift), self.nominal.data_ptr(), self.best.data_ptr(), self.best_cost.data_ptr(),
                                            self._stream()))
        return self.nominal

    def refit(self, elite, alpha=0.0, sigma_min=(0.0, 0.0, 0.0), shift=1):
        """rk_plan_refit of the planner's nominal and sigma_table to the `elite` best candidates of the last rollout (alpha:
        smoothing toward the previous distribution; sigma_min: floor of the new sigma); also sets best / best_cost.
        shift as in select.  With shift != 0 the new table is written to a second buffer that then becomes sigma_table."""
        rf = _cabi.PlanRefit()
        rf.elite, rf.alpha = int(elite), float(alpha)
        rf.sigma_min[:] = tuple(float(x) for x in sigma_min)
        out = self.sigma_table if shift == 0 else self._sigma_next  # in place only without a shift
        _cabi.check(self.lib.rk_plan_refit(self.cost.data_ptr(), self.candidates.data_ptr(), self.sigma_table.data_ptr(), self.R, self.S,
                                           self.n_seg, C.byref(rf), int(shift), self.nominal.data_ptr(), out.data_ptr(),
                                           self.best.data_ptr(), self.best_cost.data_ptr(), self._stream()))
        if out is not self.sigma_table:
            self.sigma_table, self._sigma_next = out, self.sigma_table
        return self.nominal

    def plan(self, src, ref, w_pos, w_goal, w_cur, lam=0.0, shift=1, seed=None, obstacles=None, w_obst=0.0, check_period=None):
        """One planning step (sample, rollout, select) on the current torch stream; returns the new nominal."""
        self.sample(seed=seed)
        self.rollout(src, ref, w_pos, w_goal, w_cur, obstacles=obstacles, w_obst=w_obst, check_period=check_period)
        return self.select(lam, shift)

    def plan_cem(self, src, ref, w_pos, w_goal, w_cur, iters, elite, alpha=0.0, sigma_min=(0.0, 0.0, 0.0), shift=1, seed=None,
                 obstacles=None, w_obst=0.0, check_period=None):
        """One cross-entropy planning step on the current torch stream; returns the new nominal.

        sigma_table is reset to the planner's sigma, then `iters` rounds of sample (around the nominal, with the table) ->
        rollout (obstacles as in rollout) -> refit to the `elite` best candidates.  Every round but the last refits with
        shift = 0, so that the next round samples around the same segments; the last one with `shift`.  Round i draws with
        seed (seed + i * 0x9E3779B9) mod 2^32 (seed: the planner's own when None).  iters = 1, elite = 1, alpha = 0 is
        plan(..., lam=0) bit for bit while no cost is -inf (never, with non-negative weights).  NaN and +-inf costs are never
        elites, but the elite mean, like the MPPI blend, may pass between two detours around a disc."""
        assert int(iters) >= 1, "iters >= 1"
        base = self.seed if seed is None else int(seed)
        self.sigma_table.copy_(self._sigma_cell.expand_as(self.sigma_table))
        for i in range(int(iters)):
            self.sample(seed=(base + i * 0x9E3779B9) & 0xFFFFFFFF, sigma_table=self.sigma_table)
            self.rollout(src, ref, w_pos, w_goal, w_cur, obstacles=obstacles, w_obst=w_obst, check_period=check_period)
            self.refit(elite, alpha, sigma_min, shift if i == int(iters) - 1 else 0)
        return self.nominal

    def first_command(self):
        """The command the robots execute next: a [1, R, 4] view of the nominal, ready for
        VehicleBatch.rollout(seg_len, cmd=planner.first_command(), seg_len=seg_len)."""
        return self.nominal[:1]
