"""Sampling planner for the vehicle over the C-ABI (rk_plan_* in include/robotick.h), torch owning the buffers.

One planning step for R robots with S candidates each: sample candidate command tables around the nominal plan, roll
every candidate out from its robot's current state and rank it by a stage cost, then pick (argmin) or blend (MPPI) the
candidates into the next nominal plan.  Candidate j of robot r is column r*S + j of every table.
"""
import ctypes as C

import torch

from . import _cabi
from .vehicle import _dev_index


class VehiclePlanner:
    """Owns the candidate table int32 [n_seg, R*S, 4] (rk_vdt_cmd_t records), the cost float32 [R*S], the nominal plan
    int32 [n_seg, R, 4], and best (int32 [R]) / best_cost (float32 [R]) of the last selection.  Every call is
    asynchronous on the current torch stream of the planner's device.

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
        self._keep = None

    def _stream(self):
        _cabi.check(self.lib.rk_set_device(self.dev_index))
        return C.c_void_p(torch.cuda.current_stream(self.dev_index).cuda_stream)

    def _table(self, t, shape, what):
        assert t.is_cuda and t.is_contiguous() and t.element_size() == 4 and tuple(t.shape) == shape, f"{what}: {tuple(shape)} 32-bit device tensor"
        return t.data_ptr()

    def sample(self, nominal=None, seed=None):
        """rk_plan_sample_commands: candidates around `nominal` (int32/float32 [n_seg, R, 4]; default the planner's own)."""
        nom = self.nominal if nominal is None else nominal
        s = _cabi.PlanSample()
        s.first, s.seed = self.first, (self.seed if seed is None else int(seed)) & 0xFFFFFFFF
        s.sigma[:] = self.sigma
        _cabi.check(self.lib.rk_plan_sample_commands(C.byref(self.params), C.byref(s), self._table(nom, (self.n_seg, self.R, 4), "nominal"),
                                                     self.R, self.S, self.n_seg, self.candidates.data_ptr(), self._stream()))
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

    def plan(self, src, ref, w_pos, w_goal, w_cur, lam=0.0, shift=1, seed=None, obstacles=None, w_obst=0.0, check_period=None):
        """One planning step (sample, rollout, select) on the current torch stream; returns the new nominal."""
        self.sample(seed=seed)
        self.rollout(src, ref, w_pos, w_goal, w_cur, obstacles=obstacles, w_obst=w_obst, check_period=check_period)
        return self.select(lam, shift)

    def first_command(self):
        """The command the robots execute next: a [1, R, 4] view of the nominal, ready for
        VehicleBatch.rollout(seg_len, cmd=planner.first_command(), seg_len=seg_len)."""
        return self.nominal[:1]
