"""Sampling planner for the vehicle over the C-ABI (rk_plan_* in include/robotick.h), torch owning the buffers.

One planning step for R robots with S candidates each: sample candidate command tables around the nominal plan, roll
every candidate out from its robot's current state and rank it by a stage cost, then pick (argmin) or blend (MPPI) the
candidates into the next nominal plan.  Candidate j of robot r is column r*S + j of every table.  The cross-entropy
method (plan_cem) runs several sample -> rollout -> refit rounds per step, refitting a per-robot, per-segment mean and
sigma to each round's elite candidates.  For fleets, predict() gives where each robot's nominal plan takes it and
peer_discs() turns those paths into moving keep-out discs for the robot's peers (fleet_peers builds the usual grouping).
A CostMap, a grid of cell costs shared by the robots of a world, prices walls and shelving at every checkpoint, alone or
together with discs; its cost_to_go() builds CostToGo fields, shortest-path distances to goals around the walls, that
price each candidate's end position instead of the straight line to the goal.  CostMap.inflate prices every cell by its
distance to the nearest wall through an inflation_table, so that plans and paths keep the robot's body clear of walls.
"""
import ctypes as C

import torch

from . import _cabi
from .vehicle import _dev_index


class CostMap:
    """A cost grid for rk_plan_rollout_map: cells float32 [H, W] (one world) or [n_maps, H, W], contiguous, on the
    planner's device; cell (ix, iy) of map k covers x in [x0 + ix*resolution, x0 + (ix+1)*resolution) and likewise y, with
    (x0, y0) = origin in metres.  A point off the grid reads `outside` (+inf: leaving the grid is a hard wall).  map_of:
    int32 [R] device tensor, the map of each robot (an index outside [0, n_maps) gives that robot no map term); None: map 0
    for every robot.  Cells above 0 add w_map * cell to a candidate's cost at every checkpoint; zero, negative and NaN cells
    add nothing.  The robot is a point read at checkpoints: inflate walls by the body radius plus the distance covered in
    check_period ticks (inflate, inflation_table).  Cells may be changed in place between planning steps.

    inv_res = float32(1 / resolution) is computed once here and passed as is, so a restatement can use the same bits;
    x0, y0 and outside are likewise the float32 values the device reads."""

    def __init__(self, cells, origin, resolution, outside=float("inf"), map_of=None):
        assert (cells.is_cuda and cells.is_contiguous() and cells.dtype == torch.float32 and cells.dim() in (2, 3)
                and cells.numel() > 0), "cells: float32 [H, W] or [n_maps, H, W] contiguous device tensor"
        self.cells = cells if cells.dim() == 3 else cells[None]
        self.n_maps, self.height, self.width = (int(d) for d in self.cells.shape)
        resolution = float(resolution)
        assert resolution > 0 and resolution < float("inf"), "resolution: metres per cell, finite and > 0"
        self.resolution = resolution
        self.x0, self.y0 = (C.c_float(float(v)).value for v in origin)
        self.inv_res = C.c_float(1.0 / resolution).value
        self.outside = C.c_float(float(outside)).value
        if map_of is not None:
            assert (map_of.is_cuda and map_of.is_contiguous() and map_of.dtype == torch.int32 and map_of.dim() == 1
                    and map_of.device == cells.device), "map_of: int32 [R] contiguous tensor on the cells' device"
        self.map_of = map_of

    def struct(self, w_map):
        """The rk_plan_map_t of this map with weight w_map."""
        m = _cabi.PlanMap()
        m.d_cells, m.d_map_of = self.cells.data_ptr(), None if self.map_of is None else self.map_of.data_ptr()
        m.n_maps, m.width, m.height = self.n_maps, self.width, self.height
        m.x0, m.y0, m.inv_res, m.outside, m.w_map = self.x0, self.y0, self.inv_res, self.outside, float(w_map)
        return m

    def cost_to_go(self, goals, size=None, offsets=None, k_cost=0.0, lethal=float("inf"), field_map=None, field_of=None,
                   outside=float("inf")):
        """rk_plan_cost_to_go on the current torch stream of the map's device (the call synchronises it): one field per goal,
        the shortest-path distance in metres from goals[f] (float32 [n_fields, 2], metres) through the cells below `lethal`,
        each step weighted by 1 + k_cost * cell for cells above 0, with no corner cutting.  size = (fh, fw): the window of
        every field (default: the whole map); offsets: int32 [n_fields, 2], the map cell (ox, oy) of window cell (0, 0)
        (default 0, 0); field_map: int32 [n_fields], the map of each field (default map 0).  field_of and outside go to
        the returned CostToGo.  Build fields when goals or the map change, not every planning step."""
        dev = self.cells.device
        goals = torch.as_tensor(goals, dtype=torch.float32, device=dev).contiguous()
        assert goals.dim() == 2 and goals.shape[1] == 2 and goals.shape[0] >= 1, "goals: float32 [n_fields, 2]"
        n = goals.shape[0]
        fh, fw = (self.height, self.width) if size is None else (int(size[0]), int(size[1]))
        if offsets is not None:
            offsets = torch.as_tensor(offsets, dtype=torch.int32, device=dev).contiguous()
            assert tuple(offsets.shape) == (n, 2), f"offsets: int32 [{n}, 2]"
        if field_map is not None:
            field_map = torch.as_tensor(field_map, dtype=torch.int32, device=dev).contiguous()
            assert tuple(field_map.shape) == (n,), f"field_map: int32 [{n}]"
        lib = _cabi.load()
        work_bytes = lib.rk_plan_cost_to_go_work_bytes(n, fw, fh)
        assert work_bytes > 0, "n_fields, fw, fh >= 1, fw, fh <= 2^24 and n_fields * fh * fw < 2^31"
        field = torch.empty((n, fh, fw), dtype=torch.float32, device=dev)
        work = torch.empty((work_bytes + 3) // 4, dtype=torch.int32, device=dev)
        spec = _cabi.PlanCtg()
        spec.step_axial = C.c_float(self.resolution).value
        spec.step_diag = C.c_float(self.resolution * 2.0 ** 0.5).value
        spec.k_cost, spec.lethal = float(k_cost), float(lethal)
        rounds = C.c_int32(0)
        di = _dev_index(dev)
        _cabi.check(lib.rk_set_device(di))
        mp = self.struct(0.0)
        _cabi.check(lib.rk_plan_cost_to_go(C.byref(mp), C.byref(spec), goals.data_ptr(), None if field_map is None else field_map.data_ptr(),
                                           None if offsets is None else offsets.data_ptr(), n, fw, fh, field.data_ptr(), work.data_ptr(),
                                           C.byref(rounds), C.c_void_p(torch.cuda.current_stream(di).cuda_stream)))
        ctg = CostToGo(field, self, offsets=offsets, field_of=field_of, outside=outside)
        ctg.rounds = rounds.value
        return ctg

    def inflate(self, table, lethal=float("inf")):
        """rk_plan_inflate on the current torch stream of the map's device (asynchronous): a new CostMap with the same
        origin, resolution, outside and map_of whose cell at squared cell distance d2 from the nearest obstacle of its map
        (a cell >= lethal; off the grid too when outside >= lethal) is the larger of the cell and table[d2] for
        d2 < len(table), the cell itself otherwise.  table: float32 [n] on the map's device, 1 <= n <= 65536
        (inflation_table)."""
        dev = self.cells.device
        assert (table.is_cuda and table.device == dev and table.is_contiguous() and table.dtype == torch.float32 and table.dim() == 1
                and 1 <= table.numel() <= 65536), "table: float32 [n] contiguous tensor on the map's device, 1 <= n <= 65536"
        lib = _cabi.load()
        cells = torch.empty_like(self.cells)
        work = torch.empty((lib.rk_plan_inflate_work_bytes(self.n_maps, self.width, self.height) + 3) // 4, dtype=torch.int32, device=dev)
        spec = _cabi.PlanInflate()
        spec.d_table, spec.n_table, spec.lethal = table.data_ptr(), table.numel(), float(lethal)
        di = _dev_index(dev)
        _cabi.check(lib.rk_set_device(di))
        mp = self.struct(0.0)
        _cabi.check(lib.rk_plan_inflate(C.byref(mp), C.byref(spec), cells.data_ptr(), work.data_ptr(),
                                        C.c_void_p(torch.cuda.current_stream(di).cuda_stream)))
        return CostMap(cells, (self.x0, self.y0), self.resolution, outside=self.outside, map_of=self.map_of)


def inflation_table(resolution, inscribed, radius, scaling=0.0, peak=1.0, lethal=float("inf"), device="cuda:0"):
    """The ROS-style inflation profile for CostMap.inflate: float32 [n] on `device`, entry d2 the cost at d = sqrt(d2) *
    resolution metres (float64) from the nearest obstacle: `lethal` where d <= inscribed, peak * exp(-scaling * (d -
    inscribed)) beyond, and the table ends at the last d2 whose d <= radius (at most 255 cells).  The comparisons are in
    float64, so a radius or inscribed radius that is an exact multiple of the resolution may fall just short of it.

    inscribed: the body's radius (for a body that is not round, its circumscribed radius: plan rollouts hold the heading,
    so a disc footprint is the right model) plus 0.4 * P mm for the distance covered between two checkpoints P ticks
    apart.  Make the lethal value at least the `lethal` of cost_to_go, so that the inflated wall blocks its paths."""
    resolution, inscribed, radius = float(resolution), float(inscribed), float(radius)
    assert 0.0 < resolution < float("inf"), "resolution: metres per cell, finite and > 0"
    d = torch.arange(65537, dtype=torch.float64).sqrt() * resolution
    n = int((d <= radius).sum())
    assert 1 <= n <= 65536, "radius: >= 0 and at most 255 cells"
    d = d[:n]
    v = torch.where(d <= inscribed, torch.full_like(d, float(lethal)), float(peak) * torch.exp(-float(scaling) * (d - inscribed)))
    return v.to(torch.float32).to(device)


class CostToGo:
    """A cost-to-go field for rk_plan_rollout_field: field float32 [n_fields, fh, fw] (CostMap.cost_to_go's, or any caller's
    grid) on the grid of `costmap` (its origin and resolution); offsets int32 [n_fields, 2], the grid cell of each
    window's cell (0, 0) (None: 0, 0); field_of int32 [R], the field of each robot (None: field 0; an index outside
    [0, n_fields) adds no term); outside: the value off a window.  The term w_field * cell is added once, at the end of
    each candidate's rollout; a +inf cell (blocked or unreachable) prices the candidate at +inf.  rounds: the relaxation
    rounds of the build (None for a caller's grid)."""

    def __init__(self, field, costmap, offsets=None, field_of=None, outside=float("inf")):
        assert (field.is_cuda and field.is_contiguous() and field.dtype == torch.float32 and field.dim() == 3
                and field.numel() > 0), "field: float32 [n_fields, fh, fw] contiguous device tensor"
        self.field, self.costmap = field, costmap
        self.n_fields, self.fh, self.fw = (int(d) for d in field.shape)
        for t, shape, what in ((offsets, (self.n_fields, 2), "offsets"), (field_of, None, "field_of")):
            if t is not None:
                assert (t.is_cuda and t.is_contiguous() and t.dtype == torch.int32 and t.device == field.device
                        and (shape is None and t.dim() == 1 or tuple(t.shape) == shape)), f"{what}: int32 contiguous tensor on the field's device"
        self.offsets, self.field_of = offsets, field_of
        self.outside = C.c_float(float(outside)).value
        self.rounds = None

    def struct(self, w_field):
        """The rk_plan_field_t of this field with weight w_field."""
        f = _cabi.PlanField()
        f.d_field = self.field.data_ptr()
        f.d_field_of = None if self.field_of is None else self.field_of.data_ptr()
        f.d_offset = None if self.offsets is None else self.offsets.data_ptr()
        f.n_fields, f.fw, f.fh = self.n_fields, self.fw, self.fh
        cm = self.costmap
        f.x0, f.y0, f.inv_res, f.outside, f.w_field = cm.x0, cm.y0, cm.inv_res, self.outside, float(w_field)
        return f


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
            self._pred_cost = torch.zeros(self.R, dtype=torch.float32, **kw)  # predict(): the S = 1 rollout's unused cost
            self._pred_ref = torch.zeros((self.n_seg, self.R, 2), dtype=torch.float32, **kw)
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

    def n_ck(self, check_period):
        """Checkpoints of a plan rollout every check_period ticks: n_seg * seg_len / check_period."""
        P = int(check_period)
        assert P >= 1 and self.seg_len % P == 0, "check_period must divide seg_len"
        return self.n_seg * self.seg_len // P

    def rollout(self, src, ref, w_pos, w_goal, w_cur, obstacles=None, w_obst=0.0, check_period=None, path=None, costmap=None, w_map=0.0,
                field=None, w_field=0.0):
        """rk_plan_rollout: every candidate from its robot's state in `src` (a VehicleBatch of R robots, left untouched),
        ranked against ref (float32 [n_seg, R, 2], metres: where each robot should be when each segment ends).

        obstacles: keep-out discs, float32 [m, R, 4] = {cx, cy, radius, unused} in metres per robot (one world shared by
        all robots: t.expand(m, R, 4).contiguous()).  Then rk_plan_rollout_obstacles adds w_obst * (radius^2 - d^2) for
        every disc a candidate is inside of, every check_period ticks (default seg_len; it must divide seg_len);
        w_obst = inf makes any penetrating candidate cost +inf.  A 4-D table float32 [n_ck, m, R, 4] (n_ck =
        self.n_ck(check_period)) gives each checkpoint its own discs (rk_plan_rollout_moving): moving obstacles, or the
        peers' predicted paths (peer_discs).

        path: float32 [n_ck, R*S, 2], receives every candidate's position at every checkpoint (rk_plan_rollout_moving; with
        a 4-D table or no obstacles).  It never changes the cost.

        costmap (a CostMap on the planner's device): rk_plan_rollout_map adds w_map * cell at every checkpoint (cells > 0
        only; w_map = inf makes every such cell a hard wall), into the same sum as the discs.  Without obstacles the
        checkpoints are every check_period ticks (default seg_len) with no discs.  A 3-D static disc table is then repeated
        for every checkpoint (obstacles.expand(n_ck, m, R, 4).contiguous(), the same bits as the static table): a copy of
        n_ck * m * R * 16 bytes written on every call, so pass a 4-D table to keep one.

        field (a CostToGo on the planner's device): rk_plan_rollout_field adds w_field * cell (cells > 0 only; finite
        w_field) of the robot's field under each candidate's end position, once, after the last checkpoint; costmap may
        then be None.  With a field, drop w_pos and keep w_goal small (INTEGRATION.md §2)."""
        assert src.n == self.R, "the source batch must hold the planner's R robots"
        assert ref.is_cuda and ref.is_contiguous() and ref.dtype == torch.float32 and tuple(ref.shape) == (self.n_seg, self.R, 2)
        c = _cabi.PlanCost()
        c.d_ref, c.w_pos, c.w_goal, c.w_cur = ref.data_ptr(), float(w_pos), float(w_goal), float(w_cur)
        args = (C.byref(self.params), src.state.data_ptr(), self.R, self.S, self.candidates.data_ptr(), self.n_seg, self.seg_len, C.byref(c))
        if costmap is not None:
            assert costmap.cells.device.index == self.dev_index, "costmap: on the planner's device"
            assert costmap.map_of is None or costmap.map_of.shape[0] == self.R, f"costmap.map_of: int32 [{self.R}]"
        if field is not None:
            assert field.field.device.index == self.dev_index, "field: on the planner's device"
            assert field.field_of is None or field.field_of.shape[0] == self.R, f"field.field_of: int32 [{self.R}]"
        if (costmap is not None or field is not None) and obstacles is not None and obstacles.dim() == 3:
            obstacles = obstacles.expand(self.n_ck(self.seg_len if check_period is None else check_period), *obstacles.shape).contiguous()
        if obstacles is None and path is None and costmap is None and field is None:
            self._keep = ref
            _cabi.check(self.lib.rk_plan_rollout(*args, self.cost.data_ptr(), self._stream()))
            return self.cost
        P = self.seg_len if check_period is None else int(check_period)
        o = _cabi.PlanObstacles()
        o.check_period, o.w_obst = P, float(w_obst)
        if obstacles is not None:
            assert (obstacles.is_cuda and obstacles.is_contiguous() and obstacles.dtype == torch.float32 and obstacles.dim() in (3, 4)
                    and tuple(obstacles.shape[-2:]) == (self.R, 4)), "obstacles: float32 [m, R, 4] or [n_ck, m, R, 4] contiguous device tensor"
            o.d_obs, o.m = obstacles.data_ptr(), obstacles.shape[-3]
        self._keep = (ref, obstacles, path)
        if obstacles is not None and obstacles.dim() == 3:
            assert path is None, "path: with a 4-D obstacles table or none"
            _cabi.check(self.lib.rk_plan_rollout_obstacles(*args, C.byref(o), self.cost.data_ptr(), self._stream()))
            return self.cost
        n_ck = self.n_ck(P)
        assert obstacles is None or obstacles.shape[0] == n_ck, f"obstacles: {n_ck} checkpoint tables of [m, R, 4]"
        if path is not None:
            assert (path.is_cuda and path.is_contiguous() and path.dtype == torch.float32
                    and tuple(path.shape) == (n_ck, self.R * self.S, 2)), f"path: float32 [{n_ck}, {self.R * self.S}, 2] device tensor"
        pth = None if path is None else path.data_ptr()
        if costmap is None and field is None:
            _cabi.check(self.lib.rk_plan_rollout_moving(*args, C.byref(o), pth, self.cost.data_ptr(), self._stream()))
        elif field is None:
            self._keep = (ref, obstacles, path, costmap)
            mp = costmap.struct(w_map)
            _cabi.check(self.lib.rk_plan_rollout_map(*args, C.byref(o), C.byref(mp), pth, self.cost.data_ptr(), self._stream()))
        else:
            self._keep = (ref, obstacles, path, costmap, field)
            mp = None if costmap is None else C.byref(costmap.struct(w_map))
            fd = field.struct(w_field)
            _cabi.check(self.lib.rk_plan_rollout_field(*args, C.byref(o), mp, C.byref(fd), pth, self.cost.data_ptr(), self._stream()))
        return self.cost

    def predict(self, src, check_period):
        """Where each robot's nominal plan takes it from its state in `src`: float32 [n_ck, R, 2], metres, the position at
        every checkpoint (ticks check_period - 1, 2*check_period - 1, ...).  rk_plan_rollout_moving with S = 1, the nominal
        as the candidates, no discs and a path."""
        assert src.n == self.R, "the source batch must hold the planner's R robots"
        n_ck = self.n_ck(check_period)
        path = torch.empty((n_ck, self.R, 2), dtype=torch.float32, device=self.device)
        c = _cabi.PlanCost()
        c.d_ref = self._pred_ref.data_ptr()
        o = _cabi.PlanObstacles()
        o.check_period = int(check_period)
        _cabi.check(self.lib.rk_plan_rollout_moving(C.byref(self.params), src.state.data_ptr(), self.R, 1, self.nominal.data_ptr(), self.n_seg,
                                                    self.seg_len, C.byref(c), C.byref(o), path.data_ptr(), self._pred_cost.data_ptr(),
                                                    self._stream()))
        return path

    def peer_discs(self, path, peers, radius, out=None, k0=0):
        """rk_plan_peer_discs: for every checkpoint, disc k0 + k of robot r is centred where robot peers[k, r] is predicted
        to be, with `radius` (metres: the sum of the two bodies' radii and a margin); a peer index outside [0, R) or equal
        to r gives a disc that contributes nothing.  path: float32 [n_ck, R, 2] (predict); peers: int32 [m, R].
        out: float32 [n_ck, M, R, 4] whose slots k0 .. k0+m-1 are written and the others left as they are (default: a new
        [n_ck, m, R, 4] table, k0 = 0).  Returns the table, ready for rollout / plan(obstacles=...)."""
        n_ck = path.shape[0]
        assert (path.is_cuda and path.is_contiguous() and path.dtype == torch.float32
                and tuple(path.shape) == (n_ck, self.R, 2)), "path: float32 [n_ck, R, 2] device tensor"
        assert (peers.is_cuda and peers.is_contiguous() and peers.dtype == torch.int32 and peers.dim() == 2
                and peers.shape[1] == self.R), "peers: int32 [m, R] device tensor"
        m = peers.shape[0]
        if out is None:
            assert k0 == 0, "k0 > 0 needs out"
            out = torch.empty((n_ck, m, self.R, 4), dtype=torch.float32, device=self.device)
        assert (out.is_cuda and out.is_contiguous() and out.dtype == torch.float32 and out.dim() == 4
                and out.shape[0] == n_ck and tuple(out.shape[2:]) == (self.R, 4)), "out: float32 [n_ck, M, R, 4] device tensor"
        _cabi.check(self.lib.rk_plan_peer_discs(path.data_ptr(), self.R, n_ck, peers.data_ptr(), m, float(radius), out.data_ptr(), out.shape[1],
                                                int(k0), self._stream()))
        return out

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

    def plan(self, src, ref, w_pos, w_goal, w_cur, lam=0.0, shift=1, seed=None, obstacles=None, w_obst=0.0, check_period=None,
             costmap=None, w_map=0.0, field=None, w_field=0.0):
        """One planning step (sample, rollout, select) on the current torch stream; returns the new nominal.  obstacles
        (3-D static or 4-D per-checkpoint discs), costmap and field as in rollout."""
        self.sample(seed=seed)
        self.rollout(src, ref, w_pos, w_goal, w_cur, obstacles=obstacles, w_obst=w_obst, check_period=check_period, costmap=costmap,
                     w_map=w_map, field=field, w_field=w_field)
        return self.select(lam, shift)

    def plan_cem(self, src, ref, w_pos, w_goal, w_cur, iters, elite, alpha=0.0, sigma_min=(0.0, 0.0, 0.0), shift=1, seed=None,
                 obstacles=None, w_obst=0.0, check_period=None, costmap=None, w_map=0.0, field=None, w_field=0.0):
        """One cross-entropy planning step on the current torch stream; returns the new nominal.

        sigma_table is reset to the planner's sigma, then `iters` rounds of sample (around the nominal, with the table) ->
        rollout (obstacles, costmap and field as in rollout) -> refit to the `elite` best candidates.  Every round but the last refits with
        shift = 0, so that the next round samples around the same segments; the last one with `shift`.  Round i draws with
        seed (seed + i * 0x9E3779B9) mod 2^32 (seed: the planner's own when None).  iters = 1, elite = 1, alpha = 0 is
        plan(..., lam=0) bit for bit while no cost is -inf (never, with non-negative weights).  NaN and +-inf costs are never
        elites, but the elite mean, like the MPPI blend, may pass between two detours around a disc."""
        assert int(iters) >= 1, "iters >= 1"
        base = self.seed if seed is None else int(seed)
        self.sigma_table.copy_(self._sigma_cell.expand_as(self.sigma_table))
        for i in range(int(iters)):
            self.sample(seed=(base + i * 0x9E3779B9) & 0xFFFFFFFF, sigma_table=self.sigma_table)
            self.rollout(src, ref, w_pos, w_goal, w_cur, obstacles=obstacles, w_obst=w_obst, check_period=check_period, costmap=costmap,
                         w_map=w_map, field=field, w_field=w_field)
            self.refit(elite, alpha, sigma_min, shift if i == int(iters) - 1 else 0)
        return self.nominal

    def first_command(self):
        """The command the robots execute next: a [1, R, 4] view of the nominal, ready for
        VehicleBatch.rollout(seg_len, cmd=planner.first_command(), seg_len=seg_len)."""
        return self.nominal[:1]


def fleet_peers(R, G, device="cuda:0"):
    """int32 [G-1, R] peer table of fleets of G robots: robot r belongs to group r // G, and its peers are the other G-1
    robots of the group in ascending order (-1 where a short last group has fewer; such a disc contributes nothing)."""
    R, G = int(R), int(G)
    assert R >= 0 and G >= 1, "R >= 0 and G >= 1"
    r = torch.arange(R, dtype=torch.int64)
    j = torch.arange(G - 1, dtype=torch.int64)[:, None]  # peer slot k
    rank = r % G
    q = (r - rank)[None, :] + j + (j >= rank[None, :]).to(torch.int64)  # skip the robot itself
    return torch.where(q < R, q, -1).to(torch.int32).contiguous().to(device)
