"""CPU: moving keep-out discs and fleet planning (rk_plan_rollout_moving, rk_plan_peer_discs) -- the host restatement's
own equalities with the static-disc cost, the peer-disc rules, the argument checks of both entries, and the circle swap
on the port (tests/plan_fleet_ref.py): without peer discs robots of a group collide, with them they keep apart and
still reach their goals."""
import ctypes as C

import numpy as np
import pytest

import plan_fleet_ref as pfr
import plan_obst_ref as por
import plan_ref as pr
import roboken_fmskf_robot_controller_b200 as rk
from roboken_fmskf_robot_controller_b200 import _cabi, build


@pytest.fixture(scope="module")
def lib():
    build.build()
    return rk.load()


def _buf(nbytes):
    b = (C.c_uint8 * (nbytes + 16))()
    return b, C.c_void_p((C.addressof(b) + 15) & ~15)


def _obst(d_obs, m, P, w):
    o = _cabi.PlanObstacles()
    o.d_obs, o.m, o.check_period, o.w_obst = d_obs, m, P, w
    return o


def _trace(rng, K, n):
    """Trace rows [K, 16, n] whose position words are uniform in [-0.2, 0.2] m."""
    tr = np.zeros((K, 16, n), dtype=np.uint32)
    xy = rng.uniform(-0.2, 0.2, (K, 2, n)).astype(np.float32)
    tr[:, 0], tr[:, 1] = xy[:, 0].view(np.uint32), xy[:, 1].view(np.uint32)
    return tr


def _static(rng, m, R):
    obs = np.zeros((m, R, 4), dtype=np.float32)
    obs[:, :, :2] = rng.uniform(-0.2, 0.2, (m, R, 2))
    obs[:, :, 2] = rng.uniform(0.02, 0.06, (m, R))
    if m:
        obs[0, 0, 2] = np.nan
    return obs


@pytest.mark.parametrize("P", [1, 4, 12])
@pytest.mark.parametrize("m", [0, 1, 5])
def test_repeated_table_is_the_static_cost(P, m):
    rng = np.random.default_rng(10 * P + m)
    R, S, K = 6, 5, 24
    tr = _trace(rng, K, R * S)
    obs = _static(rng, m, R)
    rep = np.ascontiguousarray(np.broadcast_to(obs, (K // P, m, R, 4)))
    got = pfr.moving_obstacle_cost(tr, rep, S, P, 7.0)
    np.testing.assert_array_equal(got.view(np.uint32), por.obstacle_cost(tr, obs, S, P, 7.0).view(np.uint32))
    if m == 0:
        assert (got == 0).all() and not np.signbit(got).any()  # J + O is then J, bit for bit
    else:
        assert (got > 0).any() and (got == 0).any()


def test_each_checkpoint_reads_its_own_table():
    rng = np.random.default_rng(3)
    R, S, K, P = 2, 3, 12, 4
    tr = _trace(rng, K, R * S)
    obs = np.zeros((K // P, 1, R, 4), dtype=np.float32)
    obs[:, 0, :, 2] = np.nan
    x, y = tr[2 * P - 1, 0, 4].view(np.float32), tr[2 * P - 1, 1, 4].view(np.float32)  # candidate 4 = robot 1, j = 1
    obs[1, 0, 1] = (x, y, 0.01, 0.0)  # on candidate 4 at checkpoint 2 only
    O = pfr.moving_obstacle_cost(tr, obs, S, P, 2.0)
    assert O[4] == np.float32(2.0) * (np.float32(0.01) * np.float32(0.01))
    assert (np.delete(O, 4) == 0).all()
    obs[1, 0, 1, 2] = np.nan  # the same disc at any other checkpoint is not seen
    obs[0, 0, 1], obs[2, 0, 1] = (x, y, 0.01, 0.0), (x, y, 0.01, 0.0)
    tr[P - 1, :2, 4], tr[3 * P - 1, :2, 4] = np.float32(1.0).view(np.uint32), np.float32(1.0).view(np.uint32)
    assert (pfr.moving_obstacle_cost(tr, obs, S, P, 2.0) == 0).all()


def test_paths_are_the_checkpoint_rows():
    rng = np.random.default_rng(4)
    tr = _trace(rng, 20, 7)
    p = pfr.paths(tr, 5)
    assert p.shape == (4, 7, 2)
    for c in range(4):
        np.testing.assert_array_equal(p[c, :, 0].view(np.uint32), tr[5 * c + 4, 0])
        np.testing.assert_array_equal(p[c, :, 1].view(np.uint32), tr[5 * c + 4, 1])


def test_peer_disc_rules():
    R, n_ck = 5, 3
    path = np.arange(n_ck * R * 2, dtype=np.float32).reshape(n_ck, R, 2)
    peers = np.array([[1, 0, -1, 3, 5], [2, 1 << 30, 0, -7, 4]], dtype=np.int32)  # self: robot 3 slot 0, robot 4 slot 1
    sentinel = np.full((n_ck, 4, R, 4), 9.0, dtype=np.float32)
    out = pfr.peer_discs(path, peers, 0.25, out=sentinel.copy(), k0=1)
    np.testing.assert_array_equal(out[:, 0], sentinel[:, 0])  # slots outside [k0, k0 + m) untouched
    np.testing.assert_array_equal(out[:, 3], sentinel[:, 3])
    for k in range(2):
        for r in range(R):
            q = peers[k, r]
            cell = out[:, 1 + k, r]
            if 0 <= q < R and q != r:
                np.testing.assert_array_equal(cell[:, :2], path[:, q])
                assert (cell[:, 2] == np.float32(0.25)).all() and (cell[:, 3] == 0).all()
            else:
                np.testing.assert_array_equal(cell.view(np.uint32), np.broadcast_to(pfr.NAN_DISC.view(np.uint32), (n_ck, 4)))


@pytest.mark.parametrize("R,G", [(8, 4), (10, 4), (6, 1), (5, 5), (0, 3)])
def test_fleet_peers(R, G):
    from roboken_fmskf_robot_controller_b200.planner import fleet_peers

    exp = pfr.fleet_peers(R, G)
    got = fleet_peers(R, G, device="cpu").numpy()
    assert got.dtype == np.int32 and got.shape == (G - 1, R)
    np.testing.assert_array_equal(got, exp)
    for r in range(R):
        mates = {q for q in range(R) if q // G == r // G and q != r}
        assert set(exp[:, r][exp[:, r] >= 0]) == mates


def test_moving_argument_errors(lib):
    p = rk.default_params()
    c = _cabi.PlanCost()
    keep, a = _buf(4096)
    c.d_ref = a.value
    roll = lib.rk_plan_rollout_moving
    bad = {
        "m < 0": (_obst(a.value, -1, 10, 1.0), None),
        "m > 0, d_obs NULL": (_obst(None, 2, 10, 1.0), None),
        "m > 0, d_obs not 16-byte aligned": (_obst(a.value + 8, 2, 10, 1.0), None),
        "P < 1": (_obst(a.value, 2, 0, 1.0), None),
        "seg_len % P != 0": (_obst(a.value, 2, 3, 1.0), None),
        "w_obst < 0": (_obst(a.value, 2, 5, -1.0), None),
        "w_obst NaN": (_obst(a.value, 2, 5, float("nan")), None),
        "obst NULL": (None, None),
        "d_path not 8-byte aligned": (_obst(a.value, 0, 5, 1.0), a.value + 4),
    }
    for what, (o, path) in bad.items():
        assert roll(C.byref(p), a, 1, 4, a, 2, 10, C.byref(c), None if o is None else C.byref(o), path, a, None) == 1, what
        assert b"rk_plan_rollout_moving" in lib.rk_last_error(), f"{what}: no message"
    ok = _obst(a.value, 2, 5, float("inf"))
    assert roll(C.byref(p), a, 1, 4, a, 2, 0, C.byref(c), C.byref(ok), None, a, None) == 1  # seg_len < 1
    assert roll(C.byref(p), a, -1, 4, a, 2, 10, C.byref(c), C.byref(ok), None, a, None) == 1
    assert roll(C.byref(p), C.c_void_p(a.value + 4), 1, 4, a, 2, 10, C.byref(c), C.byref(ok), None, a, None) == 1
    assert roll(None, a, 1, 4, a, 2, 10, C.byref(c), C.byref(ok), None, a, None) == 1
    # R == 0 is a no-op, with or without a path
    assert roll(C.byref(p), None, 0, 4, None, 2, 10, C.byref(c), C.byref(ok), None, None, None) == 0
    assert roll(C.byref(p), None, 0, 4, None, 2, 10, C.byref(c), C.byref(ok), a, None, None) == 0


def test_peer_disc_argument_errors(lib):
    keep, a = _buf(1 << 14)
    path, peer, obs = a.value, a.value + 4096, a.value + 8192
    f = lib.rk_plan_peer_discs
    bad = {
        "R < 0": (path, -1, 2, peer, 1, 0.1, obs, 1, 0),
        "n_ck < 0": (path, 4, -1, peer, 1, 0.1, obs, 1, 0),
        "m < 0": (path, 4, 2, peer, -1, 0.1, obs, 1, 0),
        "k0 < 0": (path, 4, 2, peer, 1, 0.1, obs, 2, -1),
        "k0 + m > M": (path, 4, 2, peer, 2, 0.1, obs, 2, 1),
        "radius NaN": (path, 4, 2, peer, 1, float("nan"), obs, 1, 0),
        "radius inf": (path, 4, 2, peer, 1, float("inf"), obs, 1, 0),
        "radius < 0": (path, 4, 2, peer, 1, -0.1, obs, 1, 0),
        "d_path NULL": (None, 4, 2, peer, 1, 0.1, obs, 1, 0),
        "d_path misaligned": (path + 4, 4, 2, peer, 1, 0.1, obs, 1, 0),
        "d_peer NULL": (path, 4, 2, None, 1, 0.1, obs, 1, 0),
        "d_peer misaligned": (path, 4, 2, peer + 2, 1, 0.1, obs, 1, 0),
        "d_obs NULL": (path, 4, 2, peer, 1, 0.1, None, 1, 0),
        "d_obs misaligned": (path, 4, 2, peer, 1, 0.1, obs + 8, 1, 0),
        "d_obs overlapping d_path": (path, 4, 2, peer, 1, 0.1, path + 48, 1, 0),
    }
    for what, args in bad.items():
        assert f(*args, None) == 1, what
        assert b"rk_plan_peer_discs" in lib.rk_last_error(), f"{what}: no message"
    # nothing to write is a no-op
    for args in ((None, 0, 2, None, 1, 0.1, None, 1, 0), (None, 4, 0, None, 1, 0.1, None, 1, 0), (None, 4, 2, None, 0, 0.1, None, 3, 3)):
        assert f(*args, None) == 0


def test_fleet_entries_fail_without_a_device(lib):
    import torch

    if torch.cuda.is_available():
        pytest.skip("a GPU is present")
    p = rk.default_params()
    c = _cabi.PlanCost()
    keep, a = _buf(1 << 16)
    c.d_ref = a.value
    b = C.c_void_p(a.value + 32768)
    o = _obst(a.value, 1, 5, 2.0)
    assert lib.rk_plan_rollout_moving(C.byref(p), a, 1, 4, b, 2, 10, C.byref(c), C.byref(o), a.value + 1024, a, None) == 2
    assert b"no CPU fallback" in lib.rk_last_error()
    assert lib.rk_plan_peer_discs(a.value, 4, 2, a.value + 4096, 1, 0.1, a.value + 8192, 1, 0, None) == 2
    assert b"no CPU fallback" in lib.rk_last_error()


# The circle swap on the port: 2 groups of 4 robots on a 0.15 m circle (1 m apart), each heading for the antipodal point,
# 64 candidates of 4 x 50-tick segments, 40 planning steps with shift = 0.  Bodies of radius 15 mm: two robots collide
# closer than 30 mm.  Peer discs of radius 2 * 15 mm + 40 mm with a finite weight: the margin covers the closing distance
# over P = 5 ticks (2 * 0.4 mm per tick) and the lag of the prediction (with shift = 0 the nominal still starts with the
# segment just executed, so predict replays it).  Observed on the port: without peer discs group 0 comes to 1.4 mm (group
# 1 to 41 mm); with them the least distances are 38.9 mm and 68.2 mm, and every robot ends 7.6 - 41.7 mm from its goal.
FLEET = dict(groups=2, G=4, circle=0.15, spacing=1.0, S=64, n_seg=4, seg_len=50, P=5, steps=40, w_pos=1.0, w_goal=10.0, w_cur=1e-9,
             sigma=(100.0, 100.0, 0.2), seed=0xF1EE7, disc=0.07, w_obst=1.0e5)
BODY_M = 0.015
FLEET_GOAL_TOLERANCE_M = 0.05
FLEET_CLEARANCE_M = 2 * BODY_M  # what the test asks of every group with peer discs


def _report(out, g, G):
    pos = np.concatenate([o[3] for o in out], axis=0)
    least = pfr.least_pair_distance(pos, G)
    d = pr.distances(out[-1][2], g.shape[0], g)
    return least, d


def test_circle_swap_collides_without_peer_discs_and_not_with_them():
    free, g = pfr.fleet_loop(FLEET, avoid=False)
    least_free, d_free = _report(free, g, FLEET["G"])
    assert (least_free < 2 * BODY_M).any(), f"without peer discs no group collides: {least_free}; the scenario tests nothing"
    out, g = pfr.fleet_loop(FLEET, avoid=True)
    least, d = _report(out, g, FLEET["G"])
    assert (least > FLEET_CLEARANCE_M).all(), f"least pairwise distance per group with peer discs: {least}"
    assert (d < FLEET_GOAL_TOLERANCE_M).all(), f"distances to the goals: {d}"
