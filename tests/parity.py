"""Kernel-vs-oracle comparison helpers (used by the -m gpu tests, smoke() and bench's self-check).

Tolerances (BASELINE.json north_star / SURVEY.md §8d): pose, velocity, lidar within 1e-4 * max(1, |ref|);
reward / done / flags bit-exact -- away from grazing configurations, which the oracle identifies through the
margins it reports (distance of every evaluated inequality from its decision boundary, in length units).
"""
import numpy as np

REL_TOL = 1e-4
# Grazing filter (SURVEY.md section 8d): a sample is excluded from the exact flag comparison when any decision margin the
# oracle reports is below MARGIN_THR length units; the fraction of samples that graze must stay below MAX_EXCLUDED.
# In a K-step rollout an env that grazed at step k is not compared at steps > k either (the two trajectories may have
# legitimately diverged), so the CUMULATIVE excluded fraction grows with K: `grazing_frac` (env-steps that were
# themselves below the margin, per compared-or-grazing env-step) is held to MAX_EXCLUDED, the cumulative
# `excluded_frac` to MAX_EXCLUDED_CUMULATIVE (oracle-side measurement at K = 32: 0.02-1.1 % cumulative, < 0.1 % per step).
MARGIN_THR = 1e-3
MAX_EXCLUDED = 0.01
MAX_EXCLUDED_CUMULATIVE = 0.05
# Lidar readings are DIFFERENCES of world coordinates divided by cos(incidence): a pose that is within tolerance
# (fp32 world coordinates carry ulp(600) = 6e-5 per rounding, a few ulps after 32 steps) moves a reading by
# (pose error) x cond, cond = 1/|n.dir| of the hit edge, which the oracle reports.  All readings must satisfy
#   |err| <= (REL_TOL * max(1, |ref|) + POSE_ABS * max(W, H)) * cond
# and at least STRICT_FRAC of them the plain REL_TOL * max(1, |ref|) bound.
POSE_ABS = 1e-6
STRICT_FRAC = 0.99
# margin layout of the oracle: [0] ship-bank SAT |separation|, [1] |goal distance - r|, [2] out-of-bounds slack,
# [3] nearest-goal tie slack, [4+i] lidar ray i
M_SAT, M_GOAL, M_OOB, M_TIE, M_RAY0 = 0, 1, 2, 3, 4


SHIP_TEMPLATE = np.array([[0.0, 0.0], [0.0, 10.0], [5.0, 15.0], [10.0, 10.0], [10.0, 0.0]])   # models.py:6


def ship_hull(ship_w=2.0, ship_h=3.0):
    """The ship's hull in the body frame: SHIP_TEMPLATE scaled by (ship_w, ship_h) (game.py:275)."""
    return SHIP_TEMPLATE * np.array([ship_w, ship_h])


SHIP_HULL = ship_hull()     # the default ship


def _hull_rmax(hull):
    return float(np.sqrt((hull ** 2).sum(1)).max())


def random_states(rng, n, W, H, n_scen, bank_goals, max_steps=1000, near=None, hull=SHIP_HULL):
    """Injected-state distribution of SURVEY.md §8(d).  With `near`, every other ship is put within a box around a bank
    vertex whose half width (60 for the default hull) grows with the size of `hull` (the body-frame hull)."""
    spread = 60.0 * _hull_rmax(hull) / _hull_rmax(SHIP_HULL)
    pose = np.zeros((n, 6))
    pose[:, 0] = rng.uniform(0, W, n)
    pose[:, 1] = rng.uniform(0, H, n)
    pose[:, 2] = rng.uniform(-np.pi, np.pi, n)
    pose[:, 3:5] = rng.uniform(-40, 40, (n, 2))
    pose[:, 5] = rng.uniform(-0.3, 0.3, n)
    ints = np.zeros((n, 5), dtype=np.int32)
    ints[:, 0] = rng.choice([-10, -5, 0, 5, 10], n)
    ints[:, 1] = rng.randint(0, 32, n)
    ints[:, 2] = rng.randint(0, max_steps, n)
    ints[:, 3] = rng.randint(0, n_scen, n)
    ints[:, 4] = rng.randint(0, 50, n)
    lidar = np.where(rng.rand(n, 10) < 0.5, -1.0, rng.uniform(0, 100, (n, 10)))
    goals = bank_goals[ints[:, 3]].copy()
    ret = rng.uniform(-3, 3, n)
    if near is not None:        # adversarial: put the ship close to a vertex of one of its banks
        hull_xy, hull_n = near
        for e in range(0, n, 2):
            s = ints[e, 3]
            b = rng.randint(0, 2)
            v = hull_xy[s, b, rng.randint(0, hull_n[s, b])]
            pose[e, 0:2] = v + rng.uniform(-spread, spread, 2)
    return pose, ints, lidar, goals, ret


def lidar_origin_offset(theta, hull=SHIP_HULL):
    """(hx, hy): half extents of the rotated hull's AABB -- LiDAR.query's origin relative to the body (models.py:51-53)."""
    c, s = np.cos(theta), np.sin(theta)
    wx = hull[:, 0][None] * c[:, None] - hull[:, 1][None] * s[:, None]
    wy = hull[:, 0][None] * s[:, None] + hull[:, 1][None] * c[:, None]
    return 0.5 * (wx.max(1) - wx.min(1)), 0.5 * (wy.max(1) - wy.min(1))


def goal_shell_states(rng, n, W, H, n_scen, deltas=(-1e-2, -5e-3, -2e-3, 2e-3, 5e-3, 1e-2), hull=SHIP_HULL, radius=5.0):
    """Adversarial set "goal at distance r +- eps" (SURVEY.md section 8d): the ship at rest (so the step leaves the pose
    where it is), goal k of every env placed at distance `radius` + delta from `hull` -- off an edge or off a vertex."""
    pose = np.zeros((n, 6))
    pose[:, 0] = rng.uniform(100, W - 100, n)
    pose[:, 1] = rng.uniform(100, H - 100, n)
    pose[:, 2] = rng.uniform(-np.pi, np.pi, n)
    ints = np.zeros((n, 5), dtype=np.int32)
    ints[:, 0] = rng.choice([-10, -5, 0, 5, 10], n)
    ints[:, 1] = 31
    ints[:, 2] = rng.randint(0, 500, n)
    ints[:, 3] = rng.randint(0, n_scen, n)
    lidar = np.full((n, 10), -1.0)
    goals = np.zeros((n, 5, 2))
    goals[:, :, 0] = W * 5.0 + 100.0 * np.arange(5)[None]     # far away (and at distinct distances: no nearest-goal ties), except goal k
    goals[:, :, 1] = H * 5.0
    delta = np.asarray(deltas)[rng.randint(0, len(deltas), n)]
    c, s = np.cos(pose[:, 2]), np.sin(pose[:, 2])
    for e in range(n):
        j = rng.randint(0, 5)
        a, b = hull[j - 1], hull[j]
        if rng.rand() < 0.5:                           # off the edge a -> b (outward normal of a CCW... the template is CW here)
            t = rng.uniform(0.05, 0.95)
            q = a + t * (b - a)
            ed = (b - a) / np.linalg.norm(b - a)
            nrm = np.array([-ed[1], ed[0]])
            cen = hull.mean(0)
            if np.dot(nrm, q - cen) < 0:
                nrm = -nrm
        else:                                          # off the vertex b, along the bisector of its outward normals
            q = b
            nrm = (b - hull.mean(0))
            nrm = nrm / np.linalg.norm(nrm)
            # keep the direction inside the vertex' normal cone: the bisector of the two edge normals
            e0 = (b - a) / np.linalg.norm(b - a)
            nxt = hull[(j + 1) % 5]
            e1 = (nxt - b) / np.linalg.norm(nxt - b)
            n0, n1 = np.array([-e0[1], e0[0]]), np.array([-e1[1], e1[0]])
            cen = hull.mean(0)
            if np.dot(n0, b - cen) < 0:
                n0, n1 = -n0, -n1
            nrm = (n0 + n1) / np.linalg.norm(n0 + n1)
        loc = q + nrm * (radius + delta[e])
        k = rng.randint(0, 5)
        goals[e, k, 0] = pose[e, 0] + loc[0] * c[e] - loc[1] * s[e]
        goals[e, k, 1] = pose[e, 1] + loc[0] * s[e] + loc[1] * c[e]
    return pose, ints, lidar, goals.reshape(n, 10), np.zeros(n), delta


def origin_inside_bank_states(rng, n, hull_xy, hull_n, n_scen, hull=SHIP_HULL):
    """Adversarial set "ray origin inside a bank" (App. B Q11): the lidar origin (body origin + half the rotated hull's
    AABB) sits strictly inside one of the env's banks, so every ray reports the full length for that bank."""
    pose = np.zeros((n, 6))
    pose[:, 2] = rng.uniform(-np.pi, np.pi, n)
    ints = np.zeros((n, 5), dtype=np.int32)
    ints[:, 1] = 31
    ints[:, 3] = rng.randint(0, n_scen, n)
    hx, hy = lidar_origin_offset(pose[:, 2], hull)
    which = np.zeros(n, dtype=np.int64)
    for e in range(n):
        s = ints[e, 3]
        b = rng.randint(0, 2)
        which[e] = b
        v = hull_xy[s, b, :hull_n[s, b]]
        w = rng.dirichlet(np.ones(len(v)) * 0.7)
        pt = (w[:, None] * v).sum(0)
        pt = pt + 0.2 * (v.mean(0) - pt)               # pull towards the centroid: strictly inside
        pose[e, 0], pose[e, 1] = pt[0] - hx[e], pt[1] - hy[e]
    lidar = np.where(rng.rand(n, 10) < 0.5, -1.0, rng.uniform(0, 100, (n, 10)))
    return pose, ints, lidar, which


# Reach grid of derive_params (shipsim_abi.cu): GRID_N x GRID_N cells over [-GRID_PAD, W + GRID_PAD] x [-GRID_PAD, H + GRID_PAD],
# looked up at the lidar origin as floor((o + GRID_PAD) * inv_cell) in fp32 and clamped, so the border cells are unbounded.
GRID_N = 32
GRID_PAD = 32.0


def grid_boundaries(W, H):
    """Cell boundaries of the reach grid along x and y, float64: -GRID_PAD + i * cell for i = 0 .. GRID_N."""
    i = np.arange(GRID_N + 1)
    return -GRID_PAD + i * ((W + 2 * GRID_PAD) / GRID_N), -GRID_PAD + i * ((H + 2 * GRID_PAD) / GRID_N)


def grid_cell(o, extent):
    """The kernel's cell index of lidar-origin coordinates `o` along an axis of length `extent`, in fp32 arithmetic."""
    inv = np.float32(GRID_N / (extent + 2.0 * GRID_PAD))
    t = (np.asarray(o, dtype=np.float32) + np.float32(GRID_PAD)) * inv
    return np.clip(np.floor(t).astype(np.int64), 0, GRID_N - 1)


def lidar_origin(pose, hull=SHIP_HULL):
    hx, hy = lidar_origin_offset(pose[:, 2], hull)
    return pose[:, 0] + hx, pose[:, 1] + hy


GRID_ULPS = (-2, -1, 0, 1, 2)


def grid_boundary_states(rng, n, W, H, n_scen, bank_goals, hull=SHIP_HULL, max_steps=1000):
    """Adversarial set "lidar origin on a reach-grid cell boundary": the origin (body + half the rotated hull's AABB) lies
    on a boundary, or 1 or 2 fp32 ulps to either side of it, along x, y or both; every boundary is used, the outer ones
    (the edges of the unbounded border cells) included, and one env in eight has its origin beyond the pad.  Half the
    ships point straight up, where the offset to the origin is exact in fp32.  Returns random_states' tuple and
    `target` [n, 2]: the intended ulp offset per axis (a value outside GRID_ULPS = that axis is free)."""
    pose, ints, lidar, goals, ret = random_states(rng, n, W, H, n_scen, bank_goals, max_steps=max_steps, hull=hull)
    pose[:, 2] = np.where(rng.rand(n) < 0.5, 0.0, pose[:, 2].astype(np.float32).astype(np.float64))
    off = lidar_origin_offset(pose[:, 2], hull)
    bnd = grid_boundaries(W, H)
    ext = (W, H)
    target = np.full((n, 2), 99, dtype=np.int64)
    mode = rng.randint(0, 8, n)                        # 0-2: x, 3-5: y, 6: both, 7: beyond the pad
    for e in range(n):
        axes = (0,) if mode[e] < 3 else ((1,) if mode[e] < 6 else ((0, 1) if mode[e] == 6 else ()))
        for a in axes:
            k = GRID_ULPS[rng.randint(0, len(GRID_ULPS))]
            t = np.float32(bnd[a][rng.randint(0, GRID_N + 1)])
            for _ in range(abs(k)):
                t = np.nextafter(t, np.float32(np.inf if k > 0 else -np.inf))
            pose[e, a] = float(t) - off[a][e]
            target[e, a] = k
        if mode[e] == 7:
            a = rng.randint(0, 2)
            o = -GRID_PAD - rng.uniform(0.5, 40.0) if rng.rand() < 0.5 else ext[a] + GRID_PAD + rng.uniform(0.5, 40.0)
            pose[e, a] = o - off[a][e]
    return (pose, ints, lidar, goals, ret), target


def f32_inputs(pose, ints, lidar, goals, ret):
    """Round the injected state to fp32 so that oracle and kernel start from IDENTICAL values."""
    return (pose.astype(np.float32).astype(np.float64), ints, lidar.astype(np.float32).astype(np.float64),
            goals.astype(np.float32).astype(np.float64), ret.astype(np.float32).astype(np.float64))


def concat_states(parts):
    """Injected states (pose, ints, lidar, goals, ret) of several generators -> one state of all their envs, in order."""
    st = [np.concatenate([np.asarray(p[j]).reshape(len(p[0]), -1) for p in parts]) for j in range(5)]
    st[4] = st[4].reshape(-1)
    return tuple(st)


def load_oracle_state(orc, pose, ints, lidar, goals, ret, n_beams=10):
    """Inject a state into the oracle, as env.set_state does into the kernel; lidar [n, n_beams]."""
    n = orc.n
    orc.pose[:] = pose
    orc.ints[:] = ints
    orc.lidar[:] = -1.0
    orc.lidar[:, :n_beams] = lidar
    orc.goals[:] = goals.reshape(n, 5, 2)
    orc.ep_return[:] = ret
    # history deque: older frames are unknowable for an injected state; newest frame = current pre-step frame
    F = orc.frame
    orc.hist[:] = -1.0
    fr = np.zeros((n, F))
    fr[:, 0:2] = pose[:, 0:2]
    fr[:, 2] = ints[:, 0]
    fr[:, 3] = pose[:, 2]
    g = goals.reshape(n, 5, 2)
    d = np.sqrt(((g - pose[:, None, 0:2]) ** 2).sum(-1))
    alive = (ints[:, 1:2] >> np.arange(5)[None]) & 1
    d = np.where(alive == 1, d, np.inf)
    k = d.argmin(1)
    has = alive.any(1)
    fr[:, 4] = np.where(has, g[np.arange(n), k, 0], -1.0)
    fr[:, 5] = np.where(has, g[np.arange(n), k, 1], -1.0)
    fr[:, 6:6 + n_beams] = lidar
    orc.hist[:, -F:] = fr


def compare_steps(ref, got_obs, got_rew, got_done, margin_thr=1e-3, rel_tol=REL_TOL, label="", scale=600.0,
                  stop_at_done=False, n_beams=10):
    """ref: oracle dict of [K,N,...]; got_*: numpy [K,N,...] from the kernel.  An env is compared up to (not
    including) the first step at which any margin drops below `margin_thr` (after a grazing decision the two
    trajectories may legitimately diverge).  Returns a report dict; raises AssertionError on mismatch.  Frames of
    6 + n_beams floats; rows of one or two frames."""
    K, N = ref["reward"].shape
    mg = ref["margins"]
    F = got_obs.shape[-1]
    nb = n_beams
    Fr = 6 + nb                 # floats per frame
    graze = (mg[:, :, :4].min(-1) < margin_thr) | (mg[:, :, M_RAY0:M_RAY0 + nb].min(-1) < margin_thr)
    # valid[k, e]: no grazing at any step <= k
    valid = np.cumsum(graze, axis=0) == 0
    if stop_at_done:
        # without auto-reset the reference episode is over at `done`: what a caller that keeps stepping sees is out
        # of scope (SURVEY.md §8 f4), and an env that flies thousands of units off the map leaves fp32's range of
        # useful precision.  Compare up to and including the terminal step.
        d = ref["done"].astype(np.int64)
        valid &= (np.cumsum(d, axis=0) - d) == 0
    n_cmp = int(valid.sum())
    before = np.concatenate([np.ones_like(valid[:1]), valid[:-1]], axis=0)
    n_graze = int((graze & before).sum())       # env-steps that were themselves grazing (first exclusion of their env)
    # what could have been compared at all: with stop_at_done, steps after an env's terminal step are not the path's
    # business, so they do not count as "excluded" either
    eligible = K * N
    if stop_at_done:
        d_ = ref["done"].astype(np.int64)
        eligible = int(((np.cumsum(d_, axis=0) - d_) == 0).sum())
    tol = rel_tol * np.maximum(1.0, np.abs(ref["obs"]))
    err = np.abs(got_obs.astype(np.float64) - ref["obs"])
    strict_bad = (err > tol) & valid[:, :, None]
    # lidar slots: conditioning-aware bound.  The newest frame holds this step's readings (cond of step k); the
    # older frame holds the previous step's (cond of step k-1; unknown for k = 0 of an injected state -> that
    # frame is the injected value itself, exact).
    cond = np.maximum(1.0, mg[:, :, 4 + 32:4 + 32 + nb])
    cond_run = np.maximum.accumulate(cond, axis=0)          # sticky readings keep the cond of the step that wrote them
    lid_tol_scale = np.ones_like(tol)
    lid_abs = np.zeros_like(tol)
    new0 = F - Fr + 6
    lid_tol_scale[:, :, new0:new0 + nb] = cond_run
    lid_abs[:, :, new0:new0 + nb] = POSE_ABS * scale
    lid_abs[:, :, F - Fr:F - Fr + 2] = POSE_ABS * scale      # x, y: sums of O(scale) fp32 terms (cancellation near 0)
    if F == 2 * Fr:
        lid_abs[:, :, 0:2] = POSE_ABS * scale
        prev = np.concatenate([np.ones_like(cond_run[:1]), cond_run[:-1]], axis=0)
        lid_tol_scale[:, :, 6:6 + nb] = prev
        lid_abs[:, :, 6:6 + nb] = POSE_ABS * scale
    tol = (tol + lid_abs) * lid_tol_scale
    bad_obs = (err > tol) & valid[:, :, None]
    if bad_obs.any():
        k, e, j = np.argwhere(bad_obs)[0]
        raise AssertionError("%s obs mismatch at step %d env %d slot %d: got %r ref %r (margins %r)"
                             % (label, k, e, j, got_obs[k, e, j], ref["obs"][k, e, j], mg[k, e, :14]))
    bad_r = (np.abs(got_rew.astype(np.float64) - ref["reward"]) > 1e-6) & valid
    if bad_r.any():
        k, e = np.argwhere(bad_r)[0]
        raise AssertionError("%s reward mismatch at step %d env %d: got %r ref %r" % (label, k, e, got_rew[k, e], ref["reward"][k, e]))
    bad_d = (got_done.astype(bool) != ref["done"].astype(bool)) & valid
    if bad_d.any():
        k, e = np.argwhere(bad_d)[0]
        raise AssertionError("%s done mismatch at step %d env %d: got %r ref %r flags %r margins %r"
                             % (label, k, e, got_done[k, e], ref["done"][k, e], ref["flags"][k, e], mg[k, e, :4]))
    n_entries = int(valid.sum()) * F
    strict_frac = 1.0 - float(strict_bad.sum()) / max(1, n_entries)
    if strict_frac < STRICT_FRAC:
        raise AssertionError("%s only %.4f of the compared obs entries are within the plain %g bound" % (label, strict_frac, rel_tol))
    return dict(compared=n_cmp, total=K * N, eligible=eligible, excluded_frac=1.0 - n_cmp / float(max(1, eligible)),
                grazing_frac=n_graze / float(max(1, n_cmp + n_graze)), strict_frac=strict_frac,
                max_rel_err=float((err / np.maximum(1.0, np.abs(ref["obs"])) / lid_tol_scale)[valid].max()) if n_cmp else 0.0,
                max_pose_rel_err=float((np.maximum(0.0, err - lid_abs) / np.maximum(1.0, np.abs(ref["obs"])))[:, :, F - Fr:F - Fr + 4][valid].max()) if n_cmp else 0.0,
                frame=F)
