"""parity.py's oracle-state loader and kernel-vs-oracle comparison for lidar fans of n beams (frames of 6 + n floats).

The same code as parity.load_oracle_state / parity.compare_steps, which serve the reference's 10-beam fan, with the beam
count as an argument; the tolerances, margins and exclusion limits are parity's own."""
import numpy as np

from parity import M_RAY0, POSE_ABS, REL_TOL, STRICT_FRAC


def load_oracle_state(orc, pose, ints, lidar, goals, ret, n_beams=10):
    """parity.load_oracle_state for lidar [n, n_beams]."""
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
    lid_abs[:, :, F - Fr:F - Fr + 2] = POSE_ABS * scale          # x, y: sums of O(scale) fp32 terms (cancellation near 0)
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
