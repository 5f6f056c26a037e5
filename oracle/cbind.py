"""ctypes binding of oracle/shipsim_oracle.c.  TEST INFRASTRUCTURE ONLY (see package docstring)."""
import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
SO = os.path.join(HERE, "libshipsim_oracle.so")
SRC = os.path.join(HERE, "shipsim_oracle.c")

FLAG_COLLIDING, FLAG_GOAL, FLAG_OOB, FLAG_TIMEOUT, FLAG_ALLGOALS = 1, 2, 4, 8, 16
STAT_NAMES = ("episodes", "return_sum", "length_sum", "goal_steps", "collision", "oob", "timeout", "all_goals", "steps")
N_GOALS = 5


def build(force=False):
    """gcc the C restatement (seconds).  Idempotent."""
    if force or not os.path.exists(SO) or os.path.getmtime(SO) < os.path.getmtime(SRC):
        subprocess.check_call(["make", "-C", HERE, "-B", "libshipsim_oracle.so"], stdout=subprocess.DEVNULL)
    return SO


class _Config(C.Structure):
    _fields_ = [(n, C.c_double) for n in ("W", "H", "dt", "space_damping", "lidar_spread_deg", "lidar_distance",
                                          "ship_w", "ship_h", "mass", "thrust", "goal_radius", "step_penalty",
                                          "spawn_y")] + \
               [("seed", C.c_uint64), ("env_id_offset", C.c_int64)] + \
               [(n, C.c_int32) for n in ("max_steps", "history", "n_beams", "auto_reset", "n_scenarios", "maxv", "pick_base", "pick_count")]


class _Bank(C.Structure):
    _fields_ = [("hull_xy", C.c_void_p), ("hull_n", C.c_void_p), ("goals", C.c_void_p)]


class _State(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("pose", "lidar", "goals", "ep_return", "hist", "ints")]


_lib = None


def lib():
    global _lib
    if _lib is None:
        build()
        L = C.CDLL(SO)
        L.orc_moment_for_poly.restype = C.c_double
        L.orc_moment_for_poly.argtypes = [C.c_double, C.c_int, C.c_void_p]
        L.orc_convex_hull.restype = C.c_int
        L.orc_convex_hull.argtypes = [C.c_int, C.c_void_p, C.c_void_p]
        L.orc_poly_point_distance.restype = C.c_double
        L.orc_poly_point_distance.argtypes = [C.c_int, C.c_void_p, C.c_double, C.c_double]
        L.orc_segment_query.restype = None
        L.orc_segment_query.argtypes = [C.c_int, C.c_void_p] + [C.c_double] * 5 + [C.c_void_p]
        L.orc_polys_touch.restype = C.c_int
        L.orc_polys_touch.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p]
        L.orc_goal_span.restype = C.c_int
        L.orc_goal_span.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_double, C.c_double, C.c_void_p]
        L.orc_pick_scenario.restype = C.c_int32
        L.orc_pick_scenario.argtypes = [C.c_uint64, C.c_int64, C.c_int32, C.c_int32]
        L.orc_random_action.restype = C.c_int32
        L.orc_random_action.argtypes = [C.c_uint64, C.c_int64, C.c_uint32]
        L.orc_philox4x32.restype = None
        L.orc_philox4x32.argtypes = [C.c_uint64, C.c_uint64, C.c_uint32, C.c_uint32, C.c_void_p]
        L.orc_ship_moment.restype = C.c_double
        L.orc_ship_moment.argtypes = [C.POINTER(_Config)]
        L.orc_damping.restype = C.c_double
        L.orc_damping.argtypes = [C.POINTER(_Config)]
        L.orc_ship_hull.restype = None
        L.orc_ship_hull.argtypes = [C.POINTER(_Config), C.c_void_p]
        L.orc_reset.restype = None
        L.orc_reset.argtypes = [C.POINTER(_Config), C.POINTER(_Bank), C.POINTER(_State), C.c_int, C.c_void_p,
                                C.c_void_p, C.c_int, C.c_void_p]
        L.orc_step.restype = None
        L.orc_step.argtypes = [C.POINTER(_Config), C.POINTER(_Bank), C.POINTER(_State), C.c_int, C.c_int,
                               C.c_void_p, C.c_uint32] + [C.c_void_p] * 6 + [C.c_int]
        _lib = L
    return _lib


def _p(a):
    return None if a is None else a.ctypes.data


# ---- thin geometry helpers (numpy in / python out) ------------------------------------------------
def convex_hull(xy):
    xy = np.ascontiguousarray(xy, dtype=np.float64)
    out = np.zeros((len(xy) + 2, 2))
    m = lib().orc_convex_hull(len(xy), _p(xy), _p(out))
    return out[:m].copy()


def moment_for_poly(mass, xy):
    xy = np.ascontiguousarray(xy, dtype=np.float64)
    return lib().orc_moment_for_poly(mass, len(xy), _p(xy))


def poly_point_distance(hull, p):
    hull = np.ascontiguousarray(hull, dtype=np.float64)
    return lib().orc_poly_point_distance(len(hull), _p(hull), float(p[0]), float(p[1]))


def segment_query(hull, a, b, r=0.0):
    """-> (hit, point(2), alpha, margin)"""
    hull = np.ascontiguousarray(hull, dtype=np.float64)
    out = np.zeros(5)
    lib().orc_segment_query(len(hull), _p(hull), float(a[0]), float(a[1]), float(b[0]), float(b[1]), float(r), _p(out))
    return bool(out[0]), out[1:3].copy(), out[3], out[4]


def polys_touch(h1, h2):
    h1 = np.ascontiguousarray(h1, dtype=np.float64)
    h2 = np.ascontiguousarray(h2, dtype=np.float64)
    sep = np.zeros(1)
    t = lib().orc_polys_touch(len(h1), _p(h1), len(h2), _p(h2), _p(sep))
    return bool(t), float(sep[0])


def goal_span(hull_xy, hull_n, W, y):
    """hull_xy [2,maxv,2], hull_n [2] -> (ok, lo, hi) of game.py:322-325"""
    hull_xy = np.ascontiguousarray(hull_xy, dtype=np.float64)
    hull_n = np.ascontiguousarray(hull_n, dtype=np.int32)
    out = np.zeros(2)
    ok = lib().orc_goal_span(_p(hull_xy), _p(hull_n), hull_xy.shape[1], float(W), float(y), _p(out))
    return bool(ok), out[0], out[1]


def pick_scenario(seed, gid, episode, n):
    return lib().orc_pick_scenario(seed, gid, episode, n)


def random_action(seed, gid, step):
    return lib().orc_random_action(seed, gid, step)


def philox(seed, ctr_lo, c2, c3):
    out = np.zeros(4, dtype=np.uint32)
    lib().orc_philox4x32(seed, ctr_lo, c2, c3, _p(out))
    return out


class OracleEnv(object):
    """N independent float64 ShipEnvs stepped by the C restatement.

    bank: dict(hull_xy=[S,2,maxv,2] f64, hull_n=[S,2] i32, goals=[S,5,2] f64)
    """

    def __init__(self, n_envs, bank, W=600.0, H=600.0, speed=10.0, history=2, max_steps=1000, n_beams=10,
                 lidar_spread_deg=90.0, lidar_distance=100.0, seed=0, env_id_offset=0, auto_reset=False,
                 n_threads=1, pick_base=0, pick_count=0, ship_w=2.0, ship_h=3.0, mass=5.0, thrust=100.0,
                 goal_radius=5.0, step_penalty=-0.01, spawn_y=25.0):
        self.L = lib()
        self.n = int(n_envs)
        self.n_threads = n_threads
        self.hull_xy = np.ascontiguousarray(bank["hull_xy"], dtype=np.float64)
        self.hull_n = np.ascontiguousarray(bank["hull_n"], dtype=np.int32)
        self.bank_goals = np.ascontiguousarray(bank["goals"], dtype=np.float64)
        S, _, maxv, _ = self.hull_xy.shape
        self.cfg = _Config(W=W, H=H, dt=0.1 * speed, space_damping=0.4, lidar_spread_deg=lidar_spread_deg,
                           lidar_distance=lidar_distance, ship_w=ship_w, ship_h=ship_h, mass=mass, thrust=thrust,
                           goal_radius=goal_radius, step_penalty=step_penalty, spawn_y=spawn_y, seed=seed, env_id_offset=env_id_offset,
                           max_steps=max_steps, history=history, n_beams=n_beams, auto_reset=int(auto_reset),
                           n_scenarios=S, maxv=maxv, pick_base=int(pick_base), pick_count=int(pick_count))
        self.frame = 6 + n_beams
        self.obs_dim = self.frame * history
        self.maxbeams = self.L.orc_max_beams()
        self.mstride = self.L.orc_margin_stride()
        self.cond_offset = 4 + self.maxbeams
        self.pose = np.zeros((self.n, 6))
        self.lidar = np.full((self.n, self.maxbeams), -1.0)
        self.goals = np.zeros((self.n, 5, 2))
        self.ep_return = np.zeros(self.n)
        self.hist = np.full((self.n, self.obs_dim), -1.0)
        self.ints = np.zeros((self.n, 5), dtype=np.int32)      # rudder, alive, step_count, scenario, episode
        self.stats = np.zeros(self.L.orc_stats_len())
        self._bank = _Bank(_p(self.hull_xy), _p(self.hull_n), _p(self.bank_goals))
        self._state = _State(_p(self.pose), _p(self.lidar), _p(self.goals), _p(self.ep_return), _p(self.hist), _p(self.ints))
        self.step_counter = 0

    @property
    def moment(self):
        return self.L.orc_ship_moment(C.byref(self.cfg))

    @property
    def damping(self):
        return self.L.orc_damping(C.byref(self.cfg))

    def ship_hull(self):
        out = np.zeros((5, 2))
        self.L.orc_ship_hull(C.byref(self.cfg), _p(out))
        return out

    def reset(self, mask=None, scen=None, first=True):
        obs = np.zeros((self.n, self.obs_dim))
        m = None if mask is None else np.ascontiguousarray(mask, dtype=np.uint8)
        sc = None if scen is None else np.ascontiguousarray(scen, dtype=np.int32)
        self.L.orc_reset(C.byref(self.cfg), C.byref(self._bank), C.byref(self._state), self.n, _p(m), _p(sc),
                         int(first), _p(obs))
        if mask is not None:
            obs = np.where(np.asarray(mask, dtype=bool)[:, None], obs, self.hist)
        return obs

    def step(self, actions=None, K=None, want=("obs", "reward", "done", "flags", "margins")):
        """actions [N] or [K,N] int (None -> philox random actions, K required).  Returns a dict of
        [K,N,...] arrays (leading K squeezed when actions was 1-D)."""
        squeeze = False
        if actions is not None:
            a = np.ascontiguousarray(actions, dtype=np.int32)
            if a.ndim == 1:
                a = a[None]
                squeeze = True
            K = a.shape[0]
            assert a.shape[1] == self.n
        else:
            a = None
        out = {}
        if "obs" in want:
            out["obs"] = np.zeros((K, self.n, self.obs_dim))
        if "reward" in want:
            out["reward"] = np.zeros((K, self.n))
        if "done" in want:
            out["done"] = np.zeros((K, self.n), dtype=np.uint8)
        if "flags" in want:
            out["flags"] = np.zeros((K, self.n), dtype=np.uint8)
        if "margins" in want:
            out["margins"] = np.zeros((K, self.n, self.mstride))
        self.L.orc_step(C.byref(self.cfg), C.byref(self._bank), C.byref(self._state), self.n, K, _p(a),
                        self.step_counter, _p(out.get("obs")), _p(out.get("reward")), _p(out.get("done")),
                        _p(out.get("flags")), _p(out.get("margins")), _p(self.stats), self.n_threads)
        self.step_counter += K
        if squeeze:
            out = {k: v[0] for k, v in out.items()}
        return out

    def stats_dict(self):
        return dict(zip(STAT_NAMES, self.stats.tolist()))
