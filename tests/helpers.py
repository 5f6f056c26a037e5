"""Shared helpers for the test-suite: golden loading, bank packing, and the env / oracle pairs of the GPU suite.

A test states the configuration it runs at as one dict of knobs (`knobs(...)`) and builds the kernel's env and the
float64 oracle from that same dict (`make_env`, `make_oracle`), so that the two cannot silently disagree."""
import functools
import os
import re
import types

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")

ORACLE_THREADS = max(1, min(16, os.cpu_count() or 1))      # for the oracle runs of the larger GPU cases


def load_trajectories():
    z = np.load(os.path.join(GOLDEN, "trajectories.npz"))
    n = int(z["n_episodes"])
    eps = []
    for i in range(n):
        pre = "e%d_" % i
        eps.append({k[len(pre):]: z[k] for k in z.files if k.startswith(pre)})
    return eps


def pack_bank(hulls_list, goals_list, maxv=None):
    """hulls_list: [(hull0 (m0,2), hull1 (m1,2)), ...]; goals_list: [(5,2), ...] -> float64 bank dict."""
    S = len(hulls_list)
    if maxv is None:
        maxv = max(max(len(h0), len(h1)) for h0, h1 in hulls_list)
    hull_xy = np.zeros((S, 2, maxv, 2))
    hull_n = np.zeros((S, 2), dtype=np.int32)
    goals = np.zeros((S, 5, 2))
    for s, ((h0, h1), g) in enumerate(zip(hulls_list, goals_list)):
        for b, h in enumerate((h0, h1)):
            hull_xy[s, b, :len(h)] = h
            hull_n[s, b] = len(h)
        goals[s] = g
    return dict(hull_xy=hull_xy, hull_n=hull_n, goals=goals)


@functools.lru_cache(maxsize=None)
def fp32_bank(n, W, H, seed=0, map_N=10, wf=0.5):
    """ScenarioBank.generate's bank rounded to fp32: the map is part of the injected state, so the oracle and the kernel
    (which stores hull vertices and goals as fp32) must start from IDENTICAL geometry.  Cached and read-only: a test
    that writes into a shared bank fails instead of changing the map of the tests after it."""
    from ship_sim_gym_b200 import ScenarioBank
    d = ScenarioBank.generate(n, (W, H), seed=seed, map_N=map_N, width_frac=wf).as_dict()
    d["hull_xy"] = d["hull_xy"].astype(np.float32).astype(np.float64)
    d["goals"] = d["goals"].astype(np.float32).astype(np.float64)
    for a in d.values():
        a.setflags(write=False)
    return types.MappingProxyType(d)


# ---------------------------------------------------------------------------------------------- knobs
# Every knob the tests set, at the reference defaults: bounds, speed, history, episode cap, the lidar fan (beams,
# spread, distance), ship scale, mass, thrust, goal radius, step penalty, spawn height, and the map of fp32_bank.
DEFAULTS = dict(W=600.0, H=600.0, speed=10, hist=2, max_steps=1000, n_beams=10, spread=90.0, lidar=100.0, ship_w=2.0,
                ship_h=3.0, mass=5.0, thrust=100.0, goal_radius=5.0, step_penalty=-0.01, spawn_y=25.0, map_N=10, wf=0.5)
# knobs the Python layer does not expose: make_env sets them on shipsim_config itself
RAW_KNOBS = ("ship_w", "ship_h", "mass", "thrust", "goal_radius", "step_penalty", "spawn_y")


def knobs(**overrides):
    """DEFAULTS with `overrides` applied."""
    assert set(overrides) <= set(DEFAULTS), sorted(set(overrides) - set(DEFAULTS))
    return dict(DEFAULTS, **overrides)


def case_knobs(case):
    """knobs() at the knobs a parametrised case dict names; its other keys (name, sizes, flags) are not knobs."""
    return knobs(**{f: v for f, v in case.items() if f in DEFAULTS})


def config_classes(k):
    """(GameConfig, EnvConfig) subclasses at the knobs `k`: bounds, speed, history, episode cap and the lidar fan."""
    from ship_sim_gym_b200.config import EnvConfig, GameConfig, LidarConfig

    class GC(GameConfig):
        BOUNDS = (k["W"], k["H"])
        SPEED = k["speed"]

    class LC(LidarConfig):
        N_BEAMS = k["n_beams"]
        DISTANCE = k["lidar"]
        ANGULAR_SPREAD = k["spread"]

    class EC(EnvConfig):
        HISTORY_SIZE = k["hist"]
        MAX_STEPS = k["max_steps"]
        LIDAR_CONFIG = LC
    return GC, EC


def make_env(k, n, bank, **kw):
    """BatchedShipEnv at the knobs `k` on the bank dict `bank` (None: the env makes its own), other arguments `kw`.
    The config classes carry what the Python layer exposes (with honour_lidar_config=True, which at the reference fan
    gives the same shipsim_config as leaving it off); the RAW_KNOBS are set on the shipsim_config that env.py takes
    from _abi.default_config()."""
    from ship_sim_gym_b200 import BatchedShipEnv, ScenarioBank, _abi
    if bank is not None:
        bank = ScenarioBank(bounds=(k["W"], k["H"]), **bank)
    default_config = _abi.default_config

    def config():
        cfg = default_config()
        for f in RAW_KNOBS:
            setattr(cfg, f, k[f])
        return cfg
    _abi.default_config = config
    try:
        env = BatchedShipEnv(n, *config_classes(k), bank=bank, honour_lidar_config=True, **kw)
    finally:
        _abi.default_config = default_config
    for f in RAW_KNOBS:
        assert getattr(env.cfg, f) == float(np.float32(k[f])), f
    assert (env.cfg.bounds_w, env.cfg.bounds_h, env.cfg.max_steps, env.history) == (k["W"], k["H"], k["max_steps"], k["hist"])
    assert (env.cfg.lidar_spread_deg, env.cfg.lidar_distance) == (k["spread"], k["lidar"])
    assert env.n_beams == k["n_beams"] and env.cfg.lidar_beams == k["n_beams"] and env.n_states == 6 + k["n_beams"]
    return env


def make_oracle(k, n, bank, **kw):
    """The float64 oracle at the knobs `k`, the RAW_KNOBS rounded to fp32 as the kernel holds them; other arguments `kw`."""
    import oracle
    raw = {f: float(np.float32(k[f])) for f in RAW_KNOBS}
    return oracle.OracleEnv(n, bank, W=k["W"], H=k["H"], speed=k["speed"], history=k["hist"], max_steps=k["max_steps"],
                            n_beams=k["n_beams"], lidar_spread_deg=k["spread"], lidar_distance=k["lidar"], **raw, **kw)


# ---------------------------------------------------------------------------------------------- kernel vs kernel
def run(env, acts, K, state=None):
    """Reset `env`, inject `state` if given, roll K steps of `acts` (None: the in-kernel random agent).  Returns
    ((obs, reward, done) numpy, final state, {statistic: its change over the rollout} (shipsim_stat), launch_info)."""
    import torch
    from ship_sim_gym_b200._abi import STAT_NAMES
    env.reset()
    if state is not None:
        env.set_state(*state)
    s0 = env.stats_tensor().clone()
    out = [t.cpu().numpy() for t in env.rollout(acts, K=K)]
    torch.cuda.synchronize()
    return out, env.get_state(), dict(zip(STAT_NAMES, (env.stats_tensor() - s0).tolist())), env.launch_info()


def assert_same(a, b, label):
    """Two run() results are the same rollout: outputs and final state bit for bit, the episode counters exactly and
    the return sum up to the order of its cross-CTA additions."""
    import pytest
    (oa, ra, da), sa, ta, _ = a
    (ob, rb, db), sb, tb, _ = b
    assert np.array_equal(da, db), label + ": done"
    assert np.array_equal(ra, rb), label + ": reward"
    bad = np.argwhere(oa != ob)
    assert bad.size == 0, "%s: obs differ at %d places, first (k, env, col) = %s: %r vs %r" % (
        label, len(bad), bad[:1], oa[tuple(bad[0])] if len(bad) else None, ob[tuple(bad[0])] if len(bad) else None)
    for k in ("pose", "ints", "lidar", "goals", "ep_return"):
        assert np.array_equal(sa[k], sb[k]), "%s: final state %s" % (label, k)
    for k in ("episodes", "length_sum", "goal_steps", "collision", "oob", "timeout", "all_goals"):
        assert ta[k] == tb[k], "%s: stat %s %r vs %r" % (label, k, ta[k], tb[k])
    assert ta["return_sum"] == pytest.approx(tb["return_sum"], rel=1e-5, abs=1e-2)


def source_constant(path, pattern):
    """The number `pattern`'s first group matches in ship_sim_gym_b200/csrc/`path`."""
    with open(os.path.join(ROOT, "ship_sim_gym_b200", "csrc", path)) as f:
        return float(re.search(pattern, f.read()).group(1))
