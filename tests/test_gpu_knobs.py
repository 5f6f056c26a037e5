"""-m gpu: both step kernels against the float64 oracle at non-default values of every knob of shipsim_config -- bounds
(square and not), speed, episode cap, lidar spread and distance, ship scale, mass, thrust, goal radius, step penalty
and spawn height -- and at the geometry of the spawn row and 64-bit RNG keys.

derive_params (shipsim_abi.cu) turns the knobs into the hull, its moment, the accelerations, the culls, the fan and the
reach grid; the grid builder, the spawn-row builder and the host path's reward table read them too.  The other GPU
tests run at the reference defaults only, where a knob read from the wrong field, or a constant that silently assumes
the default, cannot show.  Every case here also checks that it is sensitive to its knob: the oracle run again with
the knobs set back to the defaults must disagree with the kernel on a stated share of the compared env-steps."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import oracle  # noqa: E402
from helpers import ORACLE_THREADS, assert_same, case_knobs, fp32_bank, knobs, make_env, make_oracle  # noqa: E402
from helpers import pack_bank, run, source_constant  # noqa: E402
import parity  # noqa: E402

# guard: (which run, share) -- the share of compared env-steps ("step": envs of the single injected step, post-step
# velocities included; "roll": env-steps of the 32-step auto-reset rollout) on which the kernel must DISAGREE with the
# oracle run at the default knobs ("uneventful": every step without an event).  The shares are about half of what
# the oracle at the case's knobs measures against the one at the defaults.
CASES = [
    dict(name="wide", W=900.0, H=400.0, guard=("step", 0.15)),
    dict(name="tall", W=400.0, H=1000.0, guard=("step", 0.15)),
    dict(name="large", W=4000.0, H=4000.0, speed=40, guard=("step", 0.3)),
    dict(name="lidar_short", lidar=20.0, guard=("step", 0.25)),
    dict(name="lidar_long", lidar=350.0, guard=("step", 0.35)),
    dict(name="spread_30", spread=30.0, guard=("step", 0.12)),
    dict(name="spread_270", spread=270.0, guard=("step", 0.2)),
    dict(name="spread_360", spread=360.0, guard=("step", 0.2)),
    dict(name="spread_450", spread=450.0, guard=("step", 0.2)),
    dict(name="spread_neg", spread=-120.0, guard=("step", 0.15)),
    dict(name="big_ship", ship_w=4.0, ship_h=5.0, shell=True, guard=("step", 0.25)),
    dict(name="big_ship_short_lidar", ship_w=4.0, ship_h=5.0, lidar=20.0, shell=True, guard=("step", 0.3)),
    # mass x 16 keeps the moment, and so the spin, of the default ship: at mass 5 this hull turns by up to 5 rad per
    # step, and within a few dozen steps the fp32 heading the kernels keep no longer resolves the pose to the tolerance
    dict(name="small_ship", ship_w=0.5, ship_h=0.5, mass=80.0, shell=True, guard=("step", 0.25)),
    dict(name="fast", mass=1.5, thrust=400.0, speed=30, guard=("step", 0.5)),
    dict(name="sluggish", mass=50.0, thrust=20.0, guard=("step", 0.15)),
    dict(name="goal_r_small", goal_radius=0.5, shell=True, guard=("step", 0.06)),
    dict(name="goal_r_big", goal_radius=40.0, shell=True, guard=("step", 0.08)),
    dict(name="penalty", step_penalty=-0.37, guard=("uneventful", 1.0)),
    dict(name="penalty_zero", step_penalty=0.0, guard=("uneventful", 1.0)),
    dict(name="spawn_mid", W=1000.0, H=1000.0, spawn_y=300.0, map_N=30, wf=0.9, guard=("roll", 0.5)),
    dict(name="cap1", max_steps=1, guard=("step", 0.2)),
    dict(name="cap2", max_steps=2, guard=("step", 0.1)),
]
IDS = [c["name"] for c in CASES]


def default_knobs_of(k):
    """The knobs set back to the defaults, on the case's map."""
    return knobs(map_N=k["map_N"], wf=k["wf"])


# ---------------------------------------------------------------------------------------------- inputs
N_STEP, N_ROLL, K_ROLL = 8192 - 5, 4096 + 3, 32


def injected_states(case, k, bank, n, seed):
    """A quarter each: random states, ships near a bank vertex, lidar origins on reach-grid cell boundaries, and either
    goals at the goal radius +- eps from the hull (goal-radius and ship cases) or more ships near a bank."""
    rng = np.random.RandomState(seed)
    hull = parity.ship_hull(k["ship_w"], k["ship_h"])
    W, H = k["W"], k["H"]
    q = n // 4
    near = (bank["hull_xy"], bank["hull_n"])
    parts = [parity.random_states(rng, q, W, H, 64, bank["goals"], max_steps=k["max_steps"], hull=hull),
             parity.random_states(rng, q, W, H, 64, bank["goals"], max_steps=k["max_steps"], near=near, hull=hull),
             parity.grid_boundary_states(rng, q, W, H, 64, bank["goals"], hull=hull, max_steps=k["max_steps"])[0]]
    m = n - 3 * q
    if case.get("shell"):
        p, i, li, g, r, _ = parity.goal_shell_states(rng, m, W, H, 64, hull=hull, radius=k["goal_radius"])
        i[:, 2] = np.minimum(i[:, 2], k["max_steps"] - 1)
        parts.append((p, i, li, g, r))
    else:
        parts.append(parity.random_states(rng, m, W, H, 64, bank["goals"], max_steps=k["max_steps"], near=near, hull=hull))
    return parity.f32_inputs(*parity.concat_states(parts)), rng.randint(0, 3, n).astype(np.int32)


def _disagree(ref, obs, rew, done):
    """[K, N] bool: env-steps where (obs, rew, done) differ from the oracle's `ref` by more than any tolerance in use."""
    tol = 1e-3 * np.maximum(1.0, np.abs(ref["obs"]))
    return ((np.abs(obs.astype(np.float64) - ref["obs"]) > tol).any(-1) | (np.abs(rew.astype(np.float64) - ref["reward"]) > 1e-6)
            | (done.astype(bool) != ref["done"].astype(bool)))


@pytest.fixture(scope="module")
def oracle_runs():
    """The oracle's results, computed once per case and shared by every kernel variant compared with them."""
    cache = {}

    def get(kind, case):
        key = (kind, case["name"])
        if key not in cache:
            cache[key] = (_single_step_ref if kind == "step" else _rollout_ref)(case)
        return cache[key]
    return get


def _single_step_ref(case):
    k = case_knobs(case)
    bank = fp32_bank(64, k["W"], k["H"], seed=3, map_N=k["map_N"], wf=k["wf"])
    st, acts = injected_states(case, k, bank, N_STEP, 7)
    out = {}
    for which, kk in (("case", k), ("default", default_knobs_of(k))):
        orc = make_oracle(kk, N_STEP, bank, auto_reset=False, n_threads=ORACLE_THREADS)
        parity.load_oracle_state(orc, *st)
        out[which] = (orc.step(acts[None]), orc.pose.copy(), orc.ints.copy(), orc.lidar[:, :10].copy())
    return bank, st, acts, out


def _rollout_ref(case):
    k = case_knobs(case)
    bank = fp32_bank(64, k["W"], k["H"], seed=7, map_N=k["map_N"], wf=k["wf"])
    acts = np.random.RandomState(21).choice([0, 0, 1, 2], size=(K_ROLL, N_ROLL)).astype(np.int32)
    out = {}
    for which, kk in (("case", k), ("default", default_knobs_of(k))):
        orc = make_oracle(kk, N_ROLL, bank, auto_reset=True, seed=11, n_threads=ORACLE_THREADS)
        orc.reset()
        out[which] = (orc.step(acts), orc.stats_dict())
    return bank, acts, out


# ---------------------------------------------------------------------------------------------- a. one injected step
@pytest.mark.parametrize("case", CASES, ids=IDS)
@pytest.mark.parametrize("lanes", [1, 32])
def test_knob_single_step_against_oracle(case, lanes, oracle_runs):
    k = case_knobs(case)
    bank, st, acts, out = oracle_runs("step", case)
    ref, pose, ints, lidar = out["case"]
    env = make_env(k, N_STEP, bank, auto_reset=False, lanes_per_env=lanes, steps_in_flight=1)
    env.reset()
    env.set_state(*st)
    o, r, d, _ = env.step(torch.tensor(acts, device=env.device))
    o, r, d = o.cpu().numpy()[None], r.cpu().numpy()[None], d.cpu().numpy()[None]
    scale = max(k["W"], k["H"])
    rep = parity.compare_steps(ref, o, r, d, label=case["name"], scale=scale)
    assert rep["excluded_frac"] < 0.01, rep
    assert rep["max_pose_rel_err"] < 2 * parity.REL_TOL
    got = env.get_state()
    ok = ref["margins"][0].min(-1) >= 1e-3
    tol = parity.REL_TOL * np.maximum(1, np.abs(pose)) + parity.POSE_ABS * scale
    assert (np.abs(got["pose"] - pose) <= tol)[ok].all()
    assert (got["ints"][ok][:, :3] == ints[ok][:, :3]).all()
    f = ref["flags"][0]
    assert (f & oracle.FLAG_COLLIDING).any() and (f & oracle.FLAG_OOB).any()
    assert (lidar >= 0).any()
    if case.get("shell"):
        assert (f & oracle.FLAG_GOAL).any()
    # d. sensitivity: the kernel disagrees with the oracle at the default knobs
    kind, share = case["guard"]
    dref, dpose = out["default"][0], out["default"][1]
    bad = _disagree(dref, o, r, d)[0] | (np.abs(got["pose"] - dpose) > 1e-3 * np.maximum(1, np.abs(dpose))).any(-1)
    if kind == "step":
        assert bad[ok].mean() >= share, (case["name"], bad[ok].mean())
    elif kind == "uneventful":
        plain = ok & (f == 0)
        assert plain.sum() > N_STEP // 10
        assert (r[0][plain] == np.float32(k["step_penalty"])).all() and (r[0][plain] != dref["reward"][0][plain]).all()
    env.close()


# ---------------------------------------------------------------------------------------------- b. 32-step auto-reset rollout
STAT_KEYS = ("episodes", "collision", "oob", "timeout", "all_goals", "length_sum")


@pytest.mark.parametrize("case", CASES, ids=IDS)
@pytest.mark.parametrize("variant", ["serial", "T8", "T32"])
def test_knob_rollout_against_oracle(case, variant, oracle_runs):
    k = case_knobs(case)
    bank, acts, out = oracle_runs("roll", case)
    ref, so = out["case"]
    kw = dict(lanes_per_env=1, steps_in_flight=1) if variant == "serial" else dict(steps_in_flight=int(variant[1:]))
    env = make_env(k, N_ROLL, bank, auto_reset=True, seed=11, **kw)
    env.reset()
    obs, rew, done = [t.cpu().numpy() for t in env.rollout(torch.tensor(acts, device=env.device))]
    assert env.launch_info()["steps_in_flight"] == kw["steps_in_flight"]
    rep = parity.compare_steps(ref, obs, rew, done, margin_thr=parity.MARGIN_THR, label=case["name"], scale=max(k["W"], k["H"]))
    assert rep["grazing_frac"] < parity.MAX_EXCLUDED and rep["excluded_frac"] < parity.MAX_EXCLUDED_CUMULATIVE, rep
    assert rep["max_pose_rel_err"] < 2 * parity.REL_TOL
    s = env.stats()
    assert s["episodes"] == float(done.sum())
    for key in STAT_KEYS:
        assert abs(s[key] - so[key]) <= max(3, 0.01 * so[key]), (key, s[key], so[key])
    assert s["steps"] == so["steps"] == N_ROLL * K_ROLL
    kind, share = case["guard"]
    if kind == "roll":
        assert _disagree(out["default"][0], obs, rew, done).mean() >= share
    env.close()


# ---------------------------------------------------------------------------------------------- c. window == serial
@pytest.mark.parametrize("case", CASES, ids=IDS)
@pytest.mark.parametrize("T", [4, 32])
def test_knob_window_is_bit_identical_to_serial(case, T):
    k = case_knobs(case)
    n, K = 1000 + 3, 37
    bank = fp32_bank(64, k["W"], k["H"], seed=13, map_N=k["map_N"], wf=k["wf"])
    rng = np.random.RandomState(3)
    acts = torch.tensor(rng.choice([0, 0, 1, 2], size=(K, n)).astype(np.int32), device="cuda")
    st = parity.f32_inputs(*parity.random_states(rng, n, k["W"], k["H"], 64, bank["goals"], max_steps=k["max_steps"],
                                                 near=(bank["hull_xy"], bank["hull_n"]), hull=parity.ship_hull(k["ship_w"], k["ship_h"])))
    ref = run(make_env(k, n, bank, auto_reset=True, seed=5, lanes_per_env=1, steps_in_flight=1), acts, K, st)
    got = run(make_env(k, n, bank, auto_reset=True, seed=5, steps_in_flight=T), acts, K, st)
    assert ref[3]["steps_in_flight"] == 1 and got[3]["steps_in_flight"] == T
    assert_same(got, ref, "%s T=%d" % (case["name"], T))
    assert ref[0][2].sum() > 0


# ---------------------------------------------------------------------------------------------- e. host path
HOST_CASES = [c for c in CASES if c["name"] in ("wide", "penalty", "cap1", "spawn_mid")]


@pytest.mark.parametrize("case", HOST_CASES, ids=[c["name"] for c in HOST_CASES])
@pytest.mark.parametrize("n,K", [(1000, 100), (300, 7)])
def test_knob_host_path_matches_rollout(case, n, K):
    """shipsim_step_host rebuilds the rows and rewards from compacted frames with a reward-code table built from the
    step penalty: bit-identical to the device-resident rollout at these knobs."""
    k = case_knobs(case)
    bank = fp32_bank(64, k["W"], k["H"], seed=2, map_N=k["map_N"], wf=k["wf"])
    rng = np.random.RandomState(4)
    envs = [make_env(k, n, bank, auto_reset=True, seed=1) for _ in range(2)]
    for e in envs:
        e.reset()
    st = parity.f32_inputs(*parity.random_states(rng, n, k["W"], k["H"], 64, bank["goals"], max_steps=k["max_steps"]))
    for it in range(3):
        if it == 1:
            for e in envs:
                e.set_state(*st)
        acts = rng.randint(0, 3, (K, n)).astype(np.int32)
        o, r, d = [t.cpu().numpy() for t in envs[0].rollout(torch.tensor(acts, device="cuda"))]
        ho, hr, hd = envs[1].step_host(acts, K=K)
        assert np.array_equal(hr, r) and np.array_equal(hd, d), "call %d" % it
        assert np.array_equal(ho, o), "call %d" % it
        if case["name"] == "penalty":
            assert (r == np.float32(k["step_penalty"])).mean() > 0.5
    for e in envs:
        e.close()


# ---------------------------------------------------------------------------------------------- 3. spawn-row geometry
def _regular(cx, cy, r, m, phase=0.0):
    a = phase + np.linspace(0, 2 * np.pi, m, endpoint=False)
    return np.stack([cx + r * np.cos(a), cy + r * np.sin(a)], 1)


def _fan_reach_planes(hull, origin, k):
    """Planes of a CCW bank that pass the fan-reach test of plane_at_pose at a ship pointing straight up, in float64."""
    v = np.asarray(hull, dtype=np.float64)
    e = np.roll(v, -1, axis=0) - v
    nrm = np.stack([e[:, 1], -e[:, 0]], 1) / np.linalg.norm(e, axis=1)[:, None]
    d = ((np.asarray(origin) - v) * nrm).sum(1)
    deg = np.pi / 180.0
    delta, start = k["spread"] / 10 * deg, (90.0 - k["spread"] / 2) * deg
    mid, half = start + delta * 4.5, abs(delta) * 4.5
    ang = np.arccos(np.clip(-(nrm[:, 0] * np.cos(mid) + nrm[:, 1] * np.sin(mid)), -1, 1))
    reach = np.cos(np.maximum(0.0, ang - half)) if half < np.pi else np.ones(len(v))
    return (d >= 0) & (d <= k["lidar"] * reach)


FAR = np.array([[500.0, 500.0], [550.0, 500.0], [525.0, 540.0]])
SPAWN_GOALS = np.array([[60.0, 560.0], [120.0, 560.0], [180.0, 560.0], [240.0, 560.0], [540.0, 560.0]])
EDGE = 2e-3     # the reach-edge offset; the oracle's graze threshold (parity.MARGIN_THR) is 1e-3


def _spawn_origin(spawn_y):
    """The lidar origin at the spawn pose: body (300, spawn_y) + half the default hull's AABB (10, 22.5)."""
    return 310.0, spawn_y + 22.5


def _spawn_bank(kind, spawn_y):
    ox, oy = _spawn_origin(spawn_y)
    if kind == "inside":
        banks = [_regular(ox, oy, 12.0, 4, np.pi / 4)]
    elif kind == "big_row":
        banks = [_regular(ox, oy + 122.5, 60.0, 30, 0.1)]
    else:                        # an edge across the middle ray (straight up) at the lidar distance +- EDGE
        banks = [np.array([[290.0, y], [330.0, y], [330.0, y + 50.0], [290.0, y + 50.0]]) for y in (oy + 100.0 - EDGE, oy + 100.0 + EDGE)]
    b = pack_bank([(h, FAR) for h in banks], [SPAWN_GOALS] * len(banks))
    b["hull_xy"] = b["hull_xy"].astype(np.float32).astype(np.float64)
    return b


@pytest.mark.parametrize("kind", ["inside", "big_row", "reach_edge"])
@pytest.mark.parametrize("spawn_y", [25.0, 300.0])
def test_spawn_row_geometry(kind, spawn_y):
    """Episodes of three steps, so that every env is reset inside the kernel every few steps and each episode's first
    step runs from the spawn row built by build_spawn_rows_kernel: the lidar origin inside a bank, more planes facing
    the fan than a scratch row holds (the big-row path), and an edge at the lidar's reach."""
    k = knobs(max_steps=3, spawn_y=spawn_y)
    bank = _spawn_bank(kind, spawn_y)
    n, K = 515, 24
    if kind == "big_row":
        n_cand = source_constant("shipsim_geom.cuh", r"constexpr int kMaxCand = (\d+);")
        assert _fan_reach_planes(bank["hull_xy"][0, 0, :bank["hull_n"][0, 0]], _spawn_origin(spawn_y), k).sum() > n_cand
    acts = np.random.RandomState(1).randint(0, 3, (K, n)).astype(np.int32)
    orc = make_oracle(k, n, bank, auto_reset=True, seed=4, n_threads=ORACLE_THREADS)
    orc.reset()
    ref = orc.step(acts)
    runs = {}
    for name, kw in (("lanes1", dict(lanes_per_env=1, steps_in_flight=1)), ("lanes8", dict(lanes_per_env=8, steps_in_flight=1)),
                     ("T4", dict(steps_in_flight=4)), ("T32", dict(steps_in_flight=32))):
        runs[name] = run(make_env(k, n, bank, auto_reset=True, seed=4, **kw), torch.tensor(acts, device="cuda"), K)
        (obs, rew, done), _, _, _ = runs[name]
        rep = parity.compare_steps(ref, obs, rew, done, margin_thr=parity.MARGIN_THR, label="%s %s" % (kind, name))
        assert rep["grazing_frac"] < parity.MAX_EXCLUDED and rep["excluded_frac"] < parity.MAX_EXCLUDED_CUMULATIVE, rep
    for name in ("T4", "T32"):
        assert_same(runs[name], runs["lanes1"], "%s %s" % (kind, name))
    first = np.concatenate([np.ones((1, n), dtype=bool), ref["done"][:-1].astype(bool)])     # steps that begin at the spawn
    lid = ref["obs"][:, :, 22:32]
    if kind == "inside":
        assert ref["done"].all() and (ref["flags"] & oracle.FLAG_COLLIDING).all()
    elif kind == "big_row":
        assert ((lid[first] >= 0).sum(-1) >= 5).all()
    else:
        mid = lid[first][:, 5]
        assert (np.abs(mid - (100.0 - EDGE)) < 1e-4).any() and (mid == -1.0).any()


# ---------------------------------------------------------------------------------------------- 4. 64-bit keys
def test_64_bit_seed_and_env_ids():
    """A seed and global env ids above 2^32: the random agent's actions and the scenario picks are keyed by all 64
    bits; truncating either anywhere between Python, ctypes and the kernels changes the episodes."""
    seed, off = 2 ** 63 + 12345, 2 ** 32 + 7
    k = knobs(max_steps=5)
    bank = fp32_bank(64, 600.0, 600.0, seed=9)
    n, K = 2048, 24
    orc = make_oracle(k, n, bank, auto_reset=True, seed=seed, env_id_offset=off, n_threads=ORACLE_THREADS)
    orc.reset()
    ref = orc.step(None, K=K)
    for kw in (dict(lanes_per_env=1, steps_in_flight=1), dict(steps_in_flight=8)):
        env = make_env(k, n, bank, auto_reset=True, seed=seed, env_id_offset=off, **kw)
        env.reset()
        obs, rew, done = [t.cpu().numpy() for t in env.rollout(None, K=K)]
        rep = parity.compare_steps(ref, obs, rew, done, margin_thr=parity.MARGIN_THR, label="64-bit keys")
        assert rep["grazing_frac"] < parity.MAX_EXCLUDED and rep["excluded_frac"] < parity.MAX_EXCLUDED_CUMULATIVE, rep
        ok = (ref["margins"][:, :, :4].min(-1) >= parity.MARGIN_THR).all(0) & (ref["margins"][:, :, 4:14].min(-1) >= parity.MARGIN_THR).all(0)
        got = env.get_state()["ints"]
        assert ok.mean() > 0.9 and np.array_equal(got[ok][:, 3:5], orc.ints[ok][:, 3:5])
        assert orc.ints[:, 4].min() >= 4                    # every env went through several resets
        env.close()
    # the keys matter: 32-bit truncations pick other scenarios
    for s, o in ((seed & 0xFFFFFFFF, off), (seed, off & 0xFFFFFFFF)):
        t = make_oracle(k, n, bank, auto_reset=True, seed=s, env_id_offset=o, n_threads=ORACLE_THREADS)
        t.reset()
        t.step(None, K=K)
        assert (t.ints[:, 3] != orc.ints[:, 3]).mean() > 0.9
