"""-m gpu: lidar fans of 1 to 32 beams (LidarConfig.N_BEAMS with honour_lidar_config=True) -- the wide step kernel.

The wide kernel is the tuned kernel's code with a 32-reading frame slot and the beam count read at run time, so besides
the float64 oracle it is held to the tuned kernel itself: lidar feeds nothing back into the dynamics, so for the same
seed, actions and map every non-lidar output must equal the 10-beam run's bit for bit."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from helpers import ORACLE_THREADS, assert_same, config_classes, fp32_bank, knobs, make_env, make_oracle, run  # noqa: E402
import parity  # noqa: E402

BEAMS = [1, 3, 7, 11, 16, 20, 32]                   # 32, 10, 4, 2, 2, 1 and 1 envs per ray pass
SPREADS = [90.0, 180.0, 360.0, -120.0]


def widen(lidar, nb, rng):
    """[n, 10] injected readings -> [n, nb]: the first min(10, nb), the rest random (-1 or a reading)."""
    n = lidar.shape[0]
    out = np.where(rng.rand(n, nb) < 0.5, -1.0, rng.uniform(0, 100, (n, nb))).astype(np.float32).astype(np.float64)
    k = min(10, nb)
    out[:, :k] = lidar[:, :k]
    return out


def injected(nb, n, seed):
    """Random states, ships near a bank vertex and lidar origins inside a bank, with nb injected readings each."""
    bank = fp32_bank(64, 600, 600, seed=3)
    rng = np.random.RandomState(seed)
    q = n // 3
    near = (bank["hull_xy"], bank["hull_n"])
    parts = [parity.random_states(rng, q, 600, 600, 64, bank["goals"]),
             parity.random_states(rng, q, 600, 600, 64, bank["goals"], near=near)]
    m = n - 2 * q
    p, i, li, _ = parity.origin_inside_bank_states(rng, m, bank["hull_xy"], bank["hull_n"], 64)
    parts.append((p, i, li, bank["goals"][i[:, 3]].reshape(m, 10), np.zeros(m)))
    pose, ints, lidar, goals, ret = parity.f32_inputs(*parity.concat_states(parts))
    return bank, (pose, ints, widen(lidar, nb, rng), goals, ret), rng.randint(0, 3, n).astype(np.int32)


# ---------------------------------------------------------------------------------------------- against the oracle
@pytest.mark.parametrize("spread", SPREADS)
@pytest.mark.parametrize("nb", BEAMS)
@pytest.mark.parametrize("lanes", [1, 32])
def test_wide_single_step_against_oracle(nb, spread, lanes):
    n = 4096 - 5
    bank, st, acts = injected(nb, n, 7 + nb)
    k = knobs(n_beams=nb, spread=spread)
    orc = make_oracle(k, n, bank, n_threads=ORACLE_THREADS)
    parity.load_oracle_state(orc, *st, n_beams=nb)
    ref = orc.step(acts[None])
    env = make_env(k, n, bank, auto_reset=False, lanes_per_env=lanes)
    env.reset()
    env.set_state(*st)
    o, r, d, _ = env.step(torch.tensor(acts, device=env.device))
    assert o.shape == (n, 2 * (6 + nb))
    o, r, d = o.cpu().numpy()[None], r.cpu().numpy()[None], d.cpu().numpy()[None]
    rep = parity.compare_steps(ref, o, r, d, label="nb=%d spread=%g" % (nb, spread), n_beams=nb)
    assert rep["excluded_frac"] < 0.01 and rep["max_pose_rel_err"] < 2 * parity.REL_TOL, rep
    lid = o[0, :, -nb:]
    assert (lid[n - n // 3:] == 100.0).mean() > 0.5        # origins inside a bank: full-length readings
    got = env.get_state()
    ok = ref["margins"][0].min(-1) >= 1e-3
    tol = parity.REL_TOL * np.maximum(1, np.abs(orc.pose)) + parity.POSE_ABS * 600
    assert (np.abs(got["pose"] - orc.pose) <= tol)[ok].all()
    assert (got["ints"][ok][:, :3] == orc.ints[ok][:, :3]).all()
    assert np.array_equal(got["lidar"], o[0, :, -nb:])       # the state keeps what the frame reports
    env.close()


STAT_KEYS = ("episodes", "collision", "oob", "timeout", "all_goals", "length_sum")


@pytest.mark.parametrize("spread", SPREADS)
@pytest.mark.parametrize("nb", BEAMS)
def test_wide_rollout_against_oracle(nb, spread):
    n, K = 2048 + 3, 32
    hist = 1 if nb in (3, 20) else 2
    bank = fp32_bank(64, 600, 600, seed=7)
    k = knobs(n_beams=nb, spread=spread, hist=hist)
    acts = np.random.RandomState(21).choice([0, 0, 1, 2], size=(K, n)).astype(np.int32)
    orc = make_oracle(k, n, bank, auto_reset=True, seed=11, n_threads=ORACLE_THREADS)
    orc.reset()
    ref = orc.step(acts)
    so = orc.stats_dict()
    env = make_env(k, n, bank, auto_reset=True, seed=11, steps_in_flight=1)
    env.reset()
    obs, rew, done = [t.cpu().numpy() for t in env.rollout(torch.tensor(acts, device=env.device))]
    assert obs.shape == (K, n, hist * (6 + nb))
    rep = parity.compare_steps(ref, obs, rew, done, margin_thr=parity.MARGIN_THR, label="nb=%d" % nb, n_beams=nb)
    assert rep["grazing_frac"] < parity.MAX_EXCLUDED and rep["excluded_frac"] < parity.MAX_EXCLUDED_CUMULATIVE, rep
    assert rep["max_pose_rel_err"] < 2 * parity.REL_TOL
    s = env.stats()
    for key in STAT_KEYS:
        assert abs(s[key] - so[key]) <= max(3, 0.01 * so[key]), (key, s[key], so[key])
    assert done.sum() > 0 and (obs[..., -nb:] >= 0).any()
    env.close()


# ---------------------------------------------------------------------------------------------- physics untouched
def _non_lidar(obs, nb, hist):
    F = 6 + nb
    return obs.reshape(obs.shape[0], obs.shape[1], hist, F)[..., :6]


@pytest.mark.parametrize("hist", [1, 2])
def test_physics_bit_identical_to_the_ten_beam_kernel(hist):
    n, K = 3000, 40
    bank = fp32_bank(64, 600, 600, seed=5)
    rng = np.random.RandomState(2)
    pose, ints, lidar, goals, ret = parity.f32_inputs(*parity.random_states(rng, n, 600, 600, 64, bank["goals"], near=(bank["hull_xy"], bank["hull_n"])))
    acts = torch.tensor(rng.choice([0, 0, 1, 2], size=(K, n)).astype(np.int32), device="cuda")
    (o10, r10, d10), s10, t10, _ = run(make_env(knobs(hist=hist, max_steps=60), n, bank, seed=9, lanes_per_env=4), acts, K,
                                        (pose, ints, lidar, goals, ret))
    for nb in BEAMS:
        (o, r, d), s, t, info = run(make_env(knobs(n_beams=nb, hist=hist, max_steps=60), n, bank, seed=9, lanes_per_env=4), acts, K,
                                    (pose, ints, widen(lidar, nb, rng), goals, ret))
        assert info["steps_in_flight"] == 1
        assert np.array_equal(_non_lidar(o, nb, hist), _non_lidar(o10, 10, hist)), nb
        assert np.array_equal(r, r10) and np.array_equal(d, d10), nb
        for key in ("pose", "ints", "goals", "ep_return"):
            assert np.array_equal(s[key], s10[key]), (nb, key)
        counts = [key for key in t if key != "return_sum"]
        assert [t[key] for key in counts] == [t10[key] for key in counts], nb           # counts and lengths
        assert t["return_sum"] == pytest.approx(t10["return_sum"], rel=1e-9)           # cross-CTA atomics: any order
    assert d10.sum() > n // 4


@pytest.mark.parametrize("spread", [90.0, 180.0])
def test_twenty_beam_even_slots_match_the_tuned_kernel(spread):
    n, K = 4096, 32
    bank = fp32_bank(64, 600, 600, seed=9)
    rng = np.random.RandomState(4)
    pose, ints, lidar, goals, ret = parity.f32_inputs(*parity.random_states(rng, n, 600, 600, 64, bank["goals"], near=(bank["hull_xy"], bank["hull_n"])))
    l20 = np.full((n, 20), -1.0)
    l20[:, 0::2] = lidar
    acts = torch.tensor(rng.choice([0, 0, 1, 2], size=(K, n)).astype(np.int32), device="cuda")
    (o10, _, _), _, _, _ = run(make_env(knobs(spread=spread), n, bank, seed=3, steps_in_flight=1), acts, K, (pose, ints, lidar, goals, ret))
    (o20, _, _), _, _, _ = run(make_env(knobs(n_beams=20, spread=spread), n, bank, seed=3, steps_in_flight=1), acts, K,
                               (pose, ints, l20, goals, ret))
    a = o10.reshape(K, n, 2, 16)[..., 6:].astype(np.float64)
    b = o20.reshape(K, n, 2, 26)[..., 6::2].astype(np.float64)
    # the two fans' rays agree to an ulp of the angle: within the lidar tolerance at the worst conditioning seen
    err = np.abs(a - b)
    assert (err <= 1e-4 * np.maximum(1, np.abs(a)) * 50).all(), err.max()
    assert (err <= 1e-4 * np.maximum(1, np.abs(a))).mean() > 0.999
    assert (a >= 0).mean() > 0.05


# ---------------------------------------------------------------------------------------------- invariances
@pytest.mark.parametrize("nb", [7, 32])
def test_lanes_launches_and_sharding_are_invisible(nb):
    n, K = 1500, 36
    bank = fp32_bank(64, 600, 600, seed=11)
    k = knobs(n_beams=nb, max_steps=40)
    rng = np.random.RandomState(8)
    pose, ints, lidar, goals, ret = parity.f32_inputs(*parity.random_states(rng, n, 600, 600, 64, bank["goals"], near=(bank["hull_xy"], bank["hull_n"])))
    st = (pose, ints, widen(lidar, nb, rng), goals, ret)
    acts = torch.tensor(rng.choice([0, 0, 1, 2], size=(K, n)).astype(np.int32), device="cuda")
    ref = run(make_env(k, n, bank, seed=6, lanes_per_env=1), acts, K, st)
    for g in (2, 4, 8, 16, 32):
        got = run(make_env(k, n, bank, seed=6, lanes_per_env=g), acts, K, st)
        assert got[3]["lanes_per_env"] == g
        assert_same(got, ref, "nb=%d lanes=%d" % (nb, g))
    # K launches of one step = one launch of K steps
    env = make_env(k, n, bank, seed=6, lanes_per_env=8)
    env.reset()
    env.set_state(*st)
    rows = [[t.cpu().numpy() for t in env.rollout(acts[k:k + 1])] for k in range(K)]
    for j in range(3):
        assert np.array_equal(np.concatenate([r[j] for r in rows]), ref[0][j])
    # sharding: two halves with env_id_offset = one batch
    h = n // 2
    parts = []
    for lo, hi in ((0, h), (h, n)):
        e = make_env(k, hi - lo, bank, seed=6, lanes_per_env=2, env_id_offset=lo)
        parts.append(run(e, acts[:, lo:hi].contiguous(), K, tuple(np.asarray(x)[lo:hi] for x in st)))
    for j in range(3):
        assert np.array_equal(np.concatenate([p[0][j] for p in parts], axis=1), ref[0][j])
    assert ref[0][2].sum() > 0


def test_full_size_build_against_small_build_and_oracle():
    """262,144 envs at one lane each: the 128-thread G = 1 build with its 68 KB of dynamic shared memory."""
    nb, n, K = 32, 262144, 8
    bank = fp32_bank(64, 600, 600, seed=5)
    k = knobs(n_beams=nb)
    big = make_env(k, n, bank, seed=12, lanes_per_env=1)
    small = make_env(k, n, bank, seed=12, lanes_per_env=2)
    a = run(big, None, K)
    b = run(small, None, K)
    assert a[3]["threads_per_cta"] == 128 and a[3]["lanes_per_env"] == 1
    assert_same(a, b, "full size")
    sub = 4096
    orc = make_oracle(k, n, bank, auto_reset=True, seed=12, n_threads=ORACLE_THREADS)
    orc.reset()
    ref = orc.step(None, K=K)
    rep = parity.compare_steps({key: v[:, :sub] for key, v in ref.items()}, a[0][0][:, :sub], a[0][1][:, :sub], a[0][2][:, :sub],
                               margin_thr=parity.MARGIN_THR, label="full size", n_beams=nb)
    assert rep["excluded_frac"] < parity.MAX_EXCLUDED_CUMULATIVE, rep


def test_auto_selection_runs_the_serial_kernel():
    env = make_env(knobs(n_beams=16), 4096, fp32_bank(64, 600, 600, seed=1))
    env.reset()
    env.rollout(None, K=64)
    torch.cuda.synchronize()
    assert env.launch_info()["steps_in_flight"] == 1
    with pytest.raises(NotImplementedError, match="steps_in_flight"):
        make_env(knobs(n_beams=16), 64, None, steps_in_flight=8, n_scenarios=4)


# ---------------------------------------------------------------------------------------------- surfaces
@pytest.mark.parametrize("hist", [1, 2])
def test_episode_log_rows_equal_no_reset_rows(hist):
    nb, n, K = 32, 700, 64
    bank = fp32_bank(64, 600, 600, seed=13)
    rng = np.random.RandomState(3)
    pose, ints, lidar, goals, ret = parity.f32_inputs(*parity.random_states(rng, n, 600, 600, 64, bank["goals"], max_steps=200,
                                                                            near=(bank["hull_xy"], bank["hull_n"])))
    st = (pose, ints, widen(lidar, nb, rng), goals, ret)
    acts = torch.tensor(rng.choice([0, 0, 1, 2], size=(K, n)).astype(np.int32), device="cuda")
    k = knobs(n_beams=nb, hist=hist, max_steps=200)
    ref = make_env(k, n, bank, auto_reset=False, seed=5, lanes_per_env=4)
    got = make_env(k, n, bank, auto_reset=True, seed=5, lanes_per_env=4)
    got.enable_episode_log(K * n)
    outs = []
    for e in (ref, got):
        e.reset()
        e.set_state(*st)
        outs.append([t.cpu().numpy() for t in e.rollout(acts)])
    (o0, _, d0), (o1, _, d1) = outs
    ep = {k: v.cpu().numpy() for k, v in got.episodes().items()}
    assert len(ep["env"]) == int(d1.sum()) > n // 8
    assert ep["terminal_obs"].shape[1] == hist * (6 + nb)
    seen = set()
    for j in range(len(ep["env"])):
        e, k = int(ep["env"][j]), int(ep["k"][j])
        if e in seen:
            continue
        seen.add(e)
        assert d0[:k, e].sum() == 0 and d0[k, e] == 1
        assert np.array_equal(ep["terminal_obs"][j], o0[k, e]), (e, k)


@pytest.mark.parametrize("n,K", [(8, 1), (5000, 40)])
def test_step_host_equals_device_rollout(n, K):
    nb = 20
    bank = fp32_bank(64, 600, 600, seed=2)
    envs = [make_env(knobs(n_beams=nb, max_steps=50), n, bank, seed=1) for _ in range(2)]
    for e in envs:
        e.reset()
    rng = np.random.RandomState(4)
    for it in range(3):
        acts = rng.randint(0, 3, (K, n)).astype(np.int32)
        o, r, d = [t.cpu().numpy() for t in envs[0].rollout(torch.tensor(acts, device="cuda"))]
        if K == 1:
            ho, hr, hd = envs[1].step_np(acts[0])
            ho, hr, hd = ho[None], hr[None], hd[None]
        else:
            ho, hr, hd = envs[1].step_host(acts, K=K)
        assert np.array_equal(ho, o) and np.array_equal(hr, r) and np.array_equal(hd.astype(np.uint8), d), it


def test_history_three_against_oracle():
    nb, n, K = 16, 1024, 24
    bank = fp32_bank(64, 600, 600, seed=7)
    k = knobs(n_beams=nb, hist=3, max_steps=30)
    acts = np.random.RandomState(5).choice([0, 0, 1, 2], size=(K, n)).astype(np.int32)
    orc = make_oracle(k, n, bank, auto_reset=True, seed=2, n_threads=ORACLE_THREADS)
    orc.reset()
    ref = orc.step(acts)
    env = make_env(k, n, bank, auto_reset=True, seed=2)
    env.reset()
    obs, rew, done = [t.cpu().numpy() for t in env.rollout(torch.tensor(acts, device=env.device))]
    assert obs.shape == (K, n, 3 * 22)
    # compare_steps knows the 1- and 2-frame layouts: hold the newest two frames to it, the oldest to the one before
    rep = parity.compare_steps(dict(ref, obs=ref["obs"][..., 22:]), obs[..., 22:], rew, done, margin_thr=parity.MARGIN_THR,
                               label="hist3", n_beams=nb)
    assert rep["excluded_frac"] < parity.MAX_EXCLUDED_CUMULATIVE, rep
    assert np.array_equal(obs[1:, :, :22], np.where(done[1:, :, None].astype(bool), -1.0, obs[:-1, :, 22:44]).astype(np.float32))
    assert done.sum() > n // 4


def test_state_round_trip_and_render():
    nb, n = 32, 64
    env = make_env(knobs(n_beams=nb), n, fp32_bank(64, 600, 600, seed=1), seed=1)
    env.reset()
    env.rollout(None, K=20)
    s = env.get_state()
    assert s["lidar"].shape == (n, nb)
    env.set_state(s["pose"], s["ints"], s["lidar"], s["goals"], s["ep_return"])
    s2 = env.get_state()
    for k in s:
        assert np.array_equal(s[k], s2[k]), k
    # render: one marker per ray of the fan at the ray's end -- every ray of a ship alone on open water is green
    lid = np.full((n, nb), -1.0)
    pose = s["pose"].copy()
    pose[:, :] = 0
    pose[:, 0], pose[:, 1] = 300.0, 300.0
    env.set_state(pose, s["ints"], lid, s["goals"], s["ep_return"])
    ints = s["ints"]
    img = env.render("rgb_array", env_index=0, size=(600, 600)).cpu().numpy()
    hx, hy = parity.lidar_origin_offset(np.zeros(1))
    ang = np.radians(90.0 - 45.0 + 90.0 / nb * np.arange(nb))
    ends = np.stack([300 + hx[0] + 100 * np.cos(ang), 300 + hy[0] + 100 * np.sin(ang)], 1)
    assert all(tuple(img[int(600 - y), int(x)]) == (0, 255, 0) for x, y in ends)
    # a reading on ray 31 moves its marker (red: a hit) to that distance
    lid[0, 31] = 50.0
    env.set_state(pose, ints, lid, s["goals"], s["ep_return"])
    img = env.render("rgb_array", env_index=0, size=(600, 600)).cpu().numpy()
    x, y = 300 + hx[0] + 50 * np.cos(ang[31]), 300 + hy[0] + 50 * np.sin(ang[31])
    assert tuple(img[int(600 - y), int(x)]) == (255, 0, 0)


def test_vec_env_episode_info_at_32_beams():
    from ship_sim_gym_b200.adapters import ShipVecEnv
    n = 128
    vec = ShipVecEnv(n, episode_info=True, seed=8, n_scenarios=32, env_config=config_classes(knobs(n_beams=32, max_steps=30))[1],
                     honour_lidar_config=True)
    obs = vec.reset()
    assert obs.shape == (n, 76)
    rng = np.random.RandomState(1)
    n_info = 0
    for t in range(70):
        obs, rew, done, infos = vec.step(rng.randint(0, 3, n))
        assert obs.shape == (n, 76)
        for e in np.nonzero(done)[0]:
            term = infos[e]["terminal_observation"]
            assert term.shape == (76,) and not (term[:38] == -1).all() or infos[e]["episode"]["l"] == 1
            assert (obs[e, :38] == -1).all()
            n_info += 1
    assert n_info > n


def test_rollout_collector_graph_replay_matches_eager_at_76_inputs():
    """MlpPolicy(obs_dim=2 * (6 + 32)) on the torch path (the fused policy kernel takes 32 inputs only): a replayed
    CUDA graph and the eager loop both make T steps of the wide kernel that obey the env's invariants."""
    from ship_sim_gym_b200.rollout import MlpPolicy, RolloutCollector
    n, T = 1024, 16
    torch.manual_seed(0)
    policy = MlpPolicy(obs_dim=76).cuda()
    out = []
    for use_graph in (False, True):
        env = make_env(knobs(n_beams=32), n, fp32_bank(64, 600, 600, seed=1), seed=1)
        col = RolloutCollector(env, policy, T=T, use_graph=use_graph)
        assert not col._kernel
        col.collect()
        launches0 = env.launch_info()["launches"]
        col.collect()
        torch.cuda.synchronize()
        out.append((col.rewards.clone(), col.dones.clone(), col.obs.clone(), env.launch_info()["launches"] - launches0))
        assert col.actions.min() >= 0 and col.actions.max() <= 2
        assert torch.isfinite(col.adv).all() and torch.isfinite(col.returns).all()
        env.close()
    assert out[0][3] == T and out[1][3] == 0
    for rew, done, obs, _ in out:
        assert obs.shape[-1] == 76
        r = rew.cpu().numpy()
        assert (np.isclose(r, 1.0) | np.isclose(r, -1.0) | np.isclose(r, -0.01)).all()
        older = obs[1:, :, :38].cpu().numpy()
        assert ((older == -1).all(-1) == done.cpu().numpy().astype(bool)).all()


def test_fresh_maps_against_oracle_at_32_beams():
    nb, n, K, S = 32, 2048, 32, 64
    k = knobs(n_beams=nb)
    env = make_env(k, n, None, n_scenarios=S, seed=11, scenario_source="device", auto_reset=True, fresh_maps=True)
    bank = env.read_scenarios()
    bd = dict(hull_xy=bank.hull_xy, hull_n=bank.hull_n, goals=bank.goals.astype(np.float32).astype(np.float64))
    orc = make_oracle(k, n, bd, auto_reset=True, seed=11, pick_base=0, pick_count=S // 4, n_threads=ORACLE_THREADS)
    env.reset()
    orc.reset()
    rng = np.random.RandomState(3)
    pose, ints, lidar, goals, ret = parity.f32_inputs(*parity.random_states(rng, n, 600, 600, S, bd["goals"], near=(bd["hull_xy"], bd["hull_n"])))
    st = (pose, ints, widen(lidar, nb, rng), goals, ret)
    env.set_state(*st)
    parity.load_oracle_state(orc, *st, n_beams=nb)
    acts = rng.randint(0, 3, (K, n)).astype(np.int32)
    obs, rew, done = [t.cpu().numpy() for t in env.rollout(torch.tensor(acts, device=env.device))]
    ref = orc.step(acts)
    rep = parity.compare_steps(ref, obs, rew, done, margin_thr=parity.MARGIN_THR, label="fresh maps", n_beams=nb)
    assert done.sum() > n // 4
    assert rep["grazing_frac"] < parity.MAX_EXCLUDED and rep["excluded_frac"] < parity.MAX_EXCLUDED_CUMULATIVE, rep
    env.close()


def test_reset_observation_layout_on_the_device():
    for nb in (1, 7, 32):
        env = make_env(knobs(n_beams=nb), 5, fp32_bank(64, 600, 600, seed=1), seed=1)
        obs = env.reset().cpu().numpy()
        F = 6 + nb
        assert obs.shape == (5, 2 * F)
        assert (obs[:, :F] == -1).all() and (obs[:, F + 2:F + 4] == 0).all() and (obs[:, F + 6:] == -1).all()
        assert (obs[:, F:F + 2] == [300.0, 25.0]).all()
