"""-m gpu: the episode log (shipsim_episode_log_bind; BatchedShipEnv.enable_episode_log / episodes()).

With auto-reset the kernels replace a done env's observation by the reset observation; the log keeps what the reset
overwrites.  Its terminal rows must be, bit for bit, the rows an auto_reset=False launch writes for the same env at the
same step, in every kernel (serial-in-time step kernel at several lanes per env, window kernel at every window), both
kernel history sizes, the host paths and the host-assembled long histories; its counts must match the done flags and the
statistics vector, and turning it on must change no output."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from helpers import config_classes, fp32_bank, knobs, make_env  # noqa: E402
import parity  # noqa: E402


def _np(ep):
    return {k: v.cpu().numpy() for k, v in ep.items()}


def _first_records(ep):
    """index of each env's first record (records are sorted by call, k, env)"""
    first = {}
    for j, e in enumerate(ep["env"]):
        first.setdefault(int(e), j)
    return first


def _f32_return(ret0, rew, k):
    """ShipEnv.cumulative_reward after step k, added in fp32 one step at a time as the kernels do"""
    r = np.float32(ret0)
    for j in range(k + 1):
        r = np.float32(r + np.float32(rew[j]))
    return r


KERNELS = [dict(steps_in_flight=1, lanes_per_env=1), dict(steps_in_flight=1, lanes_per_env=4),
           dict(steps_in_flight=1, lanes_per_env=32), dict(steps_in_flight=4), dict(steps_in_flight=8),
           dict(steps_in_flight=16), dict(steps_in_flight=32)]


@pytest.mark.parametrize("hist", [1, 2])
@pytest.mark.parametrize("kern", KERNELS, ids=lambda k: "sif%d_g%d" % (k["steps_in_flight"], k.get("lanes_per_env", 0)))
def test_terminal_rows_equal_no_reset_rows(kern, hist):
    W = H = 600
    n, K, max_steps = 700, 64, 200
    bank = fp32_bank(48, W, H, seed=13)
    rng = np.random.RandomState(3)
    st = parity.f32_inputs(*parity.random_states(rng, n, W, H, 48, bank["goals"], max_steps=max_steps,
                                                 near=(bank["hull_xy"], bank["hull_n"])))
    acts = torch.tensor(rng.choice([0, 0, 1, 2], size=(K, n)).astype(np.int32), device="cuda")
    k = knobs(hist=hist, max_steps=max_steps)
    ref = make_env(k, n, bank, auto_reset=False, seed=5, **kern)
    got = make_env(k, n, bank, auto_reset=True, seed=5, **kern)
    got.enable_episode_log(K * n)
    outs = []
    for e in (ref, got):
        e.reset()
        e.set_state(*st)
        outs.append([t.cpu().numpy() for t in e.rollout(acts)])
    assert got.launch_info()["steps_in_flight"] == kern["steps_in_flight"]
    (o0, r0, d0), (o1, r1, d1) = outs
    ep = _np(got.episodes())
    assert len(ep["env"]) == int(d1.sum()) > n // 8
    first = _first_records(ep)
    pose, ints, lidar, goals, ret = st
    for e, j in first.items():
        k = int(ep["k"][j])
        assert d0[:k, e].sum() == 0 and d0[k, e] == 1 and d1[:k + 1, e].sum() == 1, (e, k)
        assert np.array_equal(r0[:k + 1, e], r1[:k + 1, e])
        row = ep["terminal_obs"][j]
        assert np.array_equal(row, o0[k, e]), (e, k, row, o0[k, e])
        assert ep["length"][j] == ints[e, 2] + k + 1
        assert ep["return"][j] == _f32_return(ret[e], r0[:, e], k)
        assert ep["scenario"][j] == ints[e, 3] and ep["episode"][j] == ints[e, 4]
        # the reasons, read off the terminal row and the step's reward
        x, y, gx, gy = row[-16], row[-15], row[-12], row[-11]
        assert ep["oob"][j] == (x < 0 or x > W or y < 0 or y > H)
        assert ep["all_goals"][j] == (gx == -1 and gy == -1)
        assert ep["truncated"][j] == (ep["length"][j] >= max_steps and not (ep["oob"][j] or ep["all_goals"][j] or ep["collision"][j]))
        assert ep["goal"][j] == (r0[k, e] == 1.0)
        if not (ep["oob"][j] or ep["all_goals"][j] or ep["length"][j] >= max_steps):
            assert ep["collision"][j]
    assert ep["collision"].any() and ep["oob"].any() and ep["all_goals"].any() and ep["truncated"].any()


def _run_full(n, K, log, **kw):
    env = make_env(knobs(), n, fp32_bank(64, 600, 600, seed=5), seed=17, **kw)
    if log:
        env.enable_episode_log(n * K // 4)
    env.reset()
    s0 = env.stats_tensor().clone()
    out = [t.cpu().numpy() for t in env.rollout(None, K=K)]
    torch.cuda.synchronize()
    stats = (env.stats_tensor() - s0).cpu().numpy()
    return env, out, env.get_state(), stats, (_np(env.episodes()) if log else None)


def test_full_size_both_kernels_and_log_changes_nothing():
    """4,096 envs x 1,000 random-agent steps (the benchmark shape)."""
    n, K = 4096, 1000
    e_w, out_w, st_w, stats_w, ep_w = _run_full(n, K, True)
    assert e_w.launch_info()["steps_in_flight"] == 16
    e_s, out_s, st_s, stats_s, ep_s = _run_full(n, K, True, steps_in_flight=1, lanes_per_env=1)
    _, out_o, st_o, stats_o, _ = _run_full(n, K, False)
    for a, b in zip(out_w, out_o):
        assert np.array_equal(a, b)
    for k in st_w:
        assert np.array_equal(st_w[k], st_o[k]), k
    assert np.array_equal(np.delete(stats_w, 1), np.delete(stats_o, 1))
    assert stats_w[1] == pytest.approx(stats_o[1], rel=1e-5)       # (the return sums are atomics in any order)
    for k in ep_w:
        assert np.array_equal(ep_w[k], ep_s[k]), k
    # one record per done flag and vice versa
    done = out_w[2]
    kk, ee = np.nonzero(done)
    order = np.lexsort((ee, kk))
    assert np.array_equal(ep_w["k"], kk[order]) and np.array_equal(ep_w["env"], ee[order])
    # the statistics vector's deltas (shipsim_stat)
    assert len(ep_w["env"]) == stats_w[0]
    assert ep_w["length"].sum() == stats_w[2]
    assert ep_w["collision"].sum() == stats_w[4] and ep_w["oob"].sum() == stats_w[5]
    assert (ep_w["length"] >= 1000).sum() == stats_w[6] and ep_w["all_goals"].sum() == stats_w[7]
    assert ep_w["return"].astype(np.float64).sum() == pytest.approx(stats_w[1], rel=1e-5)


@pytest.mark.parametrize("regime", ["k1_zero_copy", "small_copies", "large_compacted", "dma_share"])
def test_step_host_records_equal_device_rollout(regime, monkeypatch):
    n, K = {"k1_zero_copy": (256, 1), "small_copies": (1024, 8), "large_compacted": (4096, 64), "dma_share": (4096, 64)}[regime]
    bank = fp32_bank(64, 600, 600, seed=5)
    rng = np.random.RandomState(7)
    acts = rng.randint(0, 3, (K, n)).astype(np.int32)
    dev, host = make_env(knobs(max_steps=40), n, bank, seed=9), make_env(knobs(max_steps=40), n, bank, seed=9)
    for e in (dev, host):
        e.enable_episode_log(n * (K + 30))
        e.reset()
    # a few steps first, so that episodes are under way
    warm = rng.randint(0, 3, (30, n)).astype(np.int32)
    dev.rollout(torch.tensor(warm, device="cuda"))
    host.rollout(torch.tensor(warm, device="cuda"))
    dev.episodes(), host.episodes()
    o_d = [t.cpu().numpy() for t in dev.rollout(torch.tensor(acts, device="cuda"))]
    if regime == "dma_share":
        monkeypatch.setenv("SHIPSIM_HOST_DMA_ENVS", str(n // 2))
    pin = regime in ("k1_zero_copy", "dma_share")

    def mk(*shape, dt):
        t = torch.empty(*shape, dtype=dt)
        return (t.pin_memory() if pin else t).numpy()
    out = (mk(K, n, 32, dt=torch.float32), mk(K, n, dt=torch.float32), mk(K, n, dt=torch.uint8))
    host.step_host(acts, K=K, out=out)
    for a, b in zip(out, o_d):
        assert np.array_equal(a, b)
    ed, eh = _np(dev.episodes()), _np(host.episodes())
    assert len(ed["env"]) > 0 and ed["k"].max() >= K // 2
    for k in ed:
        if k != "call":
            assert np.array_equal(ed[k], eh[k]), k


@pytest.mark.parametrize("hist", [3, 4])
def test_long_histories_terminal_obs(hist):
    n, K = 600, 40
    bank = fp32_bank(48, 600, 600, seed=13)
    rng = np.random.RandomState(11)
    k = knobs(hist=hist, max_steps=25)
    ref = make_env(k, n, bank, auto_reset=False, seed=2)
    got = make_env(k, n, bank, auto_reset=True, seed=2)
    got.enable_episode_log(n * K)
    for e in (ref, got):
        e.reset()
    st = ref.get_state()
    got.set_state(st["pose"], st["ints"], st["lidar"], st["goals"], st["ep_return"])
    acts = rng.randint(0, 3, (K, n)).astype(np.int32)
    # two single steps (step()), then a rollout: both assembly paths
    o_ref = [ref.step(torch.tensor(acts[i], device="cuda"))[0][None] for i in range(2)] + [ref.rollout(torch.tensor(acts[2:], device="cuda"))[0]]
    for i in range(2):
        got.step(torch.tensor(acts[i], device="cuda"))
    got.rollout(torch.tensor(acts[2:], device="cuda"))
    o_ref = torch.cat(o_ref).cpu().numpy()
    ep = _np(got.episodes())
    first = _first_records(ep)
    assert len(first) > n // 2
    call0 = got._calls - 3                      # step(), step(), rollout()
    for e, j in first.items():
        kk = int(ep["k"][j]) + int(ep["call"][j] - call0)
        assert np.array_equal(ep["terminal_obs"][j], o_ref[kk, e]), (e, kk)


def test_fresh_maps_first_record_names_the_scenario_played():
    from ship_sim_gym_b200 import BatchedShipEnv
    n, K = 2048, 300
    env = BatchedShipEnv(n, scenario_source="device", n_scenarios=256, seed=4, fresh_maps=True)
    env.enable_episode_log(n * 16)
    env.reset()
    env.rollout(None, K=20)
    env.episodes()
    scen0 = env.get_state()["ints"][:, 3].copy()
    env.rollout(None, K=K)
    ep = _np(env.episodes())
    first = _first_records(ep)
    assert len(first) > n // 2
    for e, j in first.items():
        assert ep["scenario"][j] == scen0[e]


def test_shards_concatenate_to_the_whole_batch():
    from ship_sim_gym_b200 import BatchedShipEnv
    n, K = 2048, 200
    whole = BatchedShipEnv(n, seed=6, n_scenarios=64)
    shards = [BatchedShipEnv(n // 2, seed=6, n_scenarios=64, env_id_offset=o) for o in (0, n // 2)]
    eps = []
    for e in [whole] + shards:
        e.enable_episode_log(n * K // 8)
        e.reset()
        e.rollout(None, K=K)
        eps.append(_np(e.episodes()))
    cat = {k: np.concatenate([eps[1][k], eps[2][k]]) for k in eps[0]}
    order = np.lexsort((cat["global_env"], cat["k"]))
    for k in eps[0]:
        if k != "env":
            assert np.array_equal(eps[0][k], cat[k][order]), k


def test_binding_needs_auto_reset():
    from ship_sim_gym_b200 import _abi
    env = make_env(knobs(), 64, fp32_bank(8, 600, 600), auto_reset=False)
    rows = torch.zeros(64, 32, device="cuda")
    meta = torch.zeros(64, 8, dtype=torch.int32, device="cuda")
    cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
    assert env.L.shipsim_episode_log_bind(env._h, rows.data_ptr(), meta.data_ptr(), 64, cnt.data_ptr()) == -3
    assert b"auto_reset" in env.L.shipsim_last_error()
    with pytest.raises(_abi.ShipsimError):
        env.enable_episode_log()


def test_overflow_writes_nothing_past_capacity_and_counts_on():
    from ship_sim_gym_b200 import _abi
    n, K, cap = 512, 100, 37
    env = make_env(knobs(max_steps=20), n, fp32_bank(16, 600, 600))
    rows = torch.full((cap + 5, 32), 7.0, device="cuda")
    meta = torch.full((cap + 5, 8), 7, dtype=torch.int32, device="cuda")
    cnt = torch.zeros(1, dtype=torch.int32, device="cuda")
    _abi.check(env.L.shipsim_episode_log_bind(env._h, rows.data_ptr(), meta.data_ptr(), cap, cnt.data_ptr()))
    env.reset()
    _, _, done = env.rollout(None, K=K)
    torch.cuda.synchronize()
    assert int(cnt.item()) == int(done.sum().item()) > cap
    assert bool((rows[cap:] == 7.0).all()) and bool((meta[cap:] == 7).all())
    assert bool((meta[:cap, _abi.EP_LENGTH] >= 1).all())
    env.enable_episode_log(cap)
    env.rollout(None, K=K)
    with pytest.raises(_abi.ShipsimError, match="records lost"):
        env.episodes()


def test_vec_env_episode_info():
    from ship_sim_gym_b200 import BatchedShipEnv
    from ship_sim_gym_b200.adapters import ShipVecEnv
    n, steps = 256, 120
    _, EC = config_classes(knobs(max_steps=50))
    vec = ShipVecEnv(n, episode_info=True, seed=8, n_scenarios=32, env_config=EC)
    plain = ShipVecEnv(n, seed=8, n_scenarios=32, env_config=EC)
    ref = BatchedShipEnv(n, seed=8, n_scenarios=32, auto_reset=False, env_config=EC)
    vec.reset(), plain.reset(), ref.reset()
    rng = np.random.RandomState(1)
    acc = np.zeros(n, dtype=np.float32)
    ended = np.zeros(n, dtype=bool)
    n_info = 0
    for t in range(steps):
        a = rng.randint(0, 3, n)
        obs, rew, done, infos = vec.step(a)
        _, _, _, pinfo = plain.step(a)
        assert all(i == {} for i in pinfo)
        ro = ref.step_np(a)[0].copy()
        acc = (acc + rew).astype(np.float32)
        for e in range(n):
            if done[e]:
                ep = infos[e]["episode"]
                assert ep["r"] == acc[e] and 1 <= ep["l"] <= 50
                assert ep["l"] == 50 or not infos[e]["TimeLimit.truncated"]
                if not ended[e]:
                    assert np.array_equal(infos[e]["terminal_observation"], ro[e])
                ended[e] = True
                acc[e] = 0
                n_info += 1
            else:
                assert infos[e] == {}
    assert n_info > n


@pytest.mark.parametrize("use_graph", [False, True])
def test_rollout_collector_episode_log(use_graph):
    from ship_sim_gym_b200 import BatchedShipEnv
    from ship_sim_gym_b200.rollout import MlpPolicy, RolloutCollector
    torch.manual_seed(0)
    n, T = 1024, 64
    env = BatchedShipEnv(n, seed=3, n_scenarios=64, env_config=config_classes(knobs(max_steps=30))[1])
    col = RolloutCollector(env, MlpPolicy().cuda(), T=T, use_graph=use_graph, episode_log=True)
    ret = torch.zeros(n, dtype=torch.float32, device="cuda")
    length = torch.zeros(n, dtype=torch.int64, device="cuda")
    for it in range(3):
        col.collect()
        ep = col.episodes()
        kk, ee = torch.nonzero(col.dones, as_tuple=True)
        order = torch.argsort(kk * n + ee)
        assert torch.equal(ep["t"], kk[order]) and torch.equal(ep["env"], ee[order]) and bool((ep["k"] == 0).all())
        # return / length from the rollout's rewards, carried across rollouts
        for t in range(T):
            ret = ret + col.rewards[t]
            length += 1
            d = col.dones[t].bool()
            sel = ep["t"] == t
            assert torch.equal(ep["return"][sel], ret[ep["env"][sel]]) and torch.equal(ep["length"][sel], length[ep["env"][sel]])
            ret = torch.where(d, torch.zeros_like(ret), ret)
            length = torch.where(d, torch.zeros_like(length), length)
        if it == 0:
            continue
        assert len(ep["env"]) > n // 2
