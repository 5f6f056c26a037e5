"""-m gpu: weighted scenario picks (shipsim_scenario_weights, BatchedShipEnv.set_scenario_weights) and LevelReplay.

Equal weights reproduce the uniform picks bit for bit; zero-weight maps are never played, by the initial reset nor by the
auto-resets of either kernel; pick frequencies follow the weights; the oracle makes the same picks; the picks do not depend
on the sharding; a captured rollout graph plays new weights on its next replay; LevelReplay.update() makes no host
synchronisation; weights and fresh maps exclude each other, and a new bank drops the weights."""
import numpy as np
import pytest
from scipy import stats

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from helpers import assert_same, fp32_bank, knobs, make_env, make_oracle, run  # noqa: E402
import parity  # noqa: E402
from weighted_picks import oracle_step_weighted  # noqa: E402

N_SCEN = 48


def skewed(n, seed=0):
    """Half the bank at weight 0, the other half at 1 .. 20."""
    rng = np.random.RandomState(seed)
    w = rng.randint(1, 21, n).astype(np.float64)
    w[rng.permutation(n)[: n // 2]] = 0.0
    return w


def weighted_env(k, n, bank, w, **kw):
    env = make_env(k, n, bank, **kw)
    if w is not None:
        env.set_scenario_weights(w)
    return env


@pytest.mark.parametrize("sif", [16, 1], ids=["window", "serial"])
def test_equal_weights_are_bit_identical_to_weights_off(sif):
    k = knobs(max_steps=12)                                   # short episodes: many auto-resets
    bank = fp32_bank(N_SCEN, 600, 600, seed=13)
    n, K = 4096, 64
    ref = run(weighted_env(k, n, bank, None, seed=5, steps_in_flight=sif), None, K)
    got = run(weighted_env(k, n, bank, np.full(N_SCEN, 0.3), seed=5, steps_in_flight=sif), None, K)
    assert got[3]["steps_in_flight"] == sif
    assert_same(got, ref, "equal weights, steps_in_flight=%d" % sif)
    assert ref[2]["episodes"] > n


def test_window_and_serial_kernels_agree_under_weights():
    k = knobs(max_steps=12)
    bank = fp32_bank(N_SCEN, 600, 600, seed=13)
    n, K, w = 4096, 64, skewed(N_SCEN)
    ref = run(weighted_env(k, n, bank, w, seed=5, steps_in_flight=1), None, K)
    got = run(weighted_env(k, n, bank, w, seed=5, steps_in_flight=16), None, K)
    assert_same(got, ref, "window vs serial, skewed weights")
    uniform = run(weighted_env(k, n, bank, None, seed=5, steps_in_flight=16), None, K)
    assert not np.array_equal(uniform[1]["ints"][:, 3], got[1]["ints"][:, 3])      # the weights did change the picks


@pytest.mark.parametrize("sif", [16, 1], ids=["window", "serial"])
def test_zero_weight_maps_are_never_played_and_frequencies_follow_the_weights(sif):
    k = knobs(max_steps=10)
    bank = fp32_bank(N_SCEN, 600, 600, seed=13)
    n, w = 65536, skewed(N_SCEN, seed=1)
    env = weighted_env(k, n, bank, w, seed=7, steps_in_flight=sif)
    env.enable_episode_log(n * 8)
    env.reset()
    first = env.get_state()["ints"][:, 3]                      # the initial reset's picks
    assert (w[first] > 0).all()
    q = env._pick_w.cpu().numpy().astype(np.float64)
    counts = np.bincount(first, minlength=N_SCEN)
    chi2 = stats.chisquare(counts[q > 0], n * q[q > 0] / q.sum())
    assert chi2.pvalue > 1e-4, chi2
    env.rollout(None, K=32)
    ep = env.episodes()
    assert len(ep["scenario"]) > n
    played = ep["scenario"].cpu().numpy()
    assert (w[played] > 0).all() and (w[env.get_state()["ints"][:, 3]] > 0).all()
    assert env.launch_info()["steps_in_flight"] == sif


def test_oracle_parity_of_auto_reset_rollouts_under_weights():
    k = knobs(max_steps=10)
    bank = fp32_bank(64, 600, 600, seed=5)
    n, K = 4096 + 3, 40
    env = weighted_env(k, n, bank, skewed(64, seed=2), auto_reset=True, seed=11, steps_in_flight=8)
    q = env._pick_w.cpu().numpy().astype(np.uint32)
    orc = make_oracle(k, n, bank, auto_reset=False, seed=11)          # auto-resets by oracle_step_weighted
    env.reset()
    ints0 = env.get_state()["ints"]
    assert (q[ints0[:, 3]] > 0).all()
    orc.reset(scen=ints0[:, 3])                                        # the initial reset's (weighted) picks
    assert np.array_equal(orc.ints, ints0)
    rng = np.random.RandomState(21)
    acts = rng.choice([0, 0, 1, 2], size=(K, n)).astype(np.int32)
    obs, rew, done = [t.cpu().numpy() for t in env.rollout(torch.tensor(acts, device=env.device))]
    ref = oracle_step_weighted(orc, acts, q)
    rep = parity.compare_steps(ref, obs, rew, done, margin_thr=parity.MARGIN_THR, label="weighted picks")
    assert rep["grazing_frac"] < parity.MAX_EXCLUDED and rep["excluded_frac"] < parity.MAX_EXCLUDED_CUMULATIVE, rep
    assert done.sum() > n
    scen = env.get_state()["ints"][:, 3]
    assert (q[scen] > 0).all() and np.mean(scen == orc.ints[:, 3]) > 0.99


def test_sharding_invariance_under_weights():
    from ship_sim_gym_b200 import BatchedShipEnv, ScenarioBank
    n, K, m = 1 << 18, 32, 4096
    bank = ScenarioBank.generate(256, (600, 600), seed=3)
    w = skewed(256, seed=3)
    big = BatchedShipEnv(n, bank=bank, seed=9, validate_actions=False, steps_in_flight=1)
    big.set_scenario_weights(w)
    big.reset()
    obs, rew, done = big.rollout(None, K=K)
    for off in (0, 37 * 1024, n - m):
        small = BatchedShipEnv(m, bank=bank, seed=9, env_id_offset=off, validate_actions=False, steps_in_flight=16)
        small.set_scenario_weights(torch.tensor(w, device="cuda"))
        small.reset()
        o, r, d = small.rollout(None, K=K)
        assert torch.equal(o, obs[:, off:off + m]) and torch.equal(r, rew[:, off:off + m]) and torch.equal(d, done[:, off:off + m])
        small.close()
    assert (w[big.get_state()["ints"][:, 3]] > 0).all() and int(done.sum()) > n // 10


def test_captured_rollout_graph_plays_new_weights_and_level_replay_makes_no_host_sync():
    from ship_sim_gym_b200 import LevelReplay
    from ship_sim_gym_b200.rollout import MlpPolicy, RolloutCollector
    torch.manual_seed(0)
    k = knobs(max_steps=8)                                    # every env resets during a 32-step rollout
    bank = fp32_bank(N_SCEN, 600, 600, seed=13)
    n, T = 2048, 32
    wa = np.zeros(N_SCEN); wa[: N_SCEN // 2] = 1.0
    wb = np.zeros(N_SCEN); wb[N_SCEN // 2:] = np.arange(1, N_SCEN // 2 + 1)
    env = weighted_env(k, n, bank, wa, seed=3)
    twin = weighted_env(k, n, bank, wb, seed=3)
    twin.reset()
    col = RolloutCollector(env, MlpPolicy().cuda(), T=T, episode_log=True)
    col.collect()                                             # captures the graph
    epoch, graph = env.params_epoch, col._graph
    assert graph is not None and (wa[env.get_state()["ints"][:, 3]] > 0).all()
    env.set_scenario_weights(wb)
    assert env.params_epoch == epoch                          # changing weights keeps the graph
    s0 = env.state.clone()
    col.collect()
    assert col._graph is graph
    assert (wb[env.get_state()["ints"][:, 3]] > 0).all()       # the replay picked from the new support
    twin.state.copy_(s0)                                      # the same rollout, eagerly, from the same state
    for t in range(T):
        o, r, d = twin.rollout(col.actions[t:t + 1])
        assert torch.equal(o[0], col.obs[t + 1]) and torch.equal(r[0], col.rewards[t]) and torch.equal(d[0], col.dones[t]), t
    replay = LevelReplay(env)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for _ in range(3):
            col.collect()
            p = replay.update()
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert col._graph is graph and env.params_epoch == epoch
    assert replay.table[:, 0].sum().item() > 3 * n and abs(p.sum().item() - 1.0) < 1e-9
    assert bool((env._pick_w > 0).all())                      # PLR's distribution keeps every map in play
    env.set_scenario_weights(None)
    assert env.params_epoch == epoch + 1


def test_errors_fresh_maps_length_and_bank_reload():
    from ship_sim_gym_b200 import BatchedShipEnv, _abi
    env = BatchedShipEnv(256, seed=1, scenario_source="device", n_scenarios=64)
    env.set_scenario_weights(np.ones(64))
    with pytest.raises(_abi.ShipsimError):
        env.fresh_maps(True)
    env.set_scenario_weights(None)
    env.fresh_maps(True)
    with pytest.raises(_abi.ShipsimError):
        env.set_scenario_weights(np.ones(64))
    env.fresh_maps(False)
    for bad in (np.ones(63), torch.ones(65, device="cuda"), np.zeros(64), [float("nan")] * 64):
        with pytest.raises(ValueError):
            env.set_scenario_weights(bad)
    k = knobs()
    bank = fp32_bank(N_SCEN, 600, 600, seed=13)
    e = weighted_env(k, 4096, bank, np.eye(N_SCEN)[5], seed=2)
    e0 = e.params_epoch
    e.reset()
    assert (e.get_state()["ints"][:, 3] == 5).all()
    e.load_scenarios(e.bank)                                  # a new bank drops the weights (and resets the batch)
    assert e._pick_w is None and e.params_epoch == e0 + 1
    assert len(np.unique(e.get_state()["ints"][:, 3])) > N_SCEN // 2
