"""-m gpu: level scores (shipsim_gae_scored, RolloutCollector(level_scores=True), LevelReplay's value-loss scores).

The map the collector attributes to every step is the map the env played at that step, read from the state of an eager
twin before each step, on the kernel path and on the generic-policy path; advantages and returns of the scored GAE are
bit-identical to shipsim_gae's; the per-map sums match the torch statement of the rule and a per-step numpy fold; a short
log capacity sends the steps of lost records to the unattributed row; a captured rollout graph keeps all of this right
over its replays, and a LevelReplay loop on the value-loss score makes no host synchronisation."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from helpers import fp32_bank, knobs, make_env  # noqa: E402

N_SCEN = 48


class GenericPolicy(torch.nn.Module):
    """An MlpPolicy the collector does not recognise: it takes the generic per-step torch path."""

    def __init__(self):
        super().__init__()
        from ship_sim_gym_b200.rollout import MlpPolicy
        self.inner = MlpPolicy()

    def forward(self, obs):
        return self.inner(obs)


def envs(n, seed=3, **kw):
    k = knobs(max_steps=8)                                    # every env resets several times in a rollout
    bank = fp32_bank(N_SCEN, 600, 600, seed=13)
    return make_env(k, n, bank, seed=seed, **kw), make_env(k, n, bank, seed=seed, **kw)


def state_scenario(env):
    return env.state[4, :, 2].view(torch.int32)


def numpy_fold(adv, scen, n_scen):
    """Per-step fold of the scores: one row per map, the last for steps of no known map."""
    adv = adv.double().cpu().numpy().ravel()
    s = scen.cpu().numpy().ravel().astype(np.int64)
    row = np.where((s >= 0) & (s < n_scen), s, n_scen)
    out = np.zeros((n_scen + 1, 3))
    np.add.at(out, row, np.stack([np.ones_like(adv), np.maximum(adv, 0.0), np.abs(adv)], 1))
    return out


def torch_scores(col):
    from ship_sim_gym_b200.rollout import score_levels
    env, log = col.env, col.env.episode_log
    return score_levels(col.adv, col.dones, log.meta, log.count, state_scenario(env), col._call0, env.n_scenarios)


def assert_close(a, b, what):
    a, b = np.asarray(a), np.asarray(b)
    assert np.allclose(a, b, rtol=1e-9, atol=1e-9 * max(1.0, float(np.abs(b).max()))), (what, np.abs(a - b).max())


def gae_plain(env, col):
    """shipsim_gae over the collector's own rewards, values and dones, into fresh buffers."""
    from ship_sim_gym_b200 import _abi
    adv, ret = torch.empty_like(col.adv), torch.empty_like(col.returns)
    _abi.check(env.L.shipsim_gae(col.rewards.data_ptr(), col.values.data_ptr(), col.dones.data_ptr(), col.T, env.num_envs, float(col.gamma),
                                 float(col.lam), adv.data_ptr(), ret.data_ptr(), env._stream()))
    return adv, ret


@pytest.mark.parametrize("path", ["kernel", "generic"])
def test_every_step_is_attributed_to_the_map_it_played(path):
    from ship_sim_gym_b200.rollout import MlpPolicy, RolloutCollector
    torch.manual_seed(0)
    n, T = 2048, 32
    env, twin = envs(n)
    policy = (MlpPolicy() if path == "kernel" else GenericPolicy()).cuda()
    col = RolloutCollector(env, policy, T=T, level_scores=True)
    assert col._kernel == (path == "kernel") and col.episode_log
    twin.reset()
    twin.state.copy_(env.state)
    col.collect()                                             # the first call runs the rollout (then captures it)
    played = torch.empty(T, n, dtype=torch.int32, device="cuda")
    for t in range(T):
        played[t] = state_scenario(twin)                      # the map step t plays
        o, r, d = twin.rollout(col.actions[t:t + 1])
        assert torch.equal(d[0], col.dones[t]) and torch.equal(r[0], col.rewards[t]), t
    assert int(col.dones.sum()) > 2 * n                       # several episodes per env
    assert torch.equal(col.scenarios, played)
    n_scen = env.n_scenarios
    fold = numpy_fold(col.adv, played, n_scen)
    assert fold[n_scen].sum() == 0 and col.level_scores[n_scen].abs().sum().item() == 0     # no record lost
    assert_close(col.level_scores.cpu().numpy(), fold, "scores vs numpy fold")
    scen_t, scores_t = torch_scores(col)
    assert torch.equal(scen_t, played)
    assert_close(col.level_scores.cpu().numpy(), scores_t.cpu().numpy(), "scores vs torch")
    adv, ret = gae_plain(env, col)
    if path == "kernel":                                      # the scored GAE computes what shipsim_gae computes, bit for bit
        assert torch.equal(adv.view(torch.int32), col.adv.view(torch.int32)) and torch.equal(ret.view(torch.int32), col.returns.view(torch.int32))


def test_scored_gae_is_bit_identical_to_gae_on_dense_synthetic_dones():
    from ship_sim_gym_b200 import _abi
    n, T = 3001, 17
    env, _ = envs(n)
    env.enable_episode_log(T * n)
    env.reset()
    g = torch.Generator(device="cuda").manual_seed(5)
    rew = torch.randn(T, n, device="cuda", generator=g)
    val = torch.randn(T + 1, n, device="cuda", generator=g)
    for p in (0.0, 0.4, 1.0):
        done = (torch.rand(T, n, device="cuda", generator=g) < p).to(torch.uint8)
        adv0, ret0, adv1, ret1 = (torch.full((T, n), float("nan"), device="cuda") for _ in range(4))
        scen = torch.zeros(T, n, dtype=torch.int32, device="cuda")
        scores = torch.zeros(env.n_scenarios + 1, 3, dtype=torch.float64, device="cuda")
        _abi.check(env.L.shipsim_gae(rew.data_ptr(), val.data_ptr(), done.data_ptr(), T, n, 0.99, 0.95, adv0.data_ptr(), ret0.data_ptr(),
                                     env._stream()))
        _abi.check(env.L.shipsim_gae_scored(env._h, rew.data_ptr(), val.data_ptr(), done.data_ptr(), T, 0.99, 0.95, env._calls, 1,
                                            adv1.data_ptr(), ret1.data_ptr(), scen.data_ptr(), scores.data_ptr(), env._stream()))
        assert torch.equal(adv0.view(torch.int32), adv1.view(torch.int32)) and torch.equal(ret0.view(torch.int32), ret1.view(torch.int32)), p
        # no records: the steps up to an env's last done have no known map
        now = state_scenario(env)
        last_done = torch.where(done.bool(), torch.arange(T, device="cuda")[:, None], torch.full_like(done, -1, dtype=torch.int64)).amax(0)
        want = torch.where(torch.arange(T, device="cuda")[:, None] > last_done, now, torch.full_like(now, -1))
        assert torch.equal(scen, want), p
        assert_close(scores.cpu().numpy(), numpy_fold(adv0, want, env.n_scenarios), "scores, p = %g" % p)


def test_short_log_capacity_sends_the_lost_steps_to_the_unattributed_row():
    from ship_sim_gym_b200.rollout import MlpPolicy, RolloutCollector
    torch.manual_seed(1)
    n, T, cap = 2048, 32, 1500
    env, _ = envs(n)
    col = RolloutCollector(env, MlpPolicy().cuda(), T=T, level_scores=True, use_graph=False)
    env.enable_episode_log(cap)                               # far fewer records than episodes: most are dropped
    col.collect()
    count = int(env.episode_log.count.item())
    assert count > cap
    n_scen = env.n_scenarios
    scen_t, scores_t = torch_scores(col)
    assert torch.equal(col.scenarios, scen_t)
    lost = col.scenarios == -1
    assert int(lost.sum()) > 0
    fold = numpy_fold(col.adv, col.scenarios, n_scen)
    assert fold[n_scen, 0] == int(lost.sum())
    assert_close(col.level_scores.cpu().numpy(), fold, "scores vs numpy fold")
    assert_close(col.level_scores.cpu().numpy(), scores_t.cpu().numpy(), "scores vs torch")
    # the steps after each env's last done never need a record
    last_done = torch.where(col.dones.bool(), torch.arange(T, device="cuda")[:, None], torch.full_like(col.dones, -1, dtype=torch.int64)).amax(0)
    after = torch.arange(T, device="cuda")[:, None] > last_done
    assert torch.equal(col.scenarios[after], state_scenario(env).expand(T, n)[after])


def test_captured_graph_replays_and_a_value_loss_level_replay_loop_without_host_sync():
    from ship_sim_gym_b200 import LevelReplay
    from ship_sim_gym_b200.rollout import MlpPolicy, RolloutCollector
    torch.manual_seed(2)
    n, T = 2048, 32
    env, _ = envs(n)
    env.set_scenario_weights(np.ones(N_SCEN))                 # weights on before the capture: new weights keep the graph
    col = RolloutCollector(env, MlpPolicy().cuda(), T=T, level_scores=True)
    col.collect()
    graph, epoch = col._graph, env.params_epoch
    assert graph is not None
    n_scen = env.n_scenarios
    for _ in range(3):
        col.collect()
        assert col._graph is graph
        scen_t, scores_t = torch_scores(col)
        assert torch.equal(col.scenarios, scen_t) and int((col.scenarios < 0).sum()) == 0
        assert_close(col.level_scores.cpu().numpy(), scores_t.cpu().numpy(), "replay scores vs torch")
        assert col.level_scores[:, 0].sum().item() == T * n   # zeroed at the start of each rollout
        adv, ret = gae_plain(env, col)
        assert torch.equal(adv, col.adv) and torch.equal(ret, col.returns)
    replay = LevelReplay(env, score="positive_value_loss")
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for _ in range(3):
            col.collect()
            p = replay.update(col.level_scores)
    finally:
        torch.cuda.set_sync_debug_mode(0)
    assert col._graph is graph and env.params_epoch == epoch
    assert abs(p.sum().item() - 1.0) < 1e-9 and bool(replay.scored.all())
    assert bool((env._pick_w > 0).all())
    steps, pos = col.level_scores[:n_scen, 0], col.level_scores[:n_scen, 1]
    assert bool((pos <= col.level_scores[:n_scen, 2]).all()) and steps.sum().item() == T * n


def test_errors_without_episode_log_or_auto_reset():
    from ship_sim_gym_b200 import _abi
    n, T = 256, 4
    f = dict(device="cuda")
    rew, val, adv, ret = torch.zeros(T, n, **f), torch.zeros(T + 1, n, **f), torch.zeros(T, n, **f), torch.zeros(T, n, **f)
    done = torch.zeros(T, n, dtype=torch.uint8, **f)
    scen = torch.zeros(T, n, dtype=torch.int32, **f)
    scores = torch.zeros(N_SCEN + 1, 3, dtype=torch.float64, **f)

    def call(env):
        return env.L.shipsim_gae_scored(env._h, rew.data_ptr(), val.data_ptr(), done.data_ptr(), T, 0.99, 0.95, 0, 1, adv.data_ptr(),
                                        ret.data_ptr(), scen.data_ptr(), scores.data_ptr(), env._stream())
    env, _ = envs(n)
    env.reset()
    assert call(env) == -3 and b"episode log" in env.L.shipsim_last_error()
    env.enable_episode_log(n)
    assert call(env) == 0
    plain, _ = envs(n, auto_reset=False)
    plain.reset()
    assert call(plain) == -3 and b"auto_reset" in plain.L.shipsim_last_error()
    assert env.L.shipsim_gae_scored(None, rew.data_ptr(), val.data_ptr(), done.data_ptr(), T, 0.99, 0.95, 0, 1, adv.data_ptr(),
                                    ret.data_ptr(), scen.data_ptr(), scores.data_ptr(), None) == -1
