"""-m gpu: the vector-env adapters for the reference's callers (stable-baselines VecEnv, RLlib VectorEnv), the
single-env facade driven like train/random.py, and the on-device policy rollout (CUDA-graph replay)."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import oracle  # noqa: E402
from helpers import fp32_bank  # noqa: E402
import parity  # noqa: E402
from ship_sim_gym_b200 import ScenarioBank  # noqa: E402


def test_vec_env_protocol_and_auto_reset_obs():
    """SubprocVecEnv worker semantics (train/stable_baselines/ppo.py:122-123): the obs returned on a done step is the
    reset obs; reward / done are those of the terminal step.  Checked against the oracle with auto-reset."""
    from ship_sim_gym_b200.adapters import ShipVecEnv
    n, T = 256, 60
    bank = ScenarioBank(bounds=(600, 600), **fp32_bank(16, 600, 600, seed=4))
    venv = ShipVecEnv(n, bank=bank, seed=9)
    orc = oracle.OracleEnv(n, bank.as_dict(), auto_reset=True, seed=9)
    assert venv.num_envs == n and venv.action_space.n == 3 and venv.observation_space.shape == (32,)
    obs = venv.reset()
    ref0 = orc.reset()
    assert isinstance(obs, np.ndarray) and obs.shape == (n, 32) and obs.dtype == np.float32
    np.testing.assert_allclose(obs, ref0, rtol=1e-6, atol=1e-4)
    rng = np.random.RandomState(0)
    acts = rng.choice([0, 0, 0, 1, 2], size=(T, n))
    got_o, got_r, got_d = [], [], []
    for t in range(T):
        venv.step_async(acts[t])
        o, r, d, infos = venv.step_wait()
        assert len(infos) == n and infos[0] == {}
        got_o.append(o); got_r.append(r); got_d.append(d)
    ref = orc.step(acts.astype(np.int32))
    rep = parity.compare_steps(ref, np.stack(got_o), np.stack(got_r), np.stack(got_d), margin_thr=parity.MARGIN_THR, label="vecenv")
    assert rep["grazing_frac"] < parity.MAX_EXCLUDED and rep["excluded_frac"] < parity.MAX_EXCLUDED_CUMULATIVE, rep
    d = np.stack(got_d)
    assert d.any(), "no episode ended: the auto-reset path was not exercised"
    k, e = np.argwhere(d)[0]
    assert (np.stack(got_o)[k, e, :16] == -1).all()              # reset obs: [-1 x 16 | reset frame] (ship_env.py:180-184)
    with pytest.raises(RuntimeError):
        venv.step_wait()
    venv.close()


def test_vector_env_protocol_reset_at():
    from ship_sim_gym_b200.adapters import ShipVectorEnv
    n = 8
    env = ShipVectorEnv(n, bank=ScenarioBank(bounds=(600, 600), **fp32_bank(16, 600, 600, seed=4)), seed=2)
    obs = env.vector_reset()
    assert len(obs) == n and obs[0].shape == (32,) and (obs[0][:16] == -1).all()
    done_seen = False
    for t in range(400):
        o, r, d, info = env.vector_step([0] * n)                  # full ahead: runs off the top of the map
        assert len(o) == len(r) == len(d) == len(info) == n and isinstance(r[0], float) and isinstance(d[0], bool)
        for i in range(n):
            if d[i]:
                done_seen = True
                o0 = env.reset_at(i)                              # RLlib resets sub-envs itself
                assert (o0[:16] == -1).all() and o0[16] == 300 and o0[17] == 25
        if done_seen:
            break
    assert done_seen
    o, r, d, _ = env.vector_step([1] * n)
    assert not any(d)
    env.close()


def test_random_agent_script_shape():
    """train/random.py:9-26 with the drop-in import: construct, reset, random actions, reset on done."""
    from ship_sim_gym_b200 import ShipEnv
    from ship_sim_gym_b200.config import EnvConfig, GameConfig

    class GC(GameConfig):
        SPEED = 30              # big steps so that episodes end quickly
    env = ShipEnv(GC, EnvConfig, bank=ScenarioBank(bounds=(600, 600), **fp32_bank(16, 600, 600, seed=4)), seed=0)
    env.seed(0)
    env.reset()
    episodes = 0
    for _ in range(300):
        ret = env.step(env.action_space.sample())
        assert len(ret) == 4 and ret[0].shape == (32,) and ret[3] == {}
        if ret[2]:
            episodes += 1
            assert env.step_count > 0
            obs = env.reset()
            assert env.step_count == 0 and env.cumulative_reward == 0 and (obs[:16] == -1).all()
    assert episodes >= 1 and env.episodes_count >= 1
    env.close()


def test_policy_rollout_graph_replay_matches_eager():
    """BASELINE configs[4]: MLP policy + envs on one GPU, whole rollout in a CUDA graph.  With the sampler's RNG
    reseeded the same way, a replayed graph and the eager loop produce the same rollout."""
    from ship_sim_gym_b200 import BatchedShipEnv
    from ship_sim_gym_b200.rollout import MlpPolicy, RolloutCollector
    n, T = 2048, 16
    bank = ScenarioBank(bounds=(600, 600), **fp32_bank(32, 600, 600, seed=4))
    torch.manual_seed(0)
    policy = MlpPolicy().cuda()
    out = []
    for use_graph in (False, True):
        env = BatchedShipEnv(n, bank=bank, seed=1)
        col = RolloutCollector(env, policy, T=T, use_graph=use_graph)
        col.collect()                                             # graph mode: warm-up + capture
        launches0 = env.launch_info()["launches"]
        col.collect()
        torch.cuda.synchronize()
        out.append((col.rewards.clone(), col.dones.clone(), col.obs.clone(), env.launch_info()["launches"] - launches0))
        assert col.actions.min() >= 0 and col.actions.max() <= 2
        assert torch.isfinite(col.adv).all() and torch.isfinite(col.returns).all()
        env.close()
    # eager: T host-side calls into shipsim_step; graph replay: none (the launches are inside the graph)
    assert out[0][3] == T and out[1][3] == 0
    # same physics either way: every transition obeys the env's invariants
    for rew, done, obs, _ in out:
        r = rew.cpu().numpy()
        assert (np.isclose(r, 1.0) | np.isclose(r, -1.0) | np.isclose(r, -0.01)).all()
        first = obs[1:, :, :16].cpu().numpy()
        d = done.cpu().numpy().astype(bool)
        assert ((first == -1).all(-1) == d).all()                 # the older frame is all -1 exactly on reset steps


@pytest.mark.parametrize("n", [16384, 1000, 7])
def test_policy_kernel_matches_the_torch_module(n):
    """shipsim_mlp_policy_forward (csrc/shipsim_policy.cu: both MlpPolicy trunks, heads and the Gumbel-max sample in one
    launch; train/stable_baselines/ppo.py:88) against the plain fp32 torch module: logits and values within 2e-5, the same
    action wherever the decision is not a near-tie, ragged batch sizes included."""
    from ship_sim_gym_b200 import BatchedShipEnv
    from ship_sim_gym_b200.rollout import MlpPolicy, RolloutCollector
    torch.manual_seed(n)
    policy = MlpPolicy().cuda()
    for lin in (policy.pi[4], policy.vf[4]):                      # livelier heads than the default init
        lin.weight.data.mul_(4.0)
    env = BatchedShipEnv(n, bank=ScenarioBank(bounds=(600, 600), **fp32_bank(8, 600, 600, seed=4)), seed=1)
    col = RolloutCollector(env, policy, T=2, use_graph=False)
    assert col._kernel
    obs = torch.rand(n, 32, device="cuda") * 600.0
    obs[: n // 4, :16] = -1.0                                     # reset rows look like this
    col.obs[0].copy_(obs)
    col._noise.uniform_().clamp_(1e-10, 1.0).log_().neg_().log_().neg_()
    with torch.no_grad():
        col._refresh_fused()
        col._forward_kernel(0)
        torch.cuda.synchronize()
        logits, v = policy(obs)
    got = col._out[0]
    assert torch.allclose(got[:, :3], logits, atol=2e-5, rtol=1e-5) and torch.allclose(got[:, 3], v, atol=2e-5, rtol=1e-5)
    z = logits + col._noise[0]
    top2 = z.topk(2, dim=-1).values
    clear = (top2[:, 0] - top2[:, 1]) > 1e-3
    assert clear.float().mean() > 0.95
    assert (col.actions[0][clear] == z.argmax(-1)[clear]).all()
    assert col.actions[0].min() >= 0 and col.actions[0].max() <= 2 and len(torch.unique(col.actions[0])) == (3 if n > 100 else len(torch.unique(col.actions[0])))
    # the collector with the kernel: same invariants as the torch path, 2 launches of ours per step
    col.collect()
    torch.cuda.synchronize()
    assert torch.isfinite(col.adv).all() and (col.logp <= 0).all() and col.actions.min() >= 0 and col.actions.max() <= 2
    with torch.no_grad():
        lg, vv = policy(col.obs[1])
    assert torch.allclose(col.values[1], vv, atol=2e-5, rtol=1e-5)
    lp = torch.log_softmax(lg, -1).gather(-1, col.actions[1][:, None]).squeeze(-1)
    assert torch.allclose(col.logp[1], lp, atol=1e-4)
    # advantages / returns of the kernel path (shipsim_gae) against the torch formulation of the same recurrence
    adv_k, ret_k = col.adv.clone(), col.returns.clone()
    col._gae()
    assert torch.allclose(adv_k, col.adv, atol=1e-5, rtol=1e-5) and torch.allclose(ret_k, col.returns, atol=1e-5, rtol=1e-5)
    # ... and with episode ends in the rollout (synthetic: T = 2 is too short for real ones)
    from ship_sim_gym_b200 import _abi
    col.dones.copy_((torch.rand(col.dones.shape, device="cuda") < 0.4).to(torch.uint8))
    col.rewards.normal_()
    col.values.normal_()
    _abi.check(env.L.shipsim_gae(col.rewards.data_ptr(), col.values.data_ptr(), col.dones.data_ptr(), col.T, n, float(col.gamma), float(col.lam),
                                 col.adv.data_ptr(), col.returns.data_ptr(), env._stream()))
    adv_k, ret_k = col.adv.clone(), col.returns.clone()
    col._gae()
    assert col.dones.sum() > 0 or n < 20
    assert torch.allclose(adv_k, col.adv, atol=1e-5, rtol=1e-5) and torch.allclose(ret_k, col.returns, atol=1e-5, rtol=1e-5)
    env.close()


def test_curriculum_driver_on_a_live_batch():
    """EnvConfig.MAX_STEPS as a curriculum knob: the cap changes on the live handle (shipsim_set_max_steps) and the
    time-out statistics follow it."""
    from ship_sim_gym_b200 import BatchedShipEnv, Curriculum, CurriculumDriver
    n = 1024
    env = BatchedShipEnv(n, bank=ScenarioBank(bounds=(600, 600), **fp32_bank(16, 600, 600, seed=4)), seed=0)
    cur = Curriculum([5, 12], [-10.0], repeat_condition=0)            # any mean return > -10 passes
    drv = CurriculumDriver(env, cur, knob="max_steps", min_episodes=n)
    env.reset()
    idle = torch.ones(8, n, dtype=torch.int32, device=env.device)     # rudder only: nobody moves, episodes only time out
    obs, rew, done = env.rollout(idle)
    assert done[4].all() and done.sum() == n                          # MAX_STEPS = 5 (ship_env.py:131)
    s = env.stats()
    assert s["timeout"] == n and s["length_sum"] == 5 * n
    adv, mean = drv.update()
    assert adv and mean == pytest.approx(-0.05) and int(cur) == 12
    obs, rew, done = env.rollout(torch.ones(15, n, dtype=torch.int32, device=env.device))
    # 3 steps of the running episode were done under the old cap; it now ends at step count 12
    assert done[8].all() and done.sum() == n
    with pytest.raises(ValueError):
        env.set_max_steps(0)
    env.close()


def test_rgb_array_render_of_one_env():
    """`rgb_array` rendering of a selected env (SURVEY §8 f4; ShipGame.render / get_screen, game.py:133-138,197-229)."""
    import numpy as np
    from ship_sim_gym_b200 import BatchedShipEnv, ShipEnv
    from ship_sim_gym_b200.config import EnvConfig, GameConfig
    env = BatchedShipEnv(64, seed=1)
    obs = env.reset()
    img = env.render("rgb_array", env_index=5).cpu().numpy()
    assert img.shape == (600, 600, 3) and img.dtype == np.uint8
    assert env.get_screen(5).shape == (600, 600, 3)
    assert env.render() is None                                  # `human` mode only prints in the reference
    # the yellow marker sits on the spawn point (300, 25): screen y points down
    assert tuple(img[600 - 25, 300]) == (255, 255, 0)
    # water far from everything is the reference's background colour
    st = env.get_state()
    assert tuple(img[600 - 300, 300]) in ((0, 0, 200), (0, 200, 0))
    # each remaining goal shows as a green disc
    gx, gy = st["goals"][5, 2]
    assert tuple(img[int(round(600 - gy)) - 1, int(gx)]) == (0, 200, 0)
    # the left bank hugs x = 0 somewhere along the river, the hull is white just above the marker
    assert (img[:, 2] == np.array([110, 110, 110])).all(-1).any()
    assert tuple(img[600 - 25 - 20, 300 + 10]) == (255, 255, 255)
    # after some steps the picture follows the state
    import torch
    env.rollout(torch.zeros(40, 64, dtype=torch.int32, device=env.device))
    st = env.get_state()
    img2 = env.render("rgb_array", env_index=5, size=(300, 300)).cpu().numpy()
    x, y = st["pose"][5, :2]
    if 0 < x < 600 and 0 < y < 600:
        assert tuple(img2[min(299, int((600 - y) / 2)), min(299, int(x / 2))]) == (255, 255, 0)
    # the VecEnv surface: one picture per env, and the tiled overview
    from ship_sim_gym_b200.adapters import ShipVecEnv
    venv = ShipVecEnv(num_envs=7, seed=1)
    venv.reset()
    pics = venv.get_images(size=(60, 60))
    assert len(pics) == 7 and pics[0].shape == (60, 60, 3) and pics[0].dtype == np.uint8
    tiled = venv.render("rgb_array", size=(60, 60))
    assert tiled.shape == (3 * 60, 3 * 60, 3) and (tiled[:60, 60:120] == pics[1]).all() and (tiled[120:, 60:] == 0).all()
    assert venv.render() is None
    venv.close()
    single = ShipEnv(GameConfig, EnvConfig)
    single.reset()
    assert single.render("rgb_array").shape == (600, 600, 3)
