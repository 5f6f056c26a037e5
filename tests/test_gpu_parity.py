"""-m gpu: the CUDA path (through the C ABI) against the float64 oracle and the golden fixtures."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import oracle  # noqa: E402
from oracle import cbind  # noqa: E402
from helpers import case_knobs, fp32_bank, knobs, load_trajectories, make_env, make_oracle, pack_bank  # noqa: E402
import parity  # noqa: E402


def _np(*ts):
    return [t.cpu().numpy() for t in ts]


# ---------------------------------------------------------------------------------------------- golden fixtures
EPS = load_trajectories()


@pytest.mark.parametrize("lanes", [1, 2, 4, 8, 16, 32])
def test_golden_trajectories(lanes):
    """Every reference trajectory in tests/golden (real reference Python over the restated Chipmunk), replayed
    as ONE K-step launch per episode."""
    worst = 0.0
    for idx, ep in enumerate(EPS):
        W, H, speed, hist, max_steps = ep["cfg"][:5]
        if hist > 2:
            continue          # assembled by the host layer: covered by test_long_history
        h0, h1 = cbind.convex_hull(ep["raw0"]), cbind.convex_hull(ep["raw1"])
        bank = pack_bank([(h0, h1)], [ep["goals"]])
        k = knobs(W=W, H=H, speed=speed, hist=int(hist), max_steps=int(max_steps))
        env, orc = make_env(k, 1, bank, auto_reset=False, lanes_per_env=lanes), make_oracle(k, 1, bank)
        obs0 = env.reset(scenario=[0])
        orc.reset(scen=[0])
        tol0 = parity.REL_TOL * np.maximum(1, np.abs(ep["obs"][0]))
        assert (np.abs(obs0[0].cpu().numpy() - ep["obs"][0]) <= tol0).all(), "reset obs, episode %d" % idx
        acts = torch.tensor(ep["actions"], dtype=torch.int32, device=env.device)[:, None]
        obs, rew, done = _np(*env.rollout(acts))
        ref = orc.step(ep["actions"][:, None])
        ref_golden = dict(ref)
        ref_golden["obs"] = ep["obs"][1:][:, None, :]
        ref_golden["reward"] = ep["reward"][:, None]
        ref_golden["done"] = ep["done"][:, None]
        rep = parity.compare_steps(ref_golden, obs, rew, done, label="episode %d" % idx, scale=max(W, H))
        worst = max(worst, rep["max_rel_err"])
        env.close()
    assert worst <= 1.0


def test_long_history_host_layer():
    ep = [e for e in EPS if e["cfg"][3] == 3][0]
    W, H, speed, hist, max_steps = ep["cfg"][:5]
    bank = pack_bank([(cbind.convex_hull(ep["raw0"]), cbind.convex_hull(ep["raw1"]))], [ep["goals"]])
    env = make_env(knobs(W=W, H=H, speed=speed, hist=3, max_steps=int(max_steps)), 1, bank, auto_reset=False)
    obs0 = env.reset(scenario=[0])
    assert obs0.shape == (1, 48)
    np.testing.assert_allclose(obs0[0].cpu().numpy(), ep["obs"][0], rtol=1e-4, atol=1e-4)
    for t, a in enumerate(ep["actions"][:40]):
        o, r, d, info = env.step(torch.tensor([a]))
        np.testing.assert_allclose(o[0].cpu().numpy(), ep["obs"][t + 1], rtol=1e-4, atol=1e-3)
        assert float(r[0]) == pytest.approx(ep["reward"][t]) and bool(d[0]) == bool(ep["done"][t])


# ---------------------------------------------------------------------------------------------- injected states
CASES = [
    dict(name="default", W=600, H=600, speed=10),
    dict(name="random_py", W=600, H=600, speed=1),
    dict(name="sb_script", W=1000, H=1000, speed=30),
    dict(name="hard_map", W=1000, H=1000, speed=10, map_N=30, wf=0.9, spread=180),
    dict(name="history1", W=600, H=600, speed=10, hist=1),
]


@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
@pytest.mark.parametrize("adversarial", [False, True])
@pytest.mark.parametrize("lanes", [1, 8, 32])
def test_injected_single_step(case, adversarial, lanes):
    W, H = case["W"], case["H"]
    n = 8192 - 5          # not a multiple of the warp / CTA size: exercises the ragged tail
    k = case_knobs(case)
    bank = fp32_bank(64, W, H, seed=3, map_N=k["map_N"], wf=k["wf"])
    env, orc = make_env(k, n, bank, auto_reset=False, lanes_per_env=lanes), make_oracle(k, n, bank)
    env.reset()
    rng = np.random.RandomState(7 + adversarial)
    st = parity.f32_inputs(*parity.random_states(rng, n, W, H, 64, bank["goals"],
                                                 near=(bank["hull_xy"], bank["hull_n"]) if adversarial else None))
    env.set_state(*st)
    parity.load_oracle_state(orc, *st)
    acts = rng.randint(0, 3, n).astype(np.int32)
    o, r, d, _ = env.step(torch.tensor(acts, device=env.device))
    ref = orc.step(acts[None])
    rep = parity.compare_steps(ref, o.cpu().numpy()[None], r.cpu().numpy()[None], d.cpu().numpy()[None], label=case["name"], scale=max(W, H))
    assert rep["excluded_frac"] < 0.01, rep
    assert rep["max_pose_rel_err"] < 2 * parity.REL_TOL
    # the post-step state itself (velocities are not part of obs)
    got = env.get_state()
    ok = ref["margins"][0, :, :].min(-1) >= 1e-3
    tol = parity.REL_TOL * np.maximum(1, np.abs(orc.pose)) + parity.POSE_ABS * max(W, H)
    assert (np.abs(got["pose"] - orc.pose) <= tol)[ok].all()
    assert (got["ints"][ok][:, :3] == orc.ints[ok][:, :3]).all()
    # flags present in the sample (otherwise the test proves nothing)
    f = ref["flags"][0]
    assert (f & oracle.FLAG_COLLIDING).any() and (f & oracle.FLAG_OOB).any()
    if adversarial:
        assert (orc.lidar[:, :10] >= 0).any()
    env.close()


@pytest.mark.parametrize("case", CASES[:4], ids=[c["name"] for c in CASES[:4]])
@pytest.mark.parametrize("auto_reset", [False, True])
@pytest.mark.parametrize("lanes", [1, 4, 16])
def test_32_step_transitions(case, auto_reset, lanes):
    W, H = case["W"], case["H"]
    n, K = 4096 + 3, 32
    k = case_knobs(case)
    bank = fp32_bank(64, W, H, seed=5, map_N=k["map_N"], wf=k["wf"])
    env = make_env(k, n, bank, auto_reset=auto_reset, seed=11, lanes_per_env=lanes)
    orc = make_oracle(k, n, bank, auto_reset=auto_reset, seed=11)
    env.reset()
    orc.reset()
    rng = np.random.RandomState(21)
    acts = rng.choice([0, 0, 1, 2], size=(K, n)).astype(np.int32)
    obs, rew, done = _np(*env.rollout(torch.tensor(acts, device=env.device)))
    ref = orc.step(acts)
    rep = parity.compare_steps(ref, obs, rew, done, margin_thr=parity.MARGIN_THR, label=case["name"], scale=max(W, H),
                               stop_at_done=not auto_reset)
    assert rep["grazing_frac"] < parity.MAX_EXCLUDED and rep["excluded_frac"] < parity.MAX_EXCLUDED_CUMULATIVE, rep
    assert rep["max_pose_rel_err"] < 2 * parity.REL_TOL
    if auto_reset and case["speed"] >= 10:
        s = env.stats()
        so = orc.stats_dict()
        assert so["episodes"] > 0
        # statistics agree up to the (few) grazing envs
        assert abs(s["episodes"] - so["episodes"]) <= max(3, 0.01 * so["episodes"])
        assert s["episodes"] == float(done.sum())
    env.close()


# ---------------------------------------------------------------------------------------------- properties at scale
def test_k_fusion_and_sharding_invariance():
    """Full-size (65,536 envs) properties: K fused steps == K single launches (bit-exact), and the result
    does not depend on how the envs are sharded (RNG keyed by global env id)."""
    from ship_sim_gym_b200 import BatchedShipEnv, ScenarioBank
    n, K = 65536, 16
    bank = ScenarioBank.generate(128, (600, 600), seed=1)
    acts = torch.randint(0, 3, (K, n), dtype=torch.int32, device="cuda", generator=torch.Generator("cuda").manual_seed(0))
    a = BatchedShipEnv(n, bank=bank, seed=4)
    a.reset()
    oa, ra, da = a.rollout(acts)
    b = BatchedShipEnv(n, bank=bank, seed=4)
    b.reset()
    for k in range(K):
        o, r, d, _ = b.step(acts[k])
        assert torch.equal(o, oa[k]) and torch.equal(r, ra[k]) and torch.equal(d, da[k].bool())
    half = n // 2
    for off in (0, half):
        c = BatchedShipEnv(half, bank=bank, seed=4, env_id_offset=off)
        c.reset()
        oc, rc, dc = c.rollout(acts[:, off:off + half].contiguous())
        assert torch.equal(oc, oa[:, off:off + half]) and torch.equal(rc, ra[:, off:off + half]) and torch.equal(dc, da[:, off:off + half])
    s = a.stats()
    assert s["episodes"] == float(da.sum()) and s["episodes"] > 0
    assert s["collision"] + s["oob"] + s["timeout"] + s["all_goals"] >= s["episodes"]


def test_random_agent_matches_oracle_philox():
    """ACTION_RANDOM (in-kernel Philox actions, the train/random.py agent) == oracle with the same counter RNG."""
    n, K = 2048, 24
    bank = fp32_bank(32, 600, 600, seed=9)
    env, orc = make_env(knobs(), n, bank, auto_reset=True, seed=123), make_oracle(knobs(), n, bank, auto_reset=True, seed=123)
    env.reset()
    orc.reset()
    obs, rew, done = _np(*env.rollout(None, K=K))
    ref = orc.step(None, K=K)
    rep = parity.compare_steps(ref, obs, rew, done, margin_thr=parity.MARGIN_THR)
    assert rep["grazing_frac"] < parity.MAX_EXCLUDED and rep["excluded_frac"] < parity.MAX_EXCLUDED_CUMULATIVE and rep["max_pose_rel_err"] < 2 * parity.REL_TOL


def test_action_dtypes_and_host_path():
    from ship_sim_gym_b200 import BatchedShipEnv, ScenarioBank
    n, K = 1024, 8
    bank = ScenarioBank.generate(16, (600, 600), seed=2)
    acts = torch.randint(0, 3, (K, n), device="cuda")
    outs = []
    for dt in (torch.int32, torch.int64, torch.uint8):
        e = BatchedShipEnv(n, bank=bank, seed=1)
        e.reset()
        outs.append(e.rollout(acts.to(dt)))
    e = BatchedShipEnv(n, bank=bank, seed=1)
    e.reset()
    ho, hr, hd = e.step_host(acts.cpu().numpy().astype(np.int32), K=K)
    for o, r, d in outs:
        assert torch.equal(o, outs[0][0]) and torch.equal(r, outs[0][1]) and torch.equal(d, outs[0][2])
    assert np.array_equal(ho, outs[0][0].cpu().numpy()) and np.array_equal(hr, outs[0][1].cpu().numpy())
    assert np.array_equal(hd, outs[0][2].cpu().numpy())


def test_reference_intents_and_errors():
    """The property intents of the reference's (stale) tests/test_ship_env.py, on the facade."""
    from ship_sim_gym_b200 import ShipEnv, BatchedShipEnv
    from ship_sim_gym_b200.config import EnvConfig, GameConfig
    env = ShipEnv(GameConfig, EnvConfig)
    obs = env.reset()
    assert obs.shape == (32,) and (obs[:16] == -1).all()
    assert obs[16] == 300 and obs[17] == 25                       # test_reset: spawn point (tests/test_ship_env.py:17-32)
    with pytest.raises(AssertionError):
        env.step(3)                                               # Discrete(3): ship_env.py:143
    o1, r1, d1, info = env.step(1)
    assert info == {} and r1 == pytest.approx(-0.01) and not d1   # test_reward: STEP_PENALTY (:220-239)
    assert (o1[16:18] == obs[16:18]).all() and o1[18] == -5       # rudder-only action leaves the pose unchanged (:48-103)
    assert (o1[:16] == obs[16:]).all()                            # test_history_states (:106-127)
    ys = []
    for _ in range(5):
        o, r, d, _ = env.step(0)
        ys.append(o[17])
    assert all(b > a for a, b in zip(ys[1:], ys[2:]))             # forward: y strictly increases after the first step
    assert o[16] < 300                                            # rudder -5 => positive torque => drift toward -x

    class BadEC(EnvConfig):
        HISTORY_SIZE = 0
    with pytest.raises(ValueError):
        BatchedShipEnv(4, GameConfig, BadEC)
    b = BatchedShipEnv(4)
    with pytest.raises(Exception):
        b.step(torch.zeros(4, dtype=torch.int32))                 # reset() first
    b.reset()
    with pytest.raises(AssertionError):
        b.step(torch.tensor([0, 1, 2, 3]))


@pytest.mark.parametrize("lanes", [1, 8])
def test_many_candidate_planes_serial_path(lanes):
    """Banks with 28-32 short edges (regular polygons): a reach-grid cell then names more candidate planes than a
    shared-memory scratch row holds, which takes the serial lidar path and the full separating-axis pass."""
    W = H = 600
    n, K = 2048, 12
    ang0 = np.linspace(0, 2 * np.pi, 28, endpoint=False)
    ang1 = np.linspace(0, 2 * np.pi, 32, endpoint=False) + 0.05
    h0 = np.stack([150 + 110 * np.cos(ang0), 300 + 110 * np.sin(ang0)], 1)       # CCW "islands" inside the map
    h1 = np.stack([450 + 90 * np.cos(ang1), 280 + 90 * np.sin(ang1)], 1)
    goals = np.array([[300, 100], [300, 200], [300, 300], [300, 400], [300, 500]], dtype=np.float64)
    bank = pack_bank([(h0, h1)], [goals])
    bank["hull_xy"] = bank["hull_xy"].astype(np.float32).astype(np.float64)
    env = make_env(knobs(), n, bank, auto_reset=True, seed=3, lanes_per_env=lanes)
    orc = make_oracle(knobs(), n, bank, auto_reset=True, seed=3)
    env.reset()
    orc.reset()
    rng = np.random.RandomState(5)
    st = parity.f32_inputs(*parity.random_states(rng, n, W, H, 1, bank["goals"], near=(bank["hull_xy"], bank["hull_n"])))
    env.set_state(*st)
    parity.load_oracle_state(orc, *st)
    acts = rng.randint(0, 3, (K, n)).astype(np.int32)
    obs, rew, done = _np(*env.rollout(torch.tensor(acts, device=env.device)))
    ref = orc.step(acts)
    rep = parity.compare_steps(ref, obs, rew, done, margin_thr=parity.MARGIN_THR, label="islands")
    assert rep["grazing_frac"] < parity.MAX_EXCLUDED and rep["excluded_frac"] < parity.MAX_EXCLUDED_CUMULATIVE, rep
    assert (ref["flags"] & oracle.FLAG_COLLIDING).any() and (orc.lidar[:, :10] >= 0).mean() > 0.1
    env.close()


@pytest.mark.parametrize("auto_reset", [True, False])
@pytest.mark.parametrize("n,K", [(1000, 100), (300, 7)])
def test_host_path_rebuilds_history_from_frames(auto_reset, n, K):
    """shipsim_step_host ships one frame per env-step and rebuilds [previous frame | frame] rows on the host
    (reset observations included): bit-identical to the device-resident rollout, across consecutive calls, after a
    state injection, and when the caller does not ask for the done flags."""
    from ship_sim_gym_b200 import BatchedShipEnv, ScenarioBank
    bank = ScenarioBank.generate(16, (600, 600), seed=2)
    rng = np.random.RandomState(4)
    envs = [BatchedShipEnv(n, bank=bank, seed=1, auto_reset=auto_reset) for _ in range(2)]
    for e in envs:
        e.reset()
    st = parity.f32_inputs(*parity.random_states(rng, n, 600, 600, 16, bank.goals))
    for it in range(3):
        if it == 1:
            for e in envs:
                e.set_state(*st)
        acts = rng.randint(0, 3, (K, n)).astype(np.int32)
        o, r, d = [t.cpu().numpy() for t in envs[0].rollout(torch.tensor(acts, device="cuda"))]
        if it == 2:
            ho = np.empty((K, n, 32), dtype=np.float32)
            envs[1].step_host(acts, K=K, out=(ho, None, None))
        else:
            ho, hr, hd = envs[1].step_host(acts, K=K)
            assert np.array_equal(hr, r) and np.array_equal(hd, d)
        assert np.array_equal(ho, o), "call %d" % it
        if auto_reset and K >= 100:
            assert d.sum() > 0


@pytest.mark.parametrize("dma_envs", ["0", "96", "512", "1000", None])
def test_host_path_two_engine_split(dma_envs, monkeypatch):
    """shipsim_step_host with page-locked caller buffers: the envs [0, nd) come home as complete rows by DMA
    (history_rows_kernel), the others compacted and expanded by the host threads.  Every split -- none, ragged, all, and
    the self-balancing one over consecutive calls -- gives the rows, rewards and done flags of the device-resident rollout,
    bit for bit."""
    from ship_sim_gym_b200 import BatchedShipEnv, ScenarioBank
    if dma_envs is None:
        monkeypatch.delenv("SHIPSIM_HOST_DMA_ENVS", raising=False)
    else:
        monkeypatch.setenv("SHIPSIM_HOST_DMA_ENVS", dma_envs)
    if dma_envs == "96":          # the speculative copy of the changed values falls short: a host thread fetches the rest
        monkeypatch.setenv("SHIPSIM_HOST_VAR_DENSITY", "0")
    n, K = (1000, 64) if dma_envs is not None else (4096, 80)
    bank = ScenarioBank.generate(16, (600, 600), seed=2)
    rng = np.random.RandomState(5)
    envs = [BatchedShipEnv(n, bank=bank, seed=1, auto_reset=True) for _ in range(2)]
    for e in envs:
        e.reset()
    pin = lambda *s, dtype: torch.empty(*s, dtype=dtype).pin_memory()       # noqa: E731
    ho, hr, hd = pin(K, n, 32, dtype=torch.float32), pin(K, n, dtype=torch.float32), pin(K, n, dtype=torch.uint8)
    seen = set()
    for it in range(6 if dma_envs is None else 2):
        acts = rng.randint(0, 3, (K, n)).astype(np.int32)
        o, r, d = [t.cpu().numpy() for t in envs[0].rollout(torch.tensor(acts, device="cuda"))]
        ho.fill_(7.0)
        envs[1].step_host(acts, K=K, out=(ho.numpy(), hr.numpy(), hd.numpy()))
        assert np.array_equal(ho.numpy(), o) and np.array_equal(hr.numpy(), r) and np.array_equal(hd.numpy(), d), "call %d" % it
        seen.add(envs[1].host_traffic()[1])
    assert d.sum() > 0
    if dma_envs is None:
        assert len(seen) > 1          # the split moved between calls (it follows the measured balance)
    for e in envs:
        e.close()


@pytest.mark.parametrize("auto_reset", [True, False])
def test_long_history_rollout_matches_single_steps(auto_reset):
    """HISTORY_SIZE > 2 (config.py:15; SURVEY App. A note N2): rollout() assembles the rows [frame t-H+1 | ... | frame t]
    from the frames of a K-step launch and the running history, -1 behind an env's latest reset (ship_env.py:180-184).
    Same rows, bit for bit, as K calls of step(), across consecutive rollouts, and through step_host."""
    from ship_sim_gym_b200 import BatchedShipEnv, ScenarioBank
    from ship_sim_gym_b200.config import EnvConfig, GameConfig

    class EC(EnvConfig):
        HISTORY_SIZE = 4
        MAX_STEPS = 25
    n, K = 300, 40
    bank = ScenarioBank.generate(16, (600, 600), seed=2)
    envs = [BatchedShipEnv(n, GameConfig, EC, bank=bank, seed=1, auto_reset=auto_reset) for _ in range(2)]
    rng = np.random.RandomState(7)
    o0 = [e.reset() for e in envs]
    assert o0[0].shape == (n, 64) and torch.equal(o0[0], o0[1])
    for it in range(3):
        acts = torch.tensor(rng.randint(0, 3, (K, n)).astype(np.int32), device="cuda")
        if it < 2:
            ro, rr, rd = envs[0].rollout(acts)
        else:
            ho, hr, hd = envs[0].step_host(acts.cpu().numpy(), K=K)
            ro, rr, rd = torch.tensor(ho, device="cuda"), torch.tensor(hr, device="cuda"), torch.tensor(hd, device="cuda")
        assert ro.shape == (K, n, 64)
        for k in range(K):
            so, sr, sd, _ = envs[1].step(acts[k])
            assert torch.equal(ro[k], so), (it, k)
            assert torch.equal(rr[k], sr) and torch.equal(rd[k].bool(), sd)
    if auto_reset:
        assert rd.sum() > 0 and (ro[:, :, :16] == -1).all(-1).any()
    for e in envs:
        e.close()
