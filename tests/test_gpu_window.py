"""-m gpu: the time-parallel window kernel (shipsim_window.cu, `steps_in_flight` > 1) against the serial-in-time step
kernel -- bit for bit: observations, rewards, done flags, the final state and the episode counters -- and against
the float64 oracle.  The window kernel speculates T steps of an env at once and cuts the window at the first done
step, so the cases below make sure windows get cut (short episodes), straddle the end of the rollout (K not a
multiple of T), meet ragged batches, both history sizes, no-auto-reset stepping and the serial lidar path."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from helpers import assert_same, case_knobs, fp32_bank, knobs, make_env, make_oracle, pack_bank, run  # noqa: E402
import parity  # noqa: E402


CASES = [
    dict(name="default", n=1000 + 3, K=37),
    dict(name="short_episodes", n=515, K=64, max_steps=7),                    # every window gets cut
    dict(name="history1", n=700, K=33, hist=1),
    dict(name="no_auto_reset", n=900, K=40, auto_reset=False),
    dict(name="hard_map", n=1024 + 1, K=45, W=1000, H=1000, map_N=30, wf=0.9, spread=180),
    dict(name="sb_script", n=600, K=40, W=1000, H=1000, speed=30),
    dict(name="random_agent", n=800, K=50, random_agent=True),
    dict(name="K_equals_T", n=300, K=None),
]


@pytest.mark.parametrize("T", [4, 8, 16, 32])
@pytest.mark.parametrize("case", CASES, ids=[c["name"] for c in CASES])
def test_window_kernel_is_bit_identical_to_serial_kernel(case, T):
    W, H = case.get("W", 600), case.get("H", 600)
    n = case["n"]
    K = case["K"] or T
    k = case_knobs(case)
    bank = fp32_bank(48, W, H, seed=13, map_N=k["map_N"], wf=k["wf"])
    kw = dict(auto_reset=case.get("auto_reset", True), seed=5)
    rng = np.random.RandomState(3)
    acts = None if case.get("random_agent") else torch.tensor(rng.choice([0, 0, 1, 2], size=(K, n)).astype(np.int32), device="cuda")
    # start from scattered states (near the banks too) so that lidar hits, collisions and goals all occur early
    st = parity.f32_inputs(*parity.random_states(rng, n, W, H, 48, bank["goals"], near=(bank["hull_xy"], bank["hull_n"])))
    ref = run(make_env(k, n, bank, lanes_per_env=1, steps_in_flight=1, **kw), acts, K, st)
    got = run(make_env(k, n, bank, steps_in_flight=T, **kw), acts, K, st)
    assert ref[3]["steps_in_flight"] == 1 and got[3]["steps_in_flight"] == T
    assert_same(got, ref, "%s T=%d" % (case["name"], T))
    (o, r, d), _, stats, _ = ref
    if case.get("auto_reset", True) and K >= 24:
        assert d.sum() > 0 and stats["episodes"] == float(d.sum())      # windows were cut
    assert (o[..., -10:] >= 0).any()                                     # lidar hits occurred


def test_window_kernel_consecutive_rollouts_and_serial_path():
    """Several launches in a row (state, sticky lidar and goals carried through HBM between launches), on the map
    whose reach-grid cells name more candidate planes than a scratch row holds (serial lidar path + full SAT)."""
    W = H = 600
    n, K = 777, 20
    ang0 = np.linspace(0, 2 * np.pi, 28, endpoint=False)
    ang1 = np.linspace(0, 2 * np.pi, 32, endpoint=False) + 0.05
    h0 = np.stack([150 + 110 * np.cos(ang0), 300 + 110 * np.sin(ang0)], 1)
    h1 = np.stack([450 + 90 * np.cos(ang1), 280 + 90 * np.sin(ang1)], 1)
    goals = np.array([[300, 100], [300, 200], [300, 300], [300, 400], [300, 500]], dtype=np.float64)
    bank = pack_bank([(h0, h1)], [goals])
    bank["hull_xy"] = bank["hull_xy"].astype(np.float32).astype(np.float64)
    rng = np.random.RandomState(9)
    st = parity.f32_inputs(*parity.random_states(rng, n, W, H, 1, bank["goals"], near=(bank["hull_xy"], bank["hull_n"])))
    envs = [make_env(knobs(), n, bank, seed=2, **kw) for kw in (dict(lanes_per_env=4, steps_in_flight=1), dict(steps_in_flight=8),
                                                                   dict(steps_in_flight=32))]
    for e in envs:
        e.reset()
        e.set_state(*st)
    for it in range(4):
        acts = torch.tensor(rng.randint(0, 3, (K, n)).astype(np.int32), device="cuda")
        outs = [[t.cpu().numpy() for t in e.rollout(acts)] for e in envs]
        for o in outs[1:]:
            for a, b in zip(o, outs[0]):
                assert np.array_equal(a, b), "launch %d" % it
    s0 = envs[0].get_state()
    for e in envs[1:]:
        s = e.get_state()
        for k in s0:
            assert np.array_equal(s[k], s0[k]), k


@pytest.mark.parametrize("T", [8, 32])
def test_window_kernel_against_oracle(T):
    W = H = 600
    n, K = 4096 + 3, 32
    bank = fp32_bank(64, W, H, seed=5)
    env = make_env(knobs(), n, bank, auto_reset=True, seed=11, steps_in_flight=T)
    orc = make_oracle(knobs(), n, bank, auto_reset=True, seed=11)
    env.reset()
    orc.reset()
    rng = np.random.RandomState(21)
    acts = rng.choice([0, 0, 1, 2], size=(K, n)).astype(np.int32)
    obs, rew, done = [t.cpu().numpy() for t in env.rollout(torch.tensor(acts, device=env.device))]
    assert env.launch_info()["steps_in_flight"] == T
    ref = orc.step(acts)
    rep = parity.compare_steps(ref, obs, rew, done, margin_thr=parity.MARGIN_THR, label="window T=%d" % T, scale=max(W, H))
    assert rep["grazing_frac"] < parity.MAX_EXCLUDED and rep["excluded_frac"] < parity.MAX_EXCLUDED_CUMULATIVE, rep
    assert rep["max_pose_rel_err"] < 2 * parity.REL_TOL
    s, so = env.stats(), orc.stats_dict()
    assert abs(s["episodes"] - so["episodes"]) <= max(3, 0.01 * so["episodes"]) and s["episodes"] == float(done.sum())


def test_auto_selection():
    """steps_in_flight = 0: small batches with K >= window take the window kernel, K = 1 stepping and explicit
    lanes_per_env the serial one."""
    bank = fp32_bank(8, 600, 600, seed=1)
    e = make_env(knobs(), 256, bank)
    e.reset()
    e.rollout(None, K=16)
    assert e.launch_info()["steps_in_flight"] == 1            # fewer steps than the window (32 for so few envs)
    e.rollout(None, K=40)
    assert e.launch_info()["steps_in_flight"] == 32
    e.step(torch.zeros(256, dtype=torch.int32, device="cuda"))
    assert e.launch_info()["steps_in_flight"] == 1
    e2 = make_env(knobs(), 256, bank, lanes_per_env=8)
    e2.reset()
    e2.rollout(None, K=40)
    assert e2.launch_info()["steps_in_flight"] == 1
    with pytest.raises(ValueError):
        make_env(knobs(), 16, bank, steps_in_flight=5)
    # the window is as long as still lets every warp be resident (include/shipsim.h: SHIPSIM_WINDOW_AUTO_MAX_ENVS)
    for n, want in ((2368, 32), (2369, 16), (4736, 16), (4737, 8), (32768, 8), (32769, 1)):
        e3 = make_env(knobs(), n, bank)
        e3.reset()
        e3.rollout(None, K=32)
        assert e3.launch_info()["steps_in_flight"] == want, (n, e3.launch_info())
        e3.close()


def test_million_envs_agree_with_small_shards():
    """BASELINE configs[3] size (1,048,576 envs, serial-in-time kernel, one lane per env) against 4,096-env shards of
    the same global env ids run through the window kernel: results depend neither on the batch size nor on which
    kernel computed them."""
    from ship_sim_gym_b200 import BatchedShipEnv, ScenarioBank
    n, K, m = 1048576, 32, 4096
    bank = ScenarioBank.generate(256, (600, 600), seed=3)
    big = BatchedShipEnv(n, bank=bank, seed=9, validate_actions=False)
    big.reset()
    obs, rew, done = big.rollout(None, K=K)                    # in-kernel Philox actions, keyed by global env id and step
    assert big.launch_info()["steps_in_flight"] == 1 and big.launch_info()["lanes_per_env"] == 1
    for off in (0, 517 * 1024, n - m):
        small = BatchedShipEnv(m, bank=bank, seed=9, env_id_offset=off, validate_actions=False)
        small.reset()
        o, r, d = small.rollout(None, K=K)
        assert small.launch_info()["steps_in_flight"] == 16
        assert torch.equal(o, obs[:, off:off + m]) and torch.equal(r, rew[:, off:off + m]) and torch.equal(d, done[:, off:off + m])
        small.close()
    s = big.stats()
    assert s["episodes"] == float(done.sum()) and s["episodes"] > 100000
