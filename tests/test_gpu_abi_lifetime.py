"""-m gpu: what a libshipsim handle owns and when -- the device-generated bank that fresh maps regenerate in place, the
events a host-path trace reads, and the release of every buffer, stream and event when the handle is destroyed."""
import gc
import re

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

HOST_VARS = ("SHIPSIM_HOST_TRACE", "SHIPSIM_HOST_CHUNKS", "SHIPSIM_HOST_DMA_ENVS", "SHIPSIM_HOST_VAR_DENSITY", "SHIPSIM_HOST_THREADS")


@pytest.fixture
def host_env(monkeypatch):
    for var in HOST_VARS:
        monkeypatch.delenv(var, raising=False)
    return monkeypatch


def test_fresh_maps_refuse_a_host_loaded_bank():
    """Fresh maps regenerate the device-generated bank in place, in its own layout.  A host bank loaded after a device
    bank of the same size is not that bank: turning fresh maps on must fail (SHIPSIM_ERR_STATE), whatever was generated
    before."""
    from ship_sim_gym_b200 import BatchedShipEnv, ScenarioBank, _abi
    env = BatchedShipEnv(64, n_scenarios=1024, seed=1, scenario_source="device", auto_reset=True)
    bank = ScenarioBank.generate(1024, (600, 600), seed=2)
    assert bank.maxv < _abi.MAX_HULL                # a record stride other than the generated bank's
    env.load_scenarios(bank)
    with pytest.raises(_abi.ShipsimError, match="error -3"):
        env.fresh_maps(True)
    assert env.fresh_info()["enabled"] is False
    env.generate_scenarios(1024, seed=3)            # a device bank again: fresh maps are accepted
    env.fresh_maps(True)
    assert env.fresh_info()["enabled"] is True
    env.close()


def test_host_trace_asked_for_after_the_first_call(host_env, capfd):
    """SHIPSIM_HOST_TRACE set only after a handle's first frames-only step_host call: the call still gives the rows of
    rollout(), and the trace reads real chunk times."""
    from ship_sim_gym_b200 import BatchedShipEnv, ScenarioBank
    n, K = 1024, 64                                 # n * K = 65,536 env-steps: the frames-only regime
    bank = ScenarioBank.generate(16, (600, 600), seed=2)
    envs = [BatchedShipEnv(n, bank=bank, seed=1, auto_reset=True) for _ in range(2)]
    for e in envs:
        e.reset()
    rng = np.random.RandomState(5)
    for it in range(2):
        if it == 1:
            host_env.setenv("SHIPSIM_HOST_TRACE", "1")
        acts = rng.randint(0, 3, (K, n)).astype(np.int32)
        o, r, d = [t.cpu().numpy() for t in envs[0].rollout(torch.tensor(acts, device="cuda"))]
        ho, hr, hd = envs[1].step_host(acts, K=K)
        assert np.array_equal(ho, o) and np.array_equal(hr, r) and np.array_equal(hd, d), "call %d" % it
    err = capfd.readouterr().err
    home = [float(x) for x in re.findall(r"records home ([0-9.]+)", err)]
    assert len(home) == 16 and max(home) > 0.0, err
    for e in envs:
        e.close()


def test_handles_release_everything(host_env):
    """Rounds of create, step_host at K = 64 then 256 (every staging buffer regrows), generate_scenarios, fresh maps on
    and off, load_scenarios, the episode log, close: device memory comes back.  The GPU may be shared, so the bound is a
    share of one round's allocation, not zero."""
    from ship_sim_gym_b200 import BatchedShipEnv, ScenarioBank
    n, S = 4096, 64
    bank = ScenarioBank.generate(S, (600, 600), seed=4)
    acts = {K: np.random.RandomState(K).randint(0, 3, (K, n)).astype(np.int32) for K in (64, 256)}

    def free_bytes():
        gc.collect()
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        return torch.cuda.mem_get_info()[0]

    def one_round():
        env = BatchedShipEnv(n, n_scenarios=S, seed=1, scenario_source="device", auto_reset=True)
        env.reset()
        for K in (64, 256):
            env.step_host(acts[K], K=K)
        env.generate_scenarios(S, seed=3)
        env.fresh_maps(True)
        env.fresh_maps(False)
        env.load_scenarios(bank)
        env.enable_episode_log()
        used = torch.cuda.mem_get_info()[0]
        env.close()
        return used

    one_round()                                     # (the first round also loads the kernels)
    before = free_bytes()
    round_bytes = before - one_round()
    assert round_bytes > 100 << 20                  # the staging buffers alone: K = 256 rows of 4,096 envs
    before = free_bytes()
    for _ in range(19):
        one_round()
    after = free_bytes()
    # a tenth of one round over 19 rounds: a leaked bank (a few MB a round) fails, other work on a shared GPU does not
    assert before - after < round_bytes // 10, (before, after, round_bytes)
