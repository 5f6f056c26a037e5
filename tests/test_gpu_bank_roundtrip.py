"""-m gpu: a bank generated on the device, read back (shipsim_read_scenarios) and loaded from the host
(shipsim_load_scenarios) plays bit for bit like the generated bank itself, through both step kernels.  Both paths write
their scenario records with the same kernel from the same fp32-rounded vertices, so a map saved from a run and loaded
again replays that run."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from helpers import assert_same, run  # noqa: E402
import parity  # noqa: E402


@pytest.mark.parametrize("T", [16, 1])
def test_read_back_bank_plays_like_the_generated_bank(T):
    from ship_sim_gym_b200 import BatchedShipEnv
    n, K, S = 4096, 256, 4096
    kw = dict(seed=11, auto_reset=True, steps_in_flight=T)
    gen = BatchedShipEnv(n, n_scenarios=S, scenario_source="device", **kw)
    bank = gen.read_scenarios()
    loaded = BatchedShipEnv(n, bank=bank, **kw)
    rng = np.random.RandomState(5)
    acts = torch.tensor(rng.choice([0, 0, 1, 2], size=(K, n)).astype(np.int32), device="cuda")
    goals = bank.goals.astype(np.float32).astype(np.float64)            # the goals the kernels hold
    st = parity.f32_inputs(*parity.random_states(rng, n, 600, 600, S, goals, near=(bank.hull_xy, bank.hull_n)))
    want = run(gen, acts, K, st)
    got = run(loaded, acts, K, st)
    assert want[3]["steps_in_flight"] == T and got[3]["steps_in_flight"] == T
    assert_same(got, want, "loaded read-back bank, T=%d" % T)
    (obs, _, done), _, stats, _ = want
    assert done.sum() > 0 and stats["episodes"] == float(done.sum())    # auto-resets onto other maps occurred
    assert (obs[..., -10:] >= 0).any()                                   # lidar hits occurred
    gen.close()
    loaded.close()
