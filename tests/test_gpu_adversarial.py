"""-m gpu: the adversarial injected-state sets SURVEY.md section 8(d) names besides "ship near a bank edge"
(tests/test_gpu_parity.py): a goal at distance 5 +- eps from the hull, and the ray origin inside a bank."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

import oracle  # noqa: E402
from helpers import fp32_bank, knobs, make_env, make_oracle  # noqa: E402
import parity  # noqa: E402


@pytest.mark.parametrize("lanes,window", [(1, 1), (8, 1), (0, 16)])
def test_goal_at_radius_plus_minus_eps(lanes, window):
    """collide_goal (game.py:243-257) fires iff distance(goal centre, ship polygon) <= 5: goals placed 2e-3 ... 1e-2
    inside and outside that shell, off edges and off vertices, must be classified exactly as the oracle does."""
    W = H = 600
    n = 4096 + 7
    bank = fp32_bank(8, W, H, seed=2)
    rng = np.random.RandomState(17)
    pose, ints, lidar, goals, ret, delta = parity.goal_shell_states(rng, n, W, H, 8)
    st = parity.f32_inputs(pose, ints, lidar, goals, ret)
    if window > 1:          # the time-parallel kernel needs a rollout of at least one window
        env = make_env(knobs(), n, bank, auto_reset=False, steps_in_flight=window)
    else:
        env = make_env(knobs(), n, bank, auto_reset=False, lanes_per_env=lanes)
    orc = make_oracle(knobs(), n, bank)
    K = window
    env.reset()
    orc.reset()
    env.set_state(*st)
    parity.load_oracle_state(orc, *st)
    acts = np.full((K, n), 1, dtype=np.int32)          # rudder only: the ship stays where it is
    obs, rew, done = [t.cpu().numpy() for t in env.rollout(torch.tensor(acts, device=env.device))]
    assert env.launch_info()["steps_in_flight"] == window
    ref = orc.step(acts)
    rep = parity.compare_steps(ref, obs, rew, done, margin_thr=parity.MARGIN_THR, label="goal shell", stop_at_done=True)
    assert rep["grazing_frac"] < parity.MAX_EXCLUDED, rep
    f = ref["flags"][0]
    took = (f & oracle.FLAG_GOAL) != 0
    assert took[delta < 0].all() and not took[delta > 0].any()          # the set is what it claims to be
    # the kernel's decision, read straight from the reward of step 0 (+1 on a goal step, ship_env.py:68-69)
    assert ((rew[0] == 1.0) == took).all()
    assert (ref["margins"][0, :, parity.M_GOAL] < 1.5e-2).all()
    env.close()


@pytest.mark.parametrize("lanes", [1, 8, 32])
def test_ray_origin_inside_a_bank(lanes):
    """cpShapeSegmentQuery with the start point inside the shape: alpha = 0 and `point` stays at the ray end, so
    LiDAR.query stores the full ray length for every beam (App. B Q11, App. C4)."""
    W = H = 600
    n = 4096 - 3
    bank = fp32_bank(32, W, H, seed=4)
    rng = np.random.RandomState(23)
    pose, ints, lidar, which = parity.origin_inside_bank_states(rng, n, bank["hull_xy"], bank["hull_n"], 32)
    goals = bank["goals"][ints[:, 3]].reshape(n, 10)
    st = parity.f32_inputs(pose, ints, lidar, goals, np.zeros(n))
    env, orc = make_env(knobs(), n, bank, auto_reset=False, lanes_per_env=lanes), make_oracle(knobs(), n, bank)
    env.reset()
    orc.reset()
    env.set_state(*st)
    parity.load_oracle_state(orc, *st)
    acts = rng.randint(0, 3, (1, n)).astype(np.int32)
    o, r, d, _ = env.step(torch.tensor(acts[0], device=env.device))
    ref = orc.step(acts)
    rep = parity.compare_steps(ref, o.cpu().numpy()[None], r.cpu().numpy()[None], d.cpu().numpy()[None], label="origin inside")
    assert rep["grazing_frac"] < parity.MAX_EXCLUDED, rep
    got = o.cpu().numpy()[:, 22:32]
    ok = ref["margins"][0].min(-1) >= parity.MARGIN_THR
    assert np.allclose(got[ok], 100.0, rtol=0, atol=1e-3) and ok.mean() > 0.95
    assert ((ref["flags"][0] & oracle.FLAG_COLLIDING) != 0)[ok].mean() > 0.9     # the hull overlaps that bank as well
    env.close()
