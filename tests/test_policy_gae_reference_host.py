"""CPU: the float64 references of the policy and GAE kernels (tests/references.py) checked on their own -- an fp32
evaluation of the same network / recurrence lands inside the error scale they give, and the defects the GPU tests look
for land outside it, so that a kernel held to these references cannot hide such a defect in the tolerance."""
import numpy as np
import pytest

torch = pytest.importorskip("torch")

from references import H, U, env_obs, gae64, mlp_forward64, policy_weights  # noqa: E402

GAMMA_LAM = [(0.99, 0.95), (1.0, 1.0), (0.99, 0.0), (0.0, 0.95)]


def torch_fused(obs, w, l1_drop_last=False, value_reads_policy_h1=False):
    """The fused network in fp32 torch, as RolloutCollector's generic fused path evaluates it (addmm, tanh), optionally
    with one of two defects: layer 1 without its last input, or the value trunk fed the policy trunk's h1."""
    t = {k: torch.tensor(v) for k, v in w.items()}
    x = torch.tensor(obs)
    w1 = t["w1"].clone()
    if l1_drop_last:
        w1[-1] = 0.0
    h1 = torch.addmm(t["b1"], x, w1).tanh()
    if value_reads_policy_h1:
        h1 = torch.cat([h1[:, :H], h1[:, :H]], 1)
    w2 = torch.block_diag(t["w2"][0], t["w2"][1])
    h2 = torch.addmm(t["b2"], h1, w2).tanh()
    w3 = torch.zeros_like(t["w3"])
    w3[:H, :3], w3[H:, 3] = t["w3"][:H, :3], t["w3"][H:, 3]
    return torch.addmm(t["b3"], h2, w3).numpy().astype(np.float64)


@pytest.mark.parametrize("l1_scale", [1.0, 30.0])
def test_mlp_forward64_holds_fp32_torch_within_4_sigma(l1_scale):
    rng = np.random.RandomState(int(l1_scale))
    policy, w = policy_weights(7, l1_scale=l1_scale)
    obs = env_obs(rng, 4096)
    ref, sigma = mlp_forward64(obs, **w)
    assert (sigma > 0).all()
    ratio = np.abs(torch_fused(obs, w) - ref) / sigma
    assert ratio.max() <= 4.0, ratio.max()
    # the layouts are the module's: the fp32 module (observation scale not folded into w1) agrees to fp32 accuracy
    with torch.no_grad():
        logits, value = policy(torch.tensor(obs))
    mod = np.concatenate([logits.numpy(), value.numpy()[:, None]], 1)
    assert np.abs(mod - ref).max() < 1e-4
    # the defects land outside: layer 1 without its last input, the value trunk fed the policy trunk's h1
    assert (np.abs(torch_fused(obs, w, l1_drop_last=True) - ref) / sigma).max() > 4.0
    bad = np.abs(torch_fused(obs, w, value_reads_policy_h1=True) - ref) / sigma
    assert bad[:, 3].max() > 4.0 and bad[:, :3].max() <= 4.0


def loop_gae(rew, val, done, gamma, lam):
    """The recurrence one element at a time in Python floats (float64)."""
    g = float(np.float32(gamma))
    gl = float(np.float32(np.float32(gamma) * np.float32(lam)))
    T, N = rew.shape
    adv = np.empty((T, N))
    for e in range(N):
        last = 0.0
        for t in range(T - 1, -1, -1):
            nt = 0.0 if done[t, e] else 1.0
            delta = float(rew[t, e]) + g * float(val[t + 1, e]) * nt - float(val[t, e])
            last = delta + gl * nt * last
            adv[t, e] = last
    return adv


def gae32(rew, val, done, gamma, lam, ignore_lam=False, bootstrap_across_done=False):
    """The recurrence in fp32 numpy (every operation rounded), optionally with one of two defects."""
    f = np.float32
    g = f(gamma)
    gl = g if ignore_lam else f(g * f(lam))
    nt = (done == 0).astype(np.float32)
    last = np.zeros(rew.shape[1], np.float32)
    adv = np.empty_like(rew)
    for t in range(rew.shape[0] - 1, -1, -1):
        delta = rew[t] + g * val[t + 1] * (f(1) if bootstrap_across_done else nt[t]) - val[t]
        last = delta + gl * nt[t] * last
        adv[t] = last
    return adv, adv + val[:-1]


def gae_inputs(rng, T, N, p_done):
    rew = rng.choice(np.float32([1.0, -1.0, -0.01]), size=(T, N), p=[0.05, 0.05, 0.9])
    val = (rng.randn(T + 1, N) * 10).astype(np.float32)
    done = (rng.rand(T, N) < p_done).astype(np.uint8)
    return rew, val, done


@pytest.mark.parametrize("gamma,lam", GAMMA_LAM)
def test_gae64_is_the_recurrence_and_bounds_an_fp32_evaluation(gamma, lam):
    rng = np.random.RandomState(int(100 * gamma + 10 * lam))
    rew, val, done = gae_inputs(rng, 300, 64, 0.05)
    done[0, 0] = done[-1, 1] = 1
    adv, ret, badv, bret = gae64(rew, val, done, gamma, lam)
    small = slice(0, 9)
    assert np.allclose(adv[:, small], loop_gae(rew[:, small], val[:, small], done[:, small], gamma, lam), rtol=1e-12, atol=1e-12)
    assert np.array_equal(ret, adv + val[:-1].astype(np.float64))
    a32, r32 = gae32(rew, val, done, gamma, lam)
    assert (np.abs(a32 - adv) <= badv).all() and (np.abs(r32 - ret) <= bret).all()
    # a recurrence that bootstraps across a done is outside the bound (gamma = 0 never bootstraps) ...
    if gamma > 0:
        a, _ = gae32(rew, val, done, gamma, lam, bootstrap_across_done=True)
        assert (np.abs(a - adv) > badv).any()
    # ... and so is one that ignores lam (lam = 1 or gamma = 0: gamma lam = gamma, nothing to ignore)
    if lam != 1.0 and gamma != 0.0:
        a, _ = gae32(rew, val, done, gamma, lam, ignore_lam=True)
        assert (np.abs(a - adv) > badv).any()


def test_gae64_bound_is_the_unit_roundoff_on_a_single_step():
    """T = 1, no done: adv = r + gamma v1 - v0, three roundings at most."""
    rew, val, done = np.float32([[0.5]]), np.float32([[3.0], [-2.0]]), np.zeros((1, 1), np.uint8)
    adv, ret, badv, bret = gae64(rew, val, done, 0.5, 0.3)
    assert adv[0, 0] == 0.5 + 0.5 * -2.0 - 3.0
    assert badv[0, 0] == pytest.approx(4 * U * (0.5 + 1.0 + 3.0)) and bret[0, 0] > badv[0, 0]
