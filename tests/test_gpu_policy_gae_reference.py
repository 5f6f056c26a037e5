"""-m gpu: the policy-in-the-loop kernels (csrc/shipsim_policy.cu) against the float64 references of tests/references.py.

mlp_policy_kernel through shipsim_mlp_policy_forward at every grid shape it runs -- one env, part of a tile, one pass of
the grid and a slot without a tile, several passes (the grid deals 16-env tiles over gridDim.x x 8 slots per pass) --
within 4 sigma of mlp_forward64, writing exactly rows 0 .. n - 1, with rows that do not depend on which tile, slot,
pass or CTA computed them, the float64 argmax wherever the decision is clear, the first maximum on exact ties, and a
tanh that keeps its stated accuracy; argument checks before the launch; one process on two devices.  gae_kernel through
shipsim_gae within gae64's bound at short and long rollouts, odd env counts and the edge values of gamma and lam;
shipsim_gae_scored on synthetic episode logs, several steps per call and more records than one round of the scatter
grid."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from references import (TANH_EPS, U, env_obs, gae64, gumbel, loop_attribution, mlp_forward64, policy_weights,  # noqa: E402
                        synthetic_rollout)

SENTINEL_BITS = 0x7FA5A5A5      # a NaN with a payload: what the rows past n hold before and after a call
PAD = 64                        # rows past n
N_SCEN = 48
WEIGHT_NAMES = ("w1", "b1", "w2", "b2", "w3", "b3")


def lib():
    from ship_sim_gym_b200 import _abi
    return _abi.load()


def slots_per_pass(dev=0):
    """Envs one pass of mlp_policy_kernel's grid covers: 16-env tiles x 8 slots x one CTA per SM."""
    return 16 * 8 * torch.cuda.get_device_properties(dev).multi_processor_count


def cuda(a, dev="cuda"):
    return torch.from_numpy(np.ascontiguousarray(a)).to(dev)


def sentinel_out(n, dev="cuda"):
    return torch.full((n + PAD, 4), SENTINEL_BITS, dtype=torch.int32, device=dev).view(torch.float32)


def policy_call(obs, w, noise, n=None, out=None, actions=None, shift=None):
    """shipsim_mlp_policy_forward on device tensors: rows 0 .. n - 1 of obs / noise, into fresh sentinel-filled out
    [n + PAD][4] and actions [n + PAD].  `shift`: {buffer name: bytes added to its pointer}.  -> (rc, out, actions)."""
    n = obs.shape[0] if n is None else n
    dev = obs.device
    out = sentinel_out(n, dev) if out is None else out
    actions = torch.full((n + PAD,), -7, dtype=torch.int64, device=dev) if actions is None else actions
    ptr = dict(obs=obs.data_ptr(), noise=noise.data_ptr(), out=out.data_ptr(), actions=actions.data_ptr(),
               **{k: w[k].data_ptr() for k in WEIGHT_NAMES})
    for k, b in (shift or {}).items():
        ptr[k] += b
    with torch.cuda.device(dev):
        rc = lib().shipsim_mlp_policy_forward(ptr["obs"], n, *[ptr[k] for k in WEIGHT_NAMES], ptr["noise"], ptr["out"], ptr["actions"],
                                              torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
    return rc, out, actions


def assert_sentinels(out, actions, n, what):
    """Rows below n written (no sentinel bits, an action in 0..2), rows from n on untouched."""
    bits = out.view(torch.int32)
    assert not bool((bits[:n] == SENTINEL_BITS).any()), "%s: a row below n was not written" % what
    assert bool(((actions[:n] >= 0) & (actions[:n] <= 2)).all()), "%s: an action below n was not written" % what
    assert bool((bits[n:] == SENTINEL_BITS).all()), "%s: a row past n was written" % what
    assert bool((actions[n:] == -7).all()), "%s: an action past n was written" % what


# ---------------------------------------------------------------------------------------------- the policy kernel
def shapes():
    S = slots_per_pass()
    return S, [1, 15, 16, 17, S - 1, S, S + 1, 2 * S + 37, 65536, 65536 + 7]


@pytest.fixture(scope="module", params=["default", "saturated"])
def policy_case(request):
    """One weight set (heads x 4; 'saturated': layer 1 x 30 as well), env-like observations and Gumbel noise for the
    largest batch, their float64 reference, and the kernel's output at every size of shapes() on prefixes of them."""
    rng = np.random.RandomState(11 if request.param == "default" else 12)
    _, w = policy_weights(21, l1_scale=30.0 if request.param == "saturated" else 1.0)
    S, ns = shapes()
    n_max = max(ns)
    obs, noise = env_obs(rng, n_max), gumbel(rng, n_max)
    ref, sigma = mlp_forward64(obs, **w)
    wd = {k: cuda(v) for k, v in w.items()}
    obs_d, noise_d = cuda(obs), cuda(noise)
    runs = {}
    for n in ns:
        rc, out, act = policy_call(obs_d, wd, noise_d, n=n)
        assert rc == 0, lib().shipsim_last_error()
        runs[n] = (out.cpu().numpy(), act.cpu().numpy())
    return dict(name=request.param, w=w, wd=wd, obs=obs, noise=noise, obs_d=obs_d, noise_d=noise_d, ref=ref, sigma=sigma, S=S,
                runs=runs)


def test_policy_matches_float64_at_every_grid_shape(policy_case):
    c = policy_case
    worst = 0.0
    for n, (out, _) in c["runs"].items():
        ratio = np.abs(out[:n].astype(np.float64) - c["ref"][:n]) / c["sigma"][:n]
        bad = ~(ratio <= 4.0)                                 # (NaN: a row the kernel did not write)
        assert not bad.any(), "%s n=%d: %d outputs beyond 4 sigma, first (row, col) %s, max ratio %g" % (
            c["name"], n, bad.sum(), np.argwhere(bad)[0], np.nanmax(ratio))
        worst = max(worst, float(ratio.max()))
    print("policy %s: largest |kernel - float64| / sigma = %.3f" % (c["name"], worst))


def test_policy_writes_rows_below_n_and_nothing_past_them(policy_case):
    c = policy_case
    for n, (out, act) in c["runs"].items():
        assert_sentinels(torch.from_numpy(out), torch.from_numpy(act), n, "%s n=%d" % (c["name"], n))


def test_policy_rows_do_not_depend_on_tile_slot_pass_or_cta(policy_case):
    """out(n)[:m] == out(m) bit for bit; permuting the rows permutes the outputs bit for bit."""
    c = policy_case
    S = c["S"]
    n = 2 * S + 37
    big, big_act = c["runs"][n]
    for m in (1, 17, S, S + 1):
        out, act = c["runs"][m]
        assert np.array_equal(big[:m].view(np.int32), out[:m].view(np.int32)) and np.array_equal(big_act[:m], act[:m]), m
    perm = torch.from_numpy(np.random.RandomState(5).permutation(n)).cuda()
    rc, out, act = policy_call(c["obs_d"][:n][perm].contiguous(), c["wd"], c["noise_d"][:n][perm].contiguous())
    assert rc == 0
    p = perm.cpu().numpy()
    assert np.array_equal(out[:n].cpu().numpy().view(np.int32), big[:n][p].view(np.int32))
    assert np.array_equal(act[:n].cpu().numpy(), big_act[:n][p])


def test_policy_action_is_the_float64_argmax_wherever_the_margin_is_clear(policy_case):
    """Where the float64 top-two margin of logit + noise exceeds 8 sigma (each logit within 4 sigma) plus the fp32
    rounding of the two sums, the kernel's action is the float64 argmax."""
    c = policy_case
    for n, (_, act) in c["runs"].items():
        z = c["ref"][:n, :3] + c["noise"][:n].astype(np.float64)
        top = np.sort(z, 1)
        clear = top[:, 2] - top[:, 1] > 8 * c["sigma"][:n, :3].max(1) + 2 * U * np.abs(z).max(1)
        if n >= 1000:
            assert clear.mean() > 0.99, (n, clear.mean())
        assert np.array_equal(act[:n][clear], z.argmax(1)[clear]), n


def test_policy_exact_ties_go_to_the_first_maximum_and_noise_decides():
    """Identical head columns and biases, zero noise: logits tie exactly, and the first of the tied actions wins.  A
    large noise on one action forces it."""
    rng = np.random.RandomState(3)
    _, w = policy_weights(4)
    S, _ = shapes()
    n = S + 1
    obs = cuda(env_obs(rng, n))
    w["w3"][:64, 1] = w["w3"][:64, 2] = w["w3"][:64, 0]
    b = w["b3"][0]
    for b3, want in (((b, b, b - 100), 0), ((b - 100, b, b), 1), ((b, b, b), 0)):
        w["b3"][:3] = b3
        rc, out, act = policy_call(obs, {k: cuda(v) for k, v in w.items()}, torch.zeros(n, 3, device="cuda"))
        assert rc == 0
        tied = [i for i in range(3) if b3[i] == max(b3)]
        assert torch.equal(out[:n, tied[0]].view(torch.int32), out[:n, tied[-1]].view(torch.int32))     # the tie is exact
        assert bool((act[:n] == want).all()), (b3, torch.bincount(act[:n]))
    _, w = policy_weights(4)
    wd = {k: cuda(v) for k, v in w.items()}
    for a in range(3):
        noise = torch.zeros(n, 3, device="cuda")
        noise[:, a] = 1e4
        rc, _, act = policy_call(obs, wd, noise)
        assert rc == 0 and bool((act[:n] == a).all()), a


def tanh_probe_weights(B):
    """Weights under which every operation of the kernel except the layer-2 tanh is exact: input k (+-1000) drives unit
    k of both trunks to tanh(+-1000) = +-1; unit j_o (o < 3: policy units 0..2, o = 3: value unit 0) sums inputs
    k < 23 with weights +-2^(k - 20) (output 1 with the opposite sign) onto its bias B[o], a multiple of 2^-20 in
    [-8, 8]; one-hot heads copy tanh(y2) to the four outputs."""
    w = {k: np.zeros(s, np.float32) for k, s in (("w1", (32, 128)), ("b1", 128), ("w2", (2, 64, 64)), ("b2", 128), ("w3", (128, 4)),
                                                  ("b3", 4))}
    k = np.arange(32)
    w["w1"][k, k] = w["w1"][k, 64 + k] = 1.0
    p2 = np.ldexp(1.0, np.arange(23) - 20).astype(np.float32)
    w["w2"][0, :23, 0], w["w2"][0, :23, 1], w["w2"][0, :23, 2], w["w2"][1, :23, 0] = p2, -p2, p2, p2
    w["b2"][[0, 1, 2, 64]] = B
    w["w3"][[0, 1, 2, 64], [0, 1, 2, 3]] = 1.0
    return w


def test_tanh_sfu_accuracy_and_saturation():
    """At least 10^6 arguments of the layer-2 tanh, exact multiples of 2^-20 in [-16, 16] (0 and +-2^-20 included):
    |tanh_sfu - tanh| <= TANH_EPS, and exactly +-1 once tanh has saturated in fp32 (|x| >= 9.5)."""
    rng = np.random.RandomState(8)
    n = 1 << 18
    q = np.concatenate([np.arange(-4095, 4096, 2), 2 * rng.randint(-(1 << 22), 1 << 22, n - 4096) + 1])      # odd: S = q 2^-20
    bits = (q + (1 << 23) - 1) // 2                            # sum_k s_k 2^k = q with s_k = +-1
    s = np.where((bits[:, None] >> np.arange(23)) & 1, 1.0, -1.0)
    obs = np.full((n, 32), 1000.0, np.float32)
    obs[:, :23] = 1000.0 * s
    S = q * 2.0 ** -20
    worst, args, zeros = 0.0, 0, 0
    for B in ((0.0, 2.0 ** -20, -8.0, 8.0), (-1.5, 1.5, -5.0, 5.0 - 2.0 ** -20)):
        w = tanh_probe_weights(np.float32(B))
        rc, out, _ = policy_call(cuda(obs), {k: cuda(v) for k, v in w.items()}, torch.zeros(n, 3, device="cuda"))
        assert rc == 0
        y = np.stack([B[0] + S, B[1] - S, B[2] + S, B[3] + S], 1)
        got = out[:n].cpu().numpy().astype(np.float64)
        err = np.abs(got - np.tanh(y))
        i = np.unravel_index(err.argmax(), err.shape)
        assert err.max() <= TANH_EPS, "tanh_sfu(%r) = %r, tanh = %r" % (y[i], got[i], np.tanh(y[i]))
        sat = np.abs(y) >= 9.5
        assert sat.any() and np.array_equal(got[sat], np.sign(y[sat])), y[sat][got[sat] != np.sign(y[sat])][:4]
        assert (got[y == 0] == 0).all()
        worst, args, zeros = max(worst, float(err.max())), args + y.size, zeros + int((y == 0).sum())
    assert args >= 10 ** 6 and zeros > 0
    print("tanh_sfu: %d arguments, largest |tanh_sfu - tanh| = %.3g" % (args, worst))


def test_policy_rejects_misaligned_buffers_before_the_launch():
    """Every buffer the kernel moves in 16-byte units (obs, w1, b1, w2, b2, w3, out) or as int64 (actions) is checked:
    4 bytes off, the call returns SHIPSIM_ERR_ARG naming the buffer and writes nothing.  b3 and noise need only float
    alignment: 4 bytes off, the call computes what the aligned one does."""
    rng = np.random.RandomState(2)
    _, w = policy_weights(5)
    n = 100
    obs, noise = env_obs(rng, n), gumbel(rng, n)
    pad = lambda a: cuda(np.concatenate([a.ravel(), np.zeros(4, np.float32)]))      # noqa: E731  (room for the shift)
    wd = {k: pad(v) for k, v in w.items()}
    obs_d, noise_d = pad(obs), pad(noise)
    rc, want, want_act = policy_call(obs_d, wd, noise_d, n=n)
    assert rc == 0
    for name in ("obs", "w1", "b1", "w2", "b2", "w3", "out", "actions"):
        rc, out, act = policy_call(obs_d, wd, noise_d, n=n, shift={name: 4})
        assert rc == -1 and ("dev_" + name).encode() in lib().shipsim_last_error(), name
        assert bool((out.view(torch.int32) == SENTINEL_BITS).all()) and bool((act == -7).all()), name
    for name in ("b3", "noise"):
        src = wd if name == "b3" else {"noise": noise_d}
        moved = torch.zeros_like(src[name])
        moved[1:] = src[name][:-1]                            # the same values, one float further on
        kw = dict(wd, b3=moved) if name == "b3" else dict(wd)
        rc, out, act = policy_call(obs_d, kw, moved if name == "noise" else noise_d, n=n, shift={name: 4})
        assert rc == 0, name
        assert torch.equal(out.view(torch.int32), want.view(torch.int32)) and torch.equal(act, want_act), name


def test_policy_on_two_devices_in_one_process():
    """The kernel's shared-memory opt-in and its grid size are per device: cuda:0, then cuda:1, each against float64."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two visible devices")
    rng = np.random.RandomState(9)
    _, w = policy_weights(6)
    for d in (0, 1):
        dev = torch.device("cuda", d)
        n = 2 * slots_per_pass(d) + 37
        obs, noise = env_obs(rng, n), gumbel(rng, n)
        ref, sigma = mlp_forward64(obs, **w)
        rc, out, act = policy_call(cuda(obs, dev), {k: cuda(v, dev) for k, v in w.items()}, cuda(noise, dev))
        assert rc == 0, (d, lib().shipsim_last_error())
        assert_sentinels(out, act, n, "cuda:%d" % d)
        assert (np.abs(out[:n].cpu().numpy() - ref) <= 4 * sigma).all(), d


# ---------------------------------------------------------------------------------------------- GAE
GAMMA_LAM = [(0.99, 0.95), (1.0, 1.0), (0.99, 0.0), (0.0, 0.95)]
GAE_SHAPES = [(T, N) for T in (1, 2, 128, 1024) for N in (1, 255, 257, 65537)]


def done_patterns(rng, T, N):
    """Done rates 0, 0.05 and 1, and dones at t = 0 and t = T - 1 only (the largest shape: rate 0.05 with both edges)."""
    edges = np.zeros((T, N), np.uint8)
    edges[0] = edges[T - 1] = 1
    sparse = (rng.rand(T, N) < 0.05).astype(np.uint8)
    if T * N > 1 << 24:
        sparse[0], sparse[T - 1] = 1, rng.rand(N) < 0.5
        return {"0.05+edges": sparse}
    return {"0": np.zeros((T, N), np.uint8), "0.05": sparse, "1": np.ones((T, N), np.uint8), "edges": edges}


def gae_call(rew, val, done, gamma, lam):
    T, N = rew.shape
    adv = torch.full((T, N), float("nan"), device="cuda")
    ret = torch.full((T, N), float("nan"), device="cuda")
    rc = lib().shipsim_gae(rew.data_ptr(), val.data_ptr(), done.data_ptr(), T, N, gamma, lam, adv.data_ptr(), ret.data_ptr(),
                           torch.cuda.current_stream().cuda_stream)
    assert rc == 0, lib().shipsim_last_error()
    return adv, ret


@pytest.mark.parametrize("T,N", GAE_SHAPES)
def test_gae_within_the_float64_bound(T, N):
    """adv and ret of shipsim_gae within gae64's bound at every (gamma, lam) and done pattern; a column subset run on its
    own gives the same bits."""
    rng = np.random.RandomState(T * 7 + N)
    rew = rng.choice(np.float32([1.0, -1.0, -0.01]), size=(T, N), p=[0.05, 0.05, 0.9])
    val = (rng.randn(T + 1, N) * 10).astype(np.float32)
    rew_d, val_d = cuda(rew), cuda(val)
    worst = 0.0
    for pname, done in done_patterns(rng, T, N).items():
        done_d = cuda(done)
        for gamma, lam in GAMMA_LAM:
            adv, ret = gae_call(rew_d, val_d, done_d, gamma, lam)
            a64, r64, ba, br = gae64(rew, val, done, gamma, lam)
            ea = np.abs(adv.cpu().numpy() - a64)
            er = np.abs(ret.cpu().numpy() - r64)
            ok_a, ok_r = ea <= ba, er <= br                       # (NaN: an element the kernel did not write)
            assert ok_a.all() and ok_r.all(), "done %s, gamma %g, lam %g: %d adv / %d ret beyond the bound, max ratio %g" % (
                pname, gamma, lam, (~ok_a).sum(), (~ok_r).sum(), np.nanmax(ea / ba))
            worst = max(worst, float((ea / ba).max()), float((er / br).max()))
        # the columns of a subset, on their own, give the same bits
        c0, c1 = N // 3, N // 3 + max(1, N // 2)
        sub_a, sub_r = gae_call(rew_d[:, c0:c1].contiguous(), val_d[:, c0:c1].contiguous(), done_d[:, c0:c1].contiguous(), 0.99, 0.95)
        adv, ret = gae_call(rew_d, val_d, done_d, 0.99, 0.95)
        assert torch.equal(sub_a.view(torch.int32), adv[:, c0:c1].view(torch.int32)), pname
        assert torch.equal(sub_r.view(torch.int32), ret[:, c0:c1].view(torch.int32)), pname
    print("gae T=%d N=%d: largest |kernel - float64| / bound = %.3g" % (T, N, worst))


# ---------------------------------------------------------------------------------------------- scored GAE
def scored_env(n, cap):
    from helpers import fp32_bank, knobs, make_env
    env = make_env(knobs(max_steps=8), n, fp32_bank(N_SCEN, 600, 600, seed=13), seed=3)
    env.enable_episode_log(cap)
    env.reset()
    torch.cuda.synchronize()
    return env


@pytest.mark.parametrize("T,N,steps_per_call,p_done,over_capacity", [
    (23, 997, 1, 0.25, False),
    (23, 997, 4, 0.25, False),
    (23, 997, 7, 0.25, False),
    (64, 8192, 4, 0.7, False),                      # more than 1,184 x 256 records: the scatter's grid-stride loop runs twice
    (23, 997, 7, 0.25, True),                       # count above the log's capacity: the records past it are lost
])
def test_scored_gae_on_synthetic_episode_logs(T, N, steps_per_call, p_done, over_capacity):
    """The scored GAE on records written straight into the env's episode log (call0 = 1000) and the scenario of the
    running episode written into the bound state: every step attributed as loop_attribution states the rule, the
    per-map sums equal a float64 fold of the kernel's own advantages, adv / ret bit-identical to shipsim_gae's.  (The
    env is not stepped afterwards: the state holds scenario ids the kernel never reads back.)"""
    from ship_sim_gym_b200 import _abi
    call0 = 1000
    rng = np.random.RandomState(T + N + steps_per_call)
    done, meta, count, rec, now, lost = synthetic_rollout(rng, T, N, N_SCEN, call0, steps_per_call, p_done=p_done)
    rec.pop(lost)
    cap = count - 100 if over_capacity else len(meta)
    if over_capacity:                                # the steps the records past the capacity ended are lost as well
        for m in meta[cap:count]:
            t = int(m[_abi.EP_CALL] - call0) * steps_per_call + int(m[_abi.EP_K])
            if 0 <= m[_abi.EP_SCENARIO] < N_SCEN:        # (a record of a scenario outside the bank is skipped anyway)
                rec.pop((t, int(m[_abi.EP_ENV])), None)
    if T * N > 1184 * 256:
        assert count > 1184 * 256
    env = scored_env(N, cap)
    log = env.episode_log
    log.meta.copy_(cuda(meta[:cap]))
    log.count.fill_(count)
    env.state[4, :, 2].view(torch.int32).copy_(cuda(now))
    torch.cuda.synchronize()
    rew = cuda((rng.randn(T, N) * 0.3).astype(np.float32))
    val = cuda((rng.randn(T + 1, N) * 10).astype(np.float32))
    done_d = cuda(done)
    adv0, ret0 = gae_call(rew, val, done_d, 0.99, 0.95)
    torch.cuda.synchronize()                         # (the scored call runs on the env's stream)
    adv, ret = torch.full_like(adv0, float("nan")), torch.full_like(ret0, float("nan"))
    scen = torch.full((T, N), -7, dtype=torch.int32, device="cuda")
    scores = torch.zeros(N_SCEN + 1, 3, dtype=torch.float64, device="cuda")
    _abi.check(env.L.shipsim_gae_scored(env._h, rew.data_ptr(), val.data_ptr(), done_d.data_ptr(), T, 0.99, 0.95, call0, steps_per_call,
                                        adv.data_ptr(), ret.data_ptr(), scen.data_ptr(), scores.data_ptr(), env._stream()))
    torch.cuda.synchronize()
    want = loop_attribution(done, rec, now)
    got = scen.cpu().numpy()
    assert np.array_equal(got, want), "%d steps attributed differently, first (t, e) %s" % ((got != want).sum(), np.argwhere(got != want)[:1])
    assert (want == -1).any()
    assert torch.equal(adv.view(torch.int32), adv0.view(torch.int32)) and torch.equal(ret.view(torch.int32), ret0.view(torch.int32))
    a = adv.double().cpu().numpy().ravel()
    row = np.where(want.ravel() >= 0, want.ravel(), N_SCEN)
    fold = np.zeros((N_SCEN + 1, 3))
    np.add.at(fold, row, np.stack([np.ones_like(a), np.maximum(a, 0.0), np.abs(a)], 1))
    s = scores.cpu().numpy()
    assert np.allclose(s, fold, rtol=1e-9, atol=1e-9 * max(1.0, np.abs(fold).max())), np.abs(s - fold).max()
    env.close()
