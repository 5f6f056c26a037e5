"""Float64 references of the policy-in-the-loop kernels (csrc/shipsim_policy.cu), in numpy on the CPU, and the synthetic
episode logs the level-score tests feed the scored GAE.

mlp_forward64 -- shipsim_mlp_policy_forward's network (include/shipsim.h layouts), with a per-output error scale sigma;
gae64 -- shipsim_gae's recurrence, with a rigorous bound on the fp32 kernel's error;
synthetic_rollout / loop_attribution -- a rollout's dones and episode-log records, and the rule that attributes every
step to a map, one env and one step at a time (shipsim_gae_scored, rollout.score_levels)."""
import numpy as np

U = 2.0 ** -24                 # fp32 unit roundoff
TANH_EPS = 4e-7                # |tanh_sfu(x) - tanh(x)|, the kernel's claim (csrc/shipsim_policy.cu)
D, H, A = 32, 64, 3            # inputs, hidden units per trunk, actions


def mlp_forward64(obs, w1, b1, w2, b2, w3, b3, tanh_eps=TANH_EPS):
    """The fused MlpPolicy in float64 on the fp32 parameters: obs [n][32], w1 [32][128] (policy | value), b1 [128],
    w2 [2][64][64] (trunk, in, out), b2 [128], w3 [128][4] (policy rows 0..63 x columns 0..2, value rows 64..127 x
    column 3), b3 [4].  -> (out [n][4] = 3 logits | value, sigma [n][4]).

    sigma is a root-sum-square model of the fp32 evaluation's error: every fp32 operation contributes u times the size of
    what it rounds, u = 2^-24, independently; every tanh adds tanh_eps; an error in a layer's input reaches its output
    through the weights (the tanh slope is at most 1).  With m the sum of the magnitudes a unit accumulates:
      v1 = eps^2 + 33 (u m1)^2,                     m1 = |b1| + |x| |W1|
      v2 = eps^2 + 65 (u m2)^2 + v1 W2^2,           m2 = |b2| + |h1| |W2|       (per trunk)
      sigma^2 = 65 (u m3)^2 + v2 W3^2,              m3 = |b3| + |h2| |W3|
    (33 and 65: the roundings of a 32- and a 64-input dot product plus bias.)"""
    f = lambda a: np.asarray(a, np.float32).astype(np.float64)      # noqa: E731
    x, w1, b1, w2, b2, w3, b3 = f(obs), f(w1), f(b1), f(w2), f(b2), f(w3), f(b3)
    n = x.shape[0]
    assert x.shape == (n, D) and w1.shape == (D, 2 * H) and w2.shape == (2, H, H) and w3.shape == (2 * H, A + 1)
    y1 = b1 + x @ w1
    h1 = np.tanh(y1)
    v1 = tanh_eps ** 2 + 33.0 * (U * (np.abs(b1) + np.abs(x) @ np.abs(w1))) ** 2
    h2 = np.empty((n, 2 * H))
    v2 = np.empty((n, 2 * H))
    for tr in range(2):
        cols = slice(tr * H, (tr + 1) * H)
        h2[:, cols] = np.tanh(b2[cols] + h1[:, cols] @ w2[tr])
        m2 = np.abs(b2[cols]) + np.abs(h1[:, cols]) @ np.abs(w2[tr])
        v2[:, cols] = tanh_eps ** 2 + 65.0 * (U * m2) ** 2 + v1[:, cols] @ (w2[tr] ** 2)
    # the heads: logits from the policy trunk, the value from the value trunk (the other entries of w3 are not read)
    wh = np.zeros_like(w3)
    wh[:H, :A], wh[H:, A] = w3[:H, :A], w3[H:, A]
    out = b3 + h2 @ wh
    var = 65.0 * (U * (np.abs(b3) + np.abs(h2) @ np.abs(wh))) ** 2 + v2 @ (wh ** 2)
    return out, np.sqrt(var)


def policy_weights(seed, l1_scale=1.0, head_scale=4.0):
    """An MlpPolicy's parameters (torch's default init, seeded) in shipsim_mlp_policy_forward's layouts, the observation
    scale folded into w1 as RolloutCollector does, layer 1 times `l1_scale` (30 saturates most of the first layer's units)
    and the heads times `head_scale` (livelier logits than the default init).  -> (module, {w1, b1, w2, b2, w3, b3})
    with the module's own weights scaled alike: module(obs) is the fp32 evaluation of the same network."""
    import torch
    from ship_sim_gym_b200.rollout import MlpPolicy
    torch.manual_seed(seed)
    policy = MlpPolicy()
    with torch.no_grad():
        for lin in (policy.pi[0], policy.vf[0]):
            lin.weight.mul_(l1_scale)
            lin.bias.mul_(l1_scale)
        for lin in (policy.pi[4], policy.vf[4]):
            lin.weight.mul_(head_scale)
    pi, vf = policy.pi, policy.vf
    t = lambda a: a.detach().numpy().astype(np.float32)           # noqa: E731
    w = dict(w1=np.concatenate([t(pi[0].weight).T, t(vf[0].weight).T], 1) * np.float32(policy.obs_scale),
             b1=np.concatenate([t(pi[0].bias), t(vf[0].bias)]),
             w2=np.stack([t(pi[2].weight).T, t(vf[2].weight).T]),
             b2=np.concatenate([t(pi[2].bias), t(vf[2].bias)]),
             w3=np.zeros((2 * H, A + 1), np.float32),
             b3=np.concatenate([t(pi[4].bias), t(vf[4].bias)]))
    w["w3"][:H, :A], w["w3"][H:, A] = t(pi[4].weight).T, t(vf[4].weight)[0]
    return policy, {k: np.ascontiguousarray(v, np.float32) for k, v in w.items()}


def env_obs(rng, n):
    """Observation rows like the env's (two frames of 16 floats: positions, speeds, lidar distances, up to the bounds of
    600), every fourth row a reset row whose older frame is 16 x -1."""
    obs = rng.uniform(-50.0, 600.0, (n, D)).astype(np.float32)
    obs[::4, :16] = -1.0
    return obs


def gumbel(rng, n):
    return -np.log(-np.log(rng.uniform(1e-10, 1.0, (n, A)))).astype(np.float32)


def gae64(rew, val, done, gamma, lam):
    """shipsim_gae in float64 on the fp32 inputs: rew [T][N], val [T + 1][N], done [T][N] -> (adv, ret, adv_bound,
    ret_bound), float64 [T][N].  gamma is the fp32 the kernel receives; gamma * lam is formed in fp32, as launch_gae
    forms it.  The bounds hold for any fp32 evaluation of the recurrence in which every operation rounds once (FMA
    contraction included):
      B_t = 4u (|r_t| + gamma |v_t+1| + |v_t| + gl nt_t |A_t+1|) + gl nt_t B_t+1,      return: B_t + u (|A_t| + |v_t|)."""
    rew = np.asarray(rew, np.float32).astype(np.float64)
    val = np.asarray(val, np.float32).astype(np.float64)
    nt = 1.0 - (np.asarray(done) != 0)
    g = float(np.float32(gamma))
    gl = float(np.float32(np.float32(gamma) * np.float32(lam)))
    T, N = rew.shape
    assert val.shape == (T + 1, N) and nt.shape == (T, N)
    adv, bound = np.empty((T, N)), np.empty((T, N))
    last, blast = np.zeros(N), np.zeros(N)
    for t in range(T - 1, -1, -1):
        delta = rew[t] + g * val[t + 1] * nt[t] - val[t]
        bnew = 4 * U * (np.abs(rew[t]) + g * np.abs(val[t + 1]) + np.abs(val[t]) + gl * nt[t] * np.abs(last)) + gl * nt[t] * blast
        last = delta + gl * nt[t] * last
        adv[t], bound[t] = last, bnew
        blast = bnew
    ret = adv + val[:T]
    return adv, ret, bound, bound + U * (np.abs(adv) + np.abs(val[:T]))


def synthetic_rollout(rng, T, N, n_scen, call0, steps_per_call=1, p_done=0.25):
    """Random dones (ends at t = 0 and t = T - 1 included) and the episode-log records of a rollout made of calls call0 ..
    of steps_per_call steps each, shuffled, plus records of other calls and garbage rows past the count.  One record is
    dropped (lost to the log's capacity).  -> dones uint8 [T, N], meta int32 [cap, 8], count, records {(t, e): scenario},
    scenario_now [N], the lost (t, e).  Needs N > 5."""
    from ship_sim_gym_b200 import _abi
    done = (rng.rand(T, N) < p_done).astype(np.uint8)
    done[0, 0] = done[T - 1, 1] = 1
    done[:, 2] = 1                                              # an env that ends on every step
    ts, es = (a.astype(np.int64) for a in np.nonzero(done))
    scen = rng.randint(n_scen, size=len(ts))
    rec = dict(zip(zip(ts.tolist(), es.tolist()), scen.tolist()))
    rows = np.zeros((len(ts), _abi.EPISODE_META), np.int32)
    rows[:, _abi.EP_K], rows[:, _abi.EP_ENV], rows[:, _abi.EP_SCENARIO] = ts % steps_per_call, es, scen
    rows[:, _abi.EP_CALL] = call0 + ts // steps_per_call
    rows[:, _abi.EP_LENGTH], rows[:, _abi.EP_EPISODE] = rng.randint(1, 50, len(ts)), rng.randint(100, size=len(ts))
    lost = (int(np.nonzero(done[:, 3])[0][0]), 3) if done[:, 3].any() else (T - 1, 1)
    rows = rows[~((ts == lost[0]) & (es == lost[1]))]
    extra = np.zeros((3, _abi.EPISODE_META), np.int32)
    for m, call in zip(extra, (call0 - 1, call0 + (T + steps_per_call - 1) // steps_per_call)):     # records of the calls before and after
        m[_abi.EP_ENV], m[_abi.EP_SCENARIO], m[_abi.EP_CALL] = 4, n_scen - 1, call
    extra[2, _abi.EP_ENV], extra[2, _abi.EP_SCENARIO], extra[2, _abi.EP_CALL] = 5, n_scen, call0    # in the rollout, a scenario outside the bank
    rows = np.concatenate([rows, extra])
    rows = rows[rng.permutation(len(rows))]
    count = len(rows)
    garbage = rng.randint(0, 3, (7, _abi.EPISODE_META)).astype(np.int32)   # past the count: must not be read
    garbage[:, _abi.EP_CALL] = call0
    meta = np.concatenate([rows, garbage])
    now = rng.randint(n_scen, size=N).astype(np.int32)
    return done, meta, count, rec, now, lost


def loop_attribution(done, rec, now):
    """The rule, one env and one step at a time: backwards from T - 1, a done at t switches to the record of (t, e)."""
    T, N = done.shape
    want = np.empty((T, N), np.int64)
    for e in range(N):
        seg = int(now[e])
        for t in range(T - 1, -1, -1):
            if done[t, e]:
                seg = rec.get((t, e), -1)
            want[t, e] = seg
    return want
