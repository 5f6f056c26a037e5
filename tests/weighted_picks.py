"""The weighted scenario pick (shipsim_scenario_weights) stated independently of the kernels, for the tests.

The kernels search a guide table; here the rule is a plain binary search over 64-bit prefix sums.  For the hash `h` of
(seed, global env id, episode): with total = the sum of the uint32 weights, the pick is the first i with
cum[i] > floor(h * total / 2^32); a total of 0 or of 2^32 and more means the uniform pick floor(h * n / 2^32).  The hash
is restated here and checked against the oracle's uniform pick (oracle.cbind.pick_scenario), which uses the same one.

`oracle_step_weighted` drives the unmodified float64 oracle through auto-resets under weights: it steps the oracle
without auto-reset, one step at a time, and resets the envs that finished to the weighted picks -- what the oracle's
own auto-reset does with its uniform picks (same episode number, reset observation returned for the done step)."""
import numpy as np

M32 = 0xFFFFFFFF


def mix32(x):
    x &= M32
    x ^= x >> 17; x = (x * 0xED5AD4BB) & M32; x ^= x >> 11; x = (x * 0xAC4C1B51) & M32
    x ^= x >> 15; x = (x * 0x31848BAB) & M32; x ^= x >> 14
    return x


def pick_hash(seed, gid, episode):
    seed, gid = int(seed) & ((1 << 64) - 1), int(gid) & ((1 << 64) - 1)
    k = mix32((seed & M32) ^ 0x9E3779B9)
    k = mix32(k ^ (seed >> 32))
    k = mix32(k ^ (gid & M32))
    k = mix32(k ^ (gid >> 32))
    return mix32((k + (episode & M32) * 0x9E3779B9) & M32)


def prefix_sums(weights):
    w = np.asarray(weights)
    assert w.ndim == 1 and w.min(initial=0) >= 0 and w.max(initial=0) < 1 << 32, "need uint32 weights"
    return np.cumsum(w.astype(np.uint64), dtype=np.uint64)


def pick_from(h, cum):
    """The weighted pick of hash `h` from the prefix sums `cum` (prefix_sums)."""
    n, total = len(cum), int(cum[-1])
    if total == 0 or total >= 1 << 32:
        return (h * n) >> 32
    return int(np.searchsorted(cum, np.uint64((h * total) >> 32), side="right"))


def weighted_pick(seed, gid, episode, n, weights):
    cum = prefix_sums(weights)
    assert len(cum) == n
    return pick_from(pick_hash(seed, gid, episode), cum)


def oracle_step_weighted(orc, actions, weights):
    """Step `orc` (an oracle.OracleEnv made with auto_reset=False) through actions [K, N] with auto-resets that pick by
    the uint32 `weights`.  Returns the dict of [K, N, ...] arrays orc.step returns."""
    cum = prefix_sums(weights)
    seed, off = int(orc.cfg.seed), int(orc.cfg.env_id_offset)
    steps = []
    for a in np.asarray(actions):
        out = orc.step(a)
        done = out["done"].astype(bool)
        if done.any():
            idx = np.nonzero(done)[0]
            scen = np.zeros(orc.n, dtype=np.int32)
            scen[idx] = [pick_from(pick_hash(seed, off + e, int(orc.ints[e, 4]) + 1), cum) for e in idx.tolist()]
            out["obs"] = orc.reset(mask=done, scen=scen, first=False)
        steps.append(out)
    return {k: np.stack([s[k] for s in steps]) for k in steps[0]}
