"""CPU: weighted scenario picks -- the independent statement of the pick rule (tests/weighted_picks.py) on the oracle's hash,
a numpy model of the device's guide-table search against it, the quantization of float weights, Prioritized Level Replay's distribution and the all-reduce that keeps every
rank's weights identical (gloo, world size 2)."""
import os
import socket
import sys

import numpy as np
import pytest
from scipy import stats

torch = pytest.importorskip("torch")

from oracle import cbind  # noqa: E402
from weighted_picks import pick_from, pick_hash, prefix_sums, weighted_pick  # noqa: E402

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def device_model_table(w):
    """The table build_pick_table_kernel (csrc/shipsim_kernels.cu) writes, by its guide formula, in numpy: (cdf, guide, total)."""
    n = len(w)
    cdf = [int(x) for x in np.cumsum(np.asarray(w, dtype=np.uint64))]
    total = cdf[-1]
    if total == 0 or total >= 1 << 32:
        return cdf, None, 0
    guide = np.zeros(n + 1, dtype=np.int64)
    for i in range(n):                                       # j in [ceil(cdf[i-1] n / total), ceil(cdf[i] n / total)) get i
        guide[-(-(cdf[i - 1] if i else 0) * n // total):-(-cdf[i] * n // total)] = i
    guide[n] = n - 1
    return cdf, guide, total


def device_model_pick(h, table):
    """pick_weighted of csrc/shipsim_device.cuh: bucket, guide range, bounded binary search."""
    cdf, guide, total = table
    j = (h * len(cdf)) >> 32
    if total == 0:
        return j
    t = (h * total) >> 32
    lo, hi = int(guide[j]), int(guide[j + 1])
    while lo < hi:
        mid = (lo + hi) // 2
        if cdf[mid] > t:
            hi = mid
        else:
            lo = mid + 1
    return lo


def test_guide_table_matches_its_definition():
    rng = np.random.RandomState(0)
    for n in (1, 2, 7, 64, 1000):
        for w in (rng.randint(0, 5, n), np.full(n, 3), np.where(rng.rand(n) < 0.8, 0, rng.randint(1, 1 << 20, n))):
            if w.sum() == 0:
                continue
            cdf = np.cumsum(w.astype(np.uint64)).astype(object)
            total = int(cdf[-1])
            want = [int(np.argmax(np.array(cdf) > (jj * total) // n)) for jj in range(n)]
            excl = [0] + list(cdf[:-1])
            got = np.zeros(n, dtype=np.int64)
            for i in range(n):
                got[-(-excl[i] * n // total):-(-cdf[i] * n // total)] = i
            assert list(got) == want, (n, w)


@pytest.mark.parametrize("n", [1, 3, 64, 1000, 1024, 65537])
def test_equal_weights_pick_what_the_uniform_pick_picks(n):
    rng = np.random.RandomState(n)
    for wv in (1, 7, (1 << 32) // n - 1):
        w = np.full(n, wv, dtype=np.uint64)
        for _ in range(200):
            seed, gid, ep = int(rng.randint(0, 1 << 62)), int(rng.randint(0, 1 << 40)), int(rng.randint(0, 1 << 20))
            assert weighted_pick(seed, gid, ep, n, w) == cbind.pick_scenario(seed, gid, ep, n)


def test_device_search_agrees_with_oracle_at_both_ends_of_the_hash_range():
    rng = np.random.RandomState(1)
    hs = [0, 1, 2, 0x7FFFFFFF, 0xFFFFFFFE, 0xFFFFFFFF] + list(rng.randint(0, 1 << 32, 300, dtype=np.uint64))
    for n in (1, 5, 97, 1024):
        for w in (rng.randint(0, 100, n), np.where(rng.rand(n) < 0.9, 0, 1), np.full(n, 1000)):
            if w.sum() == 0:
                w[-1] = 1
            cum = np.cumsum(w.astype(np.uint64))
            table = device_model_table(w)
            for h in hs:
                t = (int(h) * int(cum[-1])) >> 32
                assert device_model_pick(int(h), table) == int(np.argmax(cum > t)), (n, int(h))
    # the restated hash is the oracle's (its uniform pick), and the two statements of the rule agree on it
    w = rng.randint(0, 9, 333)
    cum = prefix_sums(w)
    table = device_model_table(w)
    for gid in list(range(200)) + [(1 << 40) + 7, (1 << 63) - 1]:
        seed, ep = (77, 0x123456789ABCDEF)[gid % 2], gid % 5
        h = pick_hash(seed, gid, ep)
        assert cbind.pick_scenario(seed, gid, ep, 333) == (h * 333) >> 32
        assert cbind.pick_scenario(seed, gid, ep, (1 << 31) - 1) == (h * ((1 << 31) - 1)) >> 32
        assert pick_from(h, cum) == device_model_pick(h, table) == int(np.argmax(cum > (h * int(cum[-1])) >> 32))


def test_zero_weights_are_never_picked_and_frequencies_follow_the_weights():
    n = 40
    rng = np.random.RandomState(2)
    w = rng.randint(1, 50, n)
    w[rng.permutation(n)[:20]] = 0
    cum = prefix_sums(w)
    picks = np.array([pick_from(pick_hash(9, g, ep), cum) for g in range(2000) for ep in range(30)])
    counts = np.bincount(picks, minlength=n)
    assert (counts[w == 0] == 0).all()
    expect = picks.size * w / w.sum()
    chi2 = stats.chisquare(counts[w > 0], expect[w > 0])
    assert chi2.pvalue > 1e-4, chi2


def test_zero_or_overflowing_total_is_uniform():
    n = 50
    for w in (np.zeros(n, dtype=np.uint64), np.full(n, (1 << 32) // n + 1, dtype=np.uint64)):
        for g in range(300):
            assert weighted_pick(3, g, g % 7, n, w) == cbind.pick_scenario(3, g, g % 7, n)


def test_weighted_oracle_stepping_with_equal_weights_is_the_oracles_own_auto_reset():
    """oracle_step_weighted (explicit resets of the finished envs) reproduces the oracle's in-step auto-reset bit for bit
    when the weights pick what the uniform pick picks; with skewed weights no zero-weight map is played."""
    import oracle
    from ship_sim_gym_b200 import ScenarioBank
    from weighted_picks import oracle_step_weighted
    bank = ScenarioBank.generate(12, (600, 600), seed=4).as_dict()
    n, K = 64, 60
    acts = np.random.RandomState(0).randint(0, 3, (K, n)).astype(np.int32)
    kw = dict(max_steps=9, seed=5, env_id_offset=1000)
    ref = oracle.OracleEnv(n, bank, auto_reset=True, **kw)
    got = oracle.OracleEnv(n, bank, auto_reset=False, **kw)
    ref.reset()
    got.reset()
    a = ref.step(acts)
    b = oracle_step_weighted(got, acts, np.full(12, 5))
    assert a["done"].sum() > n
    for key in a:
        assert np.array_equal(a[key], b[key]), key
    assert np.array_equal(ref.ints, got.ints) and np.allclose(ref.stats, got.stats, rtol=1e-12)      # (sums: order of additions)
    w = np.zeros(12, dtype=np.int64)
    w[[1, 4, 9]] = [3, 1, 7]
    oracle_step_weighted(got, acts, w)
    assert set(np.unique(got.ints[:, 3])) <= {1, 4, 9}


def test_quantization_keeps_the_sum_below_2_31_and_positive_weights_positive():
    from ship_sim_gym_b200.env import quantize_scenario_weights
    rng = np.random.RandomState(3)
    cases = [torch.tensor(rng.rand(1000) * 1e30), torch.tensor([1e-300, 1.0, 0.0, 1e300]), torch.ones(7),
             torch.tensor([float("nan"), -5.0, float("inf"), 2.0, 1e-12]), torch.zeros(5), torch.rand(1 << 20, dtype=torch.float64)]
    for w in cases:
        q = quantize_scenario_weights(w)
        assert q.dtype == torch.int32 and q.shape == w.shape
        qs = q.long()
        assert int(qs.sum()) <= 1 << 31 and int(qs.min()) >= 0
        pos = torch.nan_to_num(w.double(), nan=0.0) > 0
        assert bool((qs[pos] >= 1).all()) and bool((qs[~pos] == 0).all())
    q = quantize_scenario_weights(torch.full((1024,), 0.37))
    assert len(set(q.tolist())) == 1                                   # equal stays equal: the uniform picks
    q = quantize_scenario_weights(torch.tensor([1.0, 2.0, 4.0]))
    assert q[1] == 2 * q[0] and abs(int(q[2]) - 2 * int(q[1])) <= 1


def test_fold_episode_log_masks_by_the_device_count():
    from ship_sim_gym_b200 import _abi
    from ship_sim_gym_b200.env import OUTCOME_COLUMNS, fold_episode_log
    meta = torch.zeros(6, 8, dtype=torch.int32)
    rec = [(2, 1.5, 10, _abi.END_COLLISION), (0, -0.5, 20, _abi.END_TIMEOUT), (2, 0.5, 30, _abi.END_ALL_GOALS | _abi.END_GOAL),
           (1, 2.0, 40, _abi.END_OOB), (3, 9.0, 50, _abi.END_COLLISION)]     # the last one lies past the count
    for r, (s, ret, ln, end) in enumerate(rec):
        meta[r, _abi.EP_SCENARIO], meta[r, _abi.EP_LENGTH], meta[r, _abi.EP_END] = s, ln, end
        meta[r, _abi.EP_RETURN] = torch.tensor([ret], dtype=torch.float32).view(torch.int32)[0]
    meta[5, _abi.EP_SCENARIO] = 1 << 30                                        # garbage past the count
    t = fold_episode_log(meta, torch.tensor([4], dtype=torch.int32), 4)
    assert t.shape == (4, len(OUTCOME_COLUMNS))
    want = np.zeros((4, 7))
    want[2] = [2, 2.0, 40, 1, 1, 0, 0]
    want[0] = [1, -0.5, 20, 0, 0, 0, 1]
    want[1] = [1, 2.0, 40, 0, 0, 1, 0]
    assert np.array_equal(t.numpy(), want)
    fold_episode_log(meta, torch.tensor([5], dtype=torch.int32), 4, out=t)       # accumulates
    assert t[3, 0] == 1 and t[2, 0] == 4


def test_replay_distribution_hand_computed_case():
    from ship_sim_gym_b200.curriculum import replay_distribution
    f64 = dict(dtype=torch.float64)
    score = torch.tensor([0.0, 5.0, 1.0, 2.0], **f64)
    played = torch.tensor([True, True, False, True])
    last = torch.tensor([3.0, 1.0, 0.0, 3.0], **f64)
    # ranks: map 2 (never played) 1, then by score: map 1 -> 2, map 3 -> 3, map 0 -> 4.  beta = 0.5: (1/rank)^2
    p = replay_distribution(score, played, last, torch.tensor(4.0, **f64), rho=0.25, beta=0.5)
    ps = np.array([1 / 16, 1 / 4, 1.0, 1 / 9])
    ps /= ps.sum()
    st = np.array([1.0, 3.0, 4.0, 1.0]) / 9.0
    assert np.allclose(p.numpy(), 0.75 * ps + 0.25 * st, rtol=1e-12) and p.sum().item() == pytest.approx(1.0)
    # nothing played yet: all maps share rank 1, staleness is uniform -> uniform
    p = replay_distribution(torch.zeros(5, **f64), torch.zeros(5, dtype=torch.bool), torch.zeros(5, **f64), torch.tensor(0.0, **f64))
    assert np.allclose(p.numpy(), 0.2)


class _FakeEnv(object):
    """What LevelReplay needs of a BatchedShipEnv, on the CPU: a per-map outcome table per update and the weights it sets."""

    def __init__(self, n, outcomes):
        self.n_scenarios, self.device, self.episode_log = n, torch.device("cpu"), object()
        self._outcomes = list(outcomes)
        self.weights = None

    def scenario_outcomes(self, clear=True):
        return self._outcomes.pop(0).clone()

    def set_scenario_weights(self, w):
        from ship_sim_gym_b200.env import quantize_scenario_weights
        self.weights = quantize_scenario_weights(w)


def _rank_outcomes(rank, n, rounds):
    rng = np.random.RandomState(100 + rank)
    out = []
    for _ in range(rounds):
        t = np.zeros((n, 7))
        ep = rng.randint(0, 3, n) * (rng.rand(n) < 0.5)
        t[:, 0] = ep
        t[:, 1] = ep * rng.randn(n)
        out.append(torch.tensor(t))
    return out


def _worker(rank, world, port, n, rounds, q):
    sys.path.insert(0, ROOT)
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    import torch.distributed as dist
    from ship_sim_gym_b200 import LevelReplay
    from ship_sim_gym_b200 import dist as sdist
    sdist.init("gloo")

    def all_reduce(t):
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return t
    env = _FakeEnv(n, _rank_outcomes(rank, n, rounds))
    lr = LevelReplay(env, all_reduce=all_reduce)
    for _ in range(rounds):
        lr.update()
    q.put((rank, env.weights.numpy().copy(), lr.table.numpy().copy()))
    dist.barrier()
    dist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def test_gloo_world_2_ranks_hold_identical_weights():
    import torch.multiprocessing as mp
    n, rounds = 64, 4
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, n, rounds, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict((r, (w, t)) for r, w, t in (q.get(timeout=120) for _ in procs))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert np.array_equal(res[0][0], res[1][0])
    # the global table is the sum of both ranks' outcomes, and one process fed that sum computes the same weights
    total = [a + b for a, b in zip(_rank_outcomes(0, n, rounds), _rank_outcomes(1, n, rounds))]
    assert np.allclose(res[0][1], sum(t.numpy() for t in total))
    from ship_sim_gym_b200 import LevelReplay
    env = _FakeEnv(n, total)
    lr = LevelReplay(env)
    for _ in range(rounds):
        lr.update()
    assert np.array_equal(env.weights.numpy(), res[0][0])
    assert (env.weights.numpy() >= 1).all()
