"""CPU: level scores for Prioritized Level Replay -- the step-to-map attribution of rollout.score_levels against a plain
loop over the episode-log records, its per-map sums against a per-step numpy fold, LevelReplay with each of its scores,
and the all-reduce that keeps every rank's weights identical under a value-loss score (gloo, world size 2)."""
import os
import socket
import sys

import numpy as np
import pytest

torch = pytest.importorskip("torch")

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

from references import loop_attribution, synthetic_rollout  # noqa: E402


def numpy_fold(adv, scen, n_scen):
    out = np.zeros((n_scen + 1, 3))
    for t in range(adv.shape[0]):
        for e in range(adv.shape[1]):
            s = scen[t, e]
            row = s if 0 <= s < n_scen else n_scen
            a = float(adv[t, e])
            out[row] += (1.0, max(a, 0.0), abs(a))
    return out


@pytest.mark.parametrize("steps_per_call", [1, 4])
def test_attribution_and_scores_against_a_plain_loop(steps_per_call):
    from ship_sim_gym_b200 import _abi
    from ship_sim_gym_b200.rollout import score_levels
    rng = np.random.RandomState(steps_per_call)
    T, N, n_scen, call0 = 23, 41, 9, 1000
    done, meta, count, rec, now, lost = synthetic_rollout(rng, T, N, n_scen, call0, steps_per_call)
    adv = rng.randn(T, N).astype(np.float32)
    scen, scores = score_levels(torch.tensor(adv), torch.tensor(done), torch.tensor(meta), torch.tensor([count], dtype=torch.int32),
                                torch.tensor(now), call0, n_scen, steps_per_call)
    want = loop_attribution(done, {k: v for k, v in rec.items() if k != lost}, now)
    assert scen.dtype == torch.int32 and np.array_equal(scen.numpy(), want)
    assert (want[:lost[0] + 1, lost[1]] == -1).any()           # the lost record leaves steps of no known map ...
    fold = numpy_fold(adv, want, n_scen)
    assert fold[n_scen, 0] > 0                                   # ... which land in the last row
    assert np.allclose(scores.numpy(), fold, rtol=1e-12, atol=1e-12)
    assert scores[:, _abi.SCORE_STEPS].sum().item() == T * N
    # added into a given table
    again = score_levels(torch.tensor(adv), torch.tensor(done), torch.tensor(meta), torch.tensor([count], dtype=torch.int32),
                         torch.tensor(now), call0, n_scen, steps_per_call, scores=scores.clone())[1]
    assert np.allclose(again.numpy(), 2 * fold, rtol=1e-12)


def test_no_dones_and_no_records():
    from ship_sim_gym_b200.rollout import score_levels
    T, N, n_scen = 5, 3, 4
    now = torch.tensor([3, 0, 2], dtype=torch.int32)
    adv = torch.tensor([[1.0, -2.0, 0.5]] * T)
    meta = torch.zeros(6, 8, dtype=torch.int32)                  # count 0: nothing is read, whatever the rows hold
    scen, scores = score_levels(adv, torch.zeros(T, N, dtype=torch.uint8), meta, torch.zeros(1, dtype=torch.int32), now, 0, n_scen)
    assert (scen == now).all()
    want = np.zeros((n_scen + 1, 3))
    want[3], want[0], want[2] = (T, T, T), (T, 0, 2 * T), (T, T / 2, T / 2)
    assert np.array_equal(scores.numpy(), want)


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


def _outcomes(rng, n, rounds):
    out = []
    for _ in range(rounds):
        t = np.zeros((n, 7))
        ep = rng.randint(0, 3, n) * (rng.rand(n) < 0.6)
        t[:, 0] = ep
        t[:, 1] = ep * rng.randn(n)
        out.append(torch.tensor(t))
    return out


def _scores(rng, n, rounds):
    out = []
    for _ in range(rounds):
        s = np.zeros((n + 1, 3))
        steps = rng.randint(0, 40, n + 1) * (rng.rand(n + 1) < 0.7)
        s[:, 0] = steps
        s[:, 1] = steps * rng.rand(n + 1)
        s[:, 2] = s[:, 1] + steps * rng.rand(n + 1)
        out.append(torch.tensor(s))
    return out


def test_return_score_is_the_distribution_it_was():
    """score="return" (the default) folds outcomes exactly as before: minus the EMA of the mean episode return, played and
    staleness from the finished episodes; a level-score table passed to it is ignored."""
    from ship_sim_gym_b200 import LevelReplay
    from ship_sim_gym_b200.curriculum import replay_distribution
    n, rounds, alpha = 32, 5, 0.5
    outs = _outcomes(np.random.RandomState(0), n, rounds)
    a, b = _FakeEnv(n, outs), _FakeEnv(n, outs)
    lr_default, lr_return = LevelReplay(a), LevelReplay(b, score="return")
    score, played, last, clock = torch.zeros(n, dtype=torch.float64), torch.zeros(n, dtype=torch.bool), torch.zeros(n, dtype=torch.float64), 0.0
    junk = _scores(np.random.RandomState(1), n, rounds)
    for r in range(rounds):
        p = lr_default.update()
        q = lr_return.update(junk[r])
        o = outs[r]
        hit = o[:, 0] > 0
        s = -o[:, 1] / o[:, 0].clamp_min(1.0)
        score = torch.where(hit, torch.where(played, (1 - alpha) * score + alpha * s, s), score)
        played |= hit
        clock += o[:, 0].sum().item()
        last = torch.where(hit, torch.full_like(last, clock), last)
        want = replay_distribution(score, played, last, torch.tensor(clock, dtype=torch.float64))
        assert torch.equal(p, want) and torch.equal(q, want)
    assert torch.equal(a.weights, b.weights)


def test_value_loss_scores_rank_the_map_with_the_larger_mean_first():
    from ship_sim_gym_b200 import LevelReplay
    n = 4
    outcome = torch.zeros(n, 7, dtype=torch.float64)
    outcome[:, 0] = 1.0                                          # every map played: ranks come from the scores alone
    outcome[:, 1] = torch.tensor([5.0, -5.0, 0.0, 1.0])          # (the return score would rank map 1 first)
    table = torch.zeros(n + 1, 3, dtype=torch.float64)
    # steps, sum max(adv, 0), sum |adv|: map 2 has the largest mean positive advantage (0.9), map 0 the largest |adv| (2.0)
    table[:n] = torch.tensor([[10, 1.0, 20.0], [100, 30.0, 40.0], [20, 18.0, 19.0], [5, 0.5, 0.5]], dtype=torch.float64)
    table[n] = torch.tensor([50, 49.0, 49.0])                   # the unattributed row is no map's
    for name, first in (("positive_value_loss", 2), ("l1_value_loss", 0), ("return", 1)):
        lr = LevelReplay(_FakeEnv(n, [outcome]), score=name, rho=0.0)
        p = lr.update(table)
        assert int(p.argmax()) == first, (name, p)
        assert abs(p.sum().item() - 1.0) < 1e-12
    lr = LevelReplay(_FakeEnv(n, [outcome]), score="positive_value_loss", alpha=1.0)
    lr.update(table)
    assert np.allclose(lr.score.numpy(), [0.1, 0.3, 0.9, 0.1])


def test_value_loss_scores_maps_played_only_by_unfinished_episodes():
    from ship_sim_gym_b200 import LevelReplay
    n = 3
    outcome = torch.zeros(n, 7, dtype=torch.float64)
    outcome[0, 0] = 2.0                                          # one finished episode on map 0 only
    table = torch.zeros(n + 1, 3, dtype=torch.float64)
    table[0] = torch.tensor([8, 4.0, 4.0])
    table[1] = torch.tensor([4, 4.0, 6.0])                      # map 1: steps of an episode still running
    lr = LevelReplay(_FakeEnv(n, [outcome, outcome]), score="positive_value_loss", alpha=0.5)
    lr.update(table)
    assert lr.scored.tolist() == [True, True, False] and lr.played.tolist() == [True, False, False]
    assert np.allclose(lr.score.numpy(), [0.5, 1.0, 0.0]) and lr.clock.item() == 2.0
    table2 = table.clone()
    table2[1] = torch.tensor([2, 0.0, 1.0])
    lr.update(table2)                                            # EMA from the first value on
    assert np.allclose(lr.score.numpy(), [0.5, 0.5, 0.0])
    with pytest.raises(ValueError):
        lr.update()                                              # a value-loss score needs the table
    with pytest.raises(ValueError):
        LevelReplay(_FakeEnv(n, []), score="max_mc")


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
    rng = np.random.RandomState(200 + rank)
    env = _FakeEnv(n, _outcomes(rng, n, rounds))
    scores = _scores(rng, n, rounds)
    lr = LevelReplay(env, all_reduce=all_reduce, score="positive_value_loss")
    for r in range(rounds):
        mine = scores[r].clone()
        lr.update(mine)
        assert torch.equal(mine, scores[r])                      # the caller's table is not reduced in place
    q.put((rank, env.weights.numpy().copy(), lr.score.numpy().copy()))
    dist.barrier()
    dist.destroy_process_group()


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    return port


def test_gloo_world_2_ranks_hold_identical_value_loss_weights():
    import torch.multiprocessing as mp
    n, rounds = 48, 4
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, n, rounds, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict((r, (w, s)) for r, w, s in (q.get(timeout=120) for _ in procs))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    assert np.array_equal(res[0][0], res[1][0]) and np.array_equal(res[0][1], res[1][1])
    # one process fed the sums of both ranks' tables computes the same weights
    from ship_sim_gym_b200 import LevelReplay
    r0, r1 = np.random.RandomState(200), np.random.RandomState(201)
    o0, o1 = _outcomes(r0, n, rounds), _outcomes(r1, n, rounds)
    s0, s1 = _scores(r0, n, rounds), _scores(r1, n, rounds)
    env = _FakeEnv(n, [a + b for a, b in zip(o0, o1)])
    lr = LevelReplay(env, score="positive_value_loss")
    for a, b in zip(s0, s1):
        lr.update(a + b)
    assert np.array_equal(env.weights.numpy(), res[0][0])
    assert (env.weights.numpy() >= 1).all()
