"""-m gpu: chained rollouts (shipsim_step_chained, BatchedShipEnv.chain_launches).  A chained window-kernel launch starts
while the previous launch of the handle still runs, each env waiting only for its own previous launch.  Every case runs
one sequence of calls twice, with chaining on and off, and asks for the same results bit for bit: obs, reward and done
of every launch, the final state and the episode counters (the return sum up to the order of its atomic additions).
Where something between two launches must break the chain, the chained-launch count says it did."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")

from helpers import fp32_bank, knobs, make_env  # noqa: E402
import parity  # noqa: E402

N_ENVS, K, W = 3001, 96, 600           # a ragged batch (the last warp has an idle env group); episodes end within a launch


def setup(T, n=N_ENVS, seed=3):
    """(make(chain) -> a reset env at a scattered start state, actions [K, n] int32 on the device)."""
    k = knobs()
    bank = fp32_bank(48, W, W, seed=13)
    rng = np.random.RandomState(seed)
    st = parity.f32_inputs(*parity.random_states(rng, n, W, W, 48, bank["goals"], near=(bank["hull_xy"], bank["hull_n"])))
    acts = torch.tensor(rng.choice([0, 0, 1, 2], size=(K, n)).astype(np.int32), device="cuda")

    def make(chain, **kw):
        env = make_env(k, n, bank, steps_in_flight=T, seed=5, **kw)
        env.chain_launches = chain
        env.reset()
        env.set_state(*st)
        return env
    return make, acts


def finish(env, outs):
    """Outputs (numpy), final state, statistics and chained-launch count of `env` after the launches that wrote `outs`."""
    torch.cuda.synchronize()
    got = [[t.cpu().numpy() for t in o] for o in outs]
    return got, env.get_state(), env.stats_tensor().cpu().numpy().copy(), env.launch_info()["chained"]


def assert_same(a, b, label):
    (oa, sa, ta, _), (ob, sb, tb, _) = a, b
    assert len(oa) == len(ob)
    for i, (x, y) in enumerate(zip(oa, ob)):
        for name, u, v in zip(("obs", "reward", "done"), x, y):
            assert np.array_equal(u, v), "%s: launch %d %s differs at %d places" % (label, i, name, int((u != v).sum()))
    for k in ("pose", "ints", "lidar", "goals", "ep_return"):
        assert np.array_equal(sa[k], sb[k]), "%s: final state %s" % (label, k)
    counters = [0] + list(range(2, 16))         # everything but the return sum is a count
    assert np.array_equal(ta[counters], tb[counters]), label + ": statistics counters"
    assert ta[1] == pytest.approx(tb[1], rel=1e-12), label + ": return sum"


@pytest.mark.parametrize("T", [8, 16, 32])
@pytest.mark.parametrize("outs", ["one_out", "distinct_outs", "random_agent"])
def test_chained_rollouts_match_unchained(T, outs):
    """Six rollouts back to back: five of them chain onto their predecessor."""
    make, acts = setup(T)
    a = None if outs == "random_agent" else acts

    def go(chain):
        env = make(chain)
        bufs = [env.alloc_rollout(K)] * 6 if outs == "one_out" else [env.alloc_rollout(K) for _ in range(6)]
        for o in bufs:
            env.rollout(a, K=K, out=o)
        return finish(env, bufs[-1:] if outs == "one_out" else bufs)

    ref, got = go(False), go(True)
    assert ref[3] == 0 and got[3] == 5
    assert_same(got, ref, "T=%d %s" % (T, outs))
    assert got[2][0] > 0                      # episodes finished inside the launches


BREAKS = {
    # an in-place edit of the actions: a new _version of the same tensor
    "actions_edited": lambda env, acts, o: acts[:, :7].fill_(1),
    "set_state": lambda env, acts, o: env.set_state(*env.get_state().values()),
    "reset": lambda env, acts, o: env.reset(),
    # fewer steps than a window: the serial-in-time kernel runs in between (steps_in_flight 16 -> 1 -> 16).  With the
    # random agent on both sides, so that the library, not the Python layer, has to see it.
    "short_launch": lambda env, acts, o: env.rollout(None, K=5, out=tuple(t[:5] for t in o)),
}


@pytest.mark.parametrize("brk", list(BREAKS))
def test_chain_breaks(brk):
    """launch, something that must break the chain, launch: nothing chains, and the results are those of the unchained
    sequence."""
    make, acts0 = setup(16)

    def go(chain):
        env, acts = make(chain), acts0.clone()
        a = None if brk == "short_launch" else acts
        bufs = [env.alloc_rollout(K) for _ in range(2)]
        env.rollout(a, K=K, out=bufs[0])
        BREAKS[brk](env, acts, bufs[0])
        env.rollout(a, K=K, out=bufs[1])
        return finish(env, bufs)

    ref, got = go(False), go(True)
    assert got[3] == 0
    assert_same(got, ref, brk)


def test_two_envs_alternating_on_one_stream_do_not_chain():
    """Two envs take turns on one stream and write one `out`: overlapping a launch with the other env's would race on
    the buffer, so neither chains."""
    make, acts = setup(16)

    acts_b = acts.flip(0).contiguous()

    def go(chain):
        a, b = make(chain), make(chain)
        out = a.alloc_rollout(K)
        for _ in range(3):
            a.rollout(acts, out=out)
            b.rollout(acts_b, out=out)
        return finish(a, [out]), finish(b, [out])

    (ra0, rb0), (ra1, rb1) = go(False), go(True)
    assert ra1[3] == 0 and rb1[3] == 0
    assert_same(ra1, ra0, "env a")
    assert_same(rb1, rb0, "env b")


def test_captured_rollouts_do_not_chain_and_replay_unchained_results():
    """A stream that is being captured into a CUDA graph never chains (the graph has no previous launch to overlap); the
    replayed graph gives the results of the same launches run eagerly without chaining."""
    make, acts = setup(16)
    ref_env = make(False, validate_actions=False)
    ref_bufs = [ref_env.alloc_rollout(K) for _ in range(3)]
    for o in ref_bufs:
        ref_env.rollout(acts, out=o)
    ref = finish(ref_env, ref_bufs)

    env = make(True, validate_actions=False)         # (no host check of the actions inside the capture)
    bufs = [env.alloc_rollout(K) for _ in range(3)]
    torch.cuda.synchronize()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        for o in bufs:
            env.rollout(acts, out=o)
    assert env.launch_info()["chained"] == 0
    g.replay()
    got = finish(env, bufs)
    assert got[3] == 0
    assert_same(got, ref, "captured")
