"""Cost of level scores (RolloutCollector(level_scores=True), shipsim_gae_scored): the policy-in-the-loop rollout at 16,384
envs, T = 128, MlpPolicy through the library's fused policy kernel, captured graph.

  python profiles/level_scores_cost.py [--rounds R] [--envs N] [--T T]

Three collectors on three envs of the same seed and bank alternate in one process: "off" (no episode log: the default),
"log" (episode_log=True: the log's own cost) and "scored" (level_scores=True: the log plus the scored GAE).  Then the
GAE launch alone on the scored collector's last rollout: shipsim_gae against shipsim_gae_scored (-1 fill, record scatter
and the scored GAE kernel).  Prints the card name and power limit first; every device time is CUDA events around work
that ends in a synchronise, median over the rounds with the spread (min - max)."""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from ship_sim_gym_b200 import BatchedShipEnv, ScenarioBank, _abi  # noqa: E402
from ship_sim_gym_b200.rollout import MlpPolicy, RolloutCollector  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown (nvidia-smi failed)"


def timed(fn, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def line(name, t, base=None):
    med = float(np.median(t))
    rel = "" if base is None else "  (x%.4f)" % (med / float(np.median(base)))
    print("%-34s %.4f ms [%.4f-%.4f]%s" % (name, med, min(t), max(t), rel), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--envs", type=int, default=16384)
    ap.add_argument("--T", type=int, default=128)
    ap.add_argument("--reps", type=int, default=10, help="rollouts per timed round")
    a = ap.parse_args()
    print("card: %s" % card(), flush=True)
    bank = ScenarioBank.generate(1024, (600, 600), seed=0)
    torch.manual_seed(0)
    policy = MlpPolicy().cuda()
    cols = {}
    for name, kw in (("off", {}), ("log", dict(episode_log=True)), ("scored", dict(level_scores=True))):
        env = BatchedShipEnv(a.envs, bank=bank, seed=0)
        cols[name] = RolloutCollector(env, policy, T=a.T, **kw)
        assert cols[name]._kernel
        cols[name].collect()                                # capture
        cols[name].collect()
    t = {m: [] for m in cols}
    for _ in range(a.rounds):
        for m, col in cols.items():
            t[m].append(timed(col.collect, a.reps))
    print("rollout, %d envs x T = %d (per rollout):" % (a.envs, a.T), flush=True)
    for m in cols:
        line("  " + m, t[m], t["off"] if m != "off" else None)
    torch.cuda.synchronize()
    col = cols["scored"]
    env = col.env
    ends = int(col.dones.sum())
    print("  episode ends in the last scored rollout: %d (%.2f %% of env-steps)" % (ends, 100.0 * ends / (a.T * a.envs)), flush=True)
    adv, ret = torch.empty_like(col.adv), torch.empty_like(col.returns)
    scen = torch.empty_like(col.scenarios)
    scores = torch.zeros_like(col.level_scores)
    args = (col.rewards.data_ptr(), col.values.data_ptr(), col.dones.data_ptr(), a.T)
    stream = env._stream()

    def plain():
        _abi.check(env.L.shipsim_gae(*args, a.envs, float(col.gamma), float(col.lam), adv.data_ptr(), ret.data_ptr(), stream))

    def scored():
        _abi.check(env.L.shipsim_gae_scored(env._h, *args, float(col.gamma), float(col.lam), col._call0, 1, adv.data_ptr(), ret.data_ptr(),
                                            scen.data_ptr(), scores.data_ptr(), stream))
    plain()
    scored()
    g = {"shipsim_gae": [], "shipsim_gae_scored": []}
    for _ in range(a.rounds):
        g["shipsim_gae"].append(timed(plain, 200))
        g["shipsim_gae_scored"].append(timed(scored, 200))
    print("GAE launch alone (per call):", flush=True)
    line("  shipsim_gae", g["shipsim_gae"])
    line("  shipsim_gae_scored", g["shipsim_gae_scored"], g["shipsim_gae"])
    assert torch.equal(scen, col.scenarios)


if __name__ == "__main__":
    main()
