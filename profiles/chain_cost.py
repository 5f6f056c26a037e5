"""Chained against unchained window-kernel launches (BatchedShipEnv.chain_launches, shipsim_step_chained), alternating on
the same handle in one process.

  python profiles/chain_cost.py [--rounds R] [--launches L]

Cases: 2,048 envs (window_kernel<32>), the headline's 4,096 envs (window_kernel<16>) and 32,768 envs (window_kernel<8>:
more CTAs than fit the machine at once), each 1,000 steps per launch of fixed random actions on the bench's map (1,024
scenarios, 600 x 600, seed 0).  A round times L back-to-back launches with chaining on, then L with it off, with CUDA
events around launches that end in a synchronise; the table gives the median over the rounds and the spread (min - max)
of the time per launch.  Prints the card name and power limit first."""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from ship_sim_gym_b200 import BatchedShipEnv, ScenarioBank  # noqa: E402

K = 1000


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown (nvidia-smi failed)"


def timed(env, acts, out, launches, chain):
    env.chain_launches = chain
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    env.rollout(acts, out=out)              # (the first launch after a switch does not overlap anything)
    e0.record()
    for _ in range(launches):
        env.rollout(acts, out=out)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--launches", type=int, default=10)
    args = ap.parse_args()
    assert torch.cuda.is_available(), "chain_cost.py measures on the GPU"
    print("card:", card())
    dev = torch.device("cuda", 0)
    bank = ScenarioBank.generate(1024, (600, 600), seed=0)
    print("| envs | window | unchained ms / launch | chained ms / launch | chained / unchained | chained launches |")
    print("|---:|---:|---:|---:|---:|---:|")
    for n in (2048, 4096, 32768):
        env = BatchedShipEnv(n, bank=bank, seed=0, auto_reset=True, device=dev, validate_actions=False)
        env.reset()
        gen = torch.Generator(device=dev).manual_seed(0)
        acts = torch.randint(0, 3, (K, n), dtype=torch.int32, device=dev, generator=gen)
        out = env.alloc_rollout(K)
        for chain in (True, False):          # warm-up: modules loaded, both kernels run once
            timed(env, acts, out, 2, chain)
        c0 = env.launch_info()["chained"]
        on, off = [], []
        for _ in range(args.rounds):
            on.append(timed(env, acts, out, args.launches, True))
            off.append(timed(env, acts, out, args.launches, False))
        info = env.launch_info()
        fmt = lambda v: "%.4f [%.4f - %.4f]" % (np.median(v), min(v), max(v))     # noqa: E731
        print("| %d | %d | %s | %s | %.3f | %d of %d |" % (n, info["steps_in_flight"], fmt(off), fmt(on), np.median(on) / np.median(off),
                                                          info["chained"] - c0, args.rounds * (args.launches + 1)))
        env.close()


if __name__ == "__main__":
    main()
