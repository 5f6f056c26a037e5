"""Cost of the lidar beam count (LidarConfig.N_BEAMS): n = 1, 10, 16 and 32 alternating on the same shapes in one process.

  python profiles/beam_cost.py [--rounds R]

Shapes: the headline (4,096 envs x 1,000 random-agent steps: window_kernel at 10 beams, the serial step kernel otherwise),
1,048,576 envs x 32 steps, and the hard map (1000 x 1000, N = 30, width 0.9, 180-degree fan) at 65,536 envs x 100 steps.
Every device time is CUDA events around launches that end in a synchronise: the median per launch over the rounds and
its range (min - max).  The bandwidth share divides the algorithmic traffic of a launch,
    B_alg(K, n) = 9 + 4 * (6 + n) * history + state bytes per env / K      bytes per env-step
(action, reward and done; the observation row; the env's state planes, amortised over the K steps of a launch), by the
launch time and by the device-to-device copy bandwidth measured in the same run.
Prints the card's name and power limit first."""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from ship_sim_gym_b200 import BatchedShipEnv, ScenarioBank  # noqa: E402
from ship_sim_gym_b200.config import EnvConfig, GameConfig, LidarConfig  # noqa: E402

BEAMS = (1, 10, 16, 32)


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown (nvidia-smi failed)"


def copy_bandwidth():
    """Device-to-device copy of 4 GiB (read + write: 8 GiB of traffic), best of 10, bytes/s."""
    a = torch.empty(1 << 30, dtype=torch.float32, device="cuda")
    b = torch.empty_like(a)
    b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    best = 1e30
    for _ in range(10):
        e0.record()
        b.copy_(a)
        e1.record()
        torch.cuda.synchronize()
        best = min(best, e0.elapsed_time(e1) / 1e3)
    del a, b
    torch.cuda.empty_cache()
    return 2.0 * (1 << 32) / best


def make(n, nb, bank, W, spread):
    class LC(LidarConfig):
        N_BEAMS = nb
        DISTANCE = 100
        ANGULAR_SPREAD = spread

    class EC(EnvConfig):
        LIDAR_CONFIG = LC

    class GC(GameConfig):
        BOUNDS = (W, W)
    env = BatchedShipEnv(n, GC, EC, bank=bank, seed=0, honour_lidar_config=True, validate_actions=False)
    env.reset()
    return env


def launch_ms(env, out, K, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        env.rollout(None, K=K, out=out)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def shape_case(name, n, K, bank, W, spread, reps, rounds, bw):
    envs = {nb: make(n, nb, bank, W, spread) for nb in BEAMS}
    outs = {}
    for nb, env in envs.items():
        outs[nb] = env.alloc_rollout(K)
        env.rollout(None, K=K, out=outs[nb])                # warm-up: modules loaded, shared-memory opt-in made
    torch.cuda.synchronize()
    t = {nb: [] for nb in BEAMS}
    for _ in range(rounds):
        for nb in BEAMS:
            t[nb].append(launch_ms(envs[nb], outs[nb], K, reps))
    base = float(np.median(t[10]))
    for nb in BEAMS:
        env = envs[nb]
        info = env.launch_info()
        kern = ("window_kernel<T=%d>" % info["steps_in_flight"] if info["steps_in_flight"] > 1
                else "step_kernel<G=%d,%d thr>" % (info["lanes_per_env"], info["threads_per_cta"]))
        med = float(np.median(t[nb]))
        state_per_env = env.L.shipsim_state_bytes(env._h) / n
        b_alg = 9 + 4 * (6 + nb) * env.history + state_per_env / K
        rate = n * K / (med * 1e-3)
        print("%-24s n=%-2d %-26s %9.4f ms [%.4f-%.4f]  x%.2f of 10 beams  %.3e env-steps/s  B_alg %.1f B  %.1f %% of copy bw"
              % (name, nb, kern, med, min(t[nb]), max(t[nb]), med / base, rate, b_alg, 100.0 * rate * b_alg / bw), flush=True)
    for env in envs.values():
        env.close()
    del outs
    torch.cuda.empty_cache()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=5)
    a = ap.parse_args()
    print("card: %s" % card(), flush=True)
    bw = copy_bandwidth()
    print("device-to-device copy bandwidth: %.0f GB/s" % (bw / 1e9), flush=True)
    bank = ScenarioBank.generate(1024, (600, 600), seed=0)
    shape_case("headline 4,096 x 1,000", 4096, 1000, bank, 600, 90.0, 3, a.rounds, bw)
    shape_case("1,048,576 x 32", 1 << 20, 32, bank, 600, 90.0, 3, a.rounds, bw)
    hbank = ScenarioBank.generate(256, (1000, 1000), seed=0, map_N=30, width_frac=0.9)
    shape_case("hard map 65,536 x 100", 65536, 100, hbank, 1000, 180.0, 5, a.rounds, bw)


if __name__ == "__main__":
    main()
