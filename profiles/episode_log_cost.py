"""Cost of the episode log (shipsim_episode_log_bind): log off vs on, alternating on the same handle in one process.

  python profiles/episode_log_cost.py [--rounds R]

Cases: the headline (4,096 envs x 1,000 random-agent steps, window_kernel<16>), 1,048,576 envs x 32 steps (serial-in-time
kernel), the 65,536-env hard map (1000 x 1000, N = 30, width 0.9, 180-degree fan; 100 steps), the 1,024-env ShipVecEnv
step rate (numpy caller) with episode_info off and on, and the two ways a numpy caller can fetch a step's records.  Prints the card name and power limit first; every device time is
CUDA events around launches that end in a synchronise, median over the rounds with the spread (min - max)."""
import argparse
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from ship_sim_gym_b200 import BatchedShipEnv, ScenarioBank  # noqa: E402
from ship_sim_gym_b200.adapters import ShipVecEnv  # noqa: E402
from ship_sim_gym_b200.config import EnvConfig, GameConfig  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 else "unknown (nvidia-smi failed)"


def launch_ms(env, K, reps):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    out = env.alloc_rollout(K)
    env.rollout(None, K=K, out=out)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(reps):
        env.rollout(None, K=K, out=out)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def kernel_case(name, env, K, reps, rounds):
    cap = env.num_envs * K // 2
    t = {"off": [], "on": []}
    eps = 0
    for _ in range(rounds):
        for mode in ("off", "on"):
            env.enable_episode_log(cap if mode == "on" else 0)
            t[mode].append(launch_ms(env, K, reps))
            if mode == "on":
                eps = int(env.episode_log.count.item())
                env.episode_log.clear()
    env.enable_episode_log(0)
    info = env.launch_info()
    kern = "window_kernel<T=%d>" % info["steps_in_flight"] if info["steps_in_flight"] > 1 else "step_kernel<G=%d>" % info["lanes_per_env"]
    med = {m: float(np.median(v)) for m, v in t.items()}
    print("%-34s %-20s off %.4f ms [%.4f-%.4f]  on %.4f ms [%.4f-%.4f]  on/off %.4f  (%d episodes per launch, %.2f per 1k env-steps)"
          % (name, kern, med["off"], min(t["off"]), max(t["off"]), med["on"], min(t["on"]), max(t["on"]), med["on"] / med["off"],
             eps // (reps + 1), 1000.0 * eps / ((reps + 1) * env.num_envs * K)), flush=True)


def vec_case(n, steps, rounds):
    rate = {"off": [], "on": []}
    vecs = {m: ShipVecEnv(n, episode_info=(m == "on"), seed=1, validate_actions=False) for m in ("off", "on")}
    rng = np.random.RandomState(0)
    acts = rng.randint(0, 3, (steps, n))
    for v in vecs.values():
        v.reset()
        for i in range(50):
            v.step(acts[i])
    for _ in range(rounds):
        for m, v in vecs.items():
            t0 = time.perf_counter()
            for i in range(steps):
                v.step(acts[i])
            rate[m].append(steps / (time.perf_counter() - t0))
    med = {m: float(np.median(r)) for m, r in rate.items()}
    print("%-34s off %.0f steps/s [%.0f-%.0f] (%.1f us)  on %.0f steps/s [%.0f-%.0f] (%.1f us)"
          % ("ShipVecEnv %d envs, numpy step" % n, med["off"], min(rate["off"]), max(rate["off"]), 1e6 / med["off"],
             med["on"], min(rate["on"]), max(rate["on"]), 1e6 / med["on"]), flush=True)


def transport_case(n, steps, rounds):
    """How a numpy caller gets a step's records (K = 1 through step_np, the count known from the done flags): read from
    page-locked host memory the kernel wrote over PCIe (what ShipVecEnv does), or one device -> host copy after the
    step's wait."""
    t = {"none": [], "mapped": [], "copy": []}
    envs = {m: BatchedShipEnv(n, seed=1, n_scenarios=1024, validate_actions=False) for m in t}
    for m, env in envs.items():
        if m != "none":
            env.enable_episode_log(64 * n, pinned=(m == "mapped"))
        env.reset()
    rng = np.random.RandomState(0)
    acts = rng.randint(0, 3, (steps, n))
    for _ in range(rounds):
        for m, env in envs.items():
            log = env.episode_log
            used = 0
            t0 = time.perf_counter()
            for i in range(steps):
                if m != "none" and used + n > 64 * n:
                    log.clear()
                    used = 0
                obs, rew, done = env.step_np(acts[i])
                k = int(np.count_nonzero(done))
                if m == "mapped":
                    got = (log.meta.numpy()[used:used + k].copy(), log.rows.numpy()[used:used + k].copy())
                elif m == "copy" and k:
                    got = (log.meta[used:used + k].cpu().numpy(), log.rows[used:used + k].cpu().numpy())
                used += k
            t[m].append((time.perf_counter() - t0) / steps * 1e6)
    print("%-34s %s" % ("step_np %d envs + records" % n, "  ".join("%s %.1f us [%.1f-%.1f]" % (m, np.median(v), min(v), max(v)) for m, v in t.items())),
          flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    a = ap.parse_args()
    print("card: %s" % card(), flush=True)
    bank = ScenarioBank.generate(1024, (600, 600), seed=0)
    env = BatchedShipEnv(4096, bank=bank, seed=0, validate_actions=False)
    env.reset()
    kernel_case("headline 4,096 x 1,000", env, 1000, 10, a.rounds)
    env.close()
    env = BatchedShipEnv(1 << 20, bank=bank, seed=0, validate_actions=False)
    env.reset()
    kernel_case("1,048,576 x 32", env, 32, 10, a.rounds)
    env.close()

    class GC(GameConfig):
        BOUNDS = (1000, 1000)
    hbank = ScenarioBank.generate(256, (1000, 1000), seed=0, map_N=30, width_frac=0.9)
    env = BatchedShipEnv(65536, GC, EnvConfig, bank=hbank, seed=0, honour_lidar_config=True, validate_actions=False)
    env.reset()
    kernel_case("hard map 65,536 x 100", env, 100, 10, a.rounds)
    env.close()
    vec_case(1024, 2000, a.rounds)
    transport_case(1024, 2000, a.rounds)


if __name__ == "__main__":
    main()
