"""Cost of weighted scenario picks (shipsim_scenario_weights): weights off, equal and skewed, alternating on the same handle
in one process.

  python profiles/scenario_weights_cost.py [--rounds R]

Cases: the headline (4,096 envs x 1,000 random-agent steps, window_kernel<16>), 1,048,576 envs x 32 steps (serial-in-time
kernel), the 65,536-env hard map (1000 x 1000, N = 30, width 0.9; 100 steps).  "equal": every weight 1 (the picks are the
uniform ones, but every reset searches the table); "skewed": half the bank at weight 0, the other half at Zipf-like
weights 1 / (1 + rank).  Then the table build itself (one set_scenario_weights call, device input) for banks of 1,024 and
65,536 maps.  Prints the card name and power limit first; every device time is CUDA events around launches that end in
a synchronise, median over the rounds with the spread (min - max)."""
import argparse
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np  # noqa: E402
import torch  # noqa: E402

from ship_sim_gym_b200 import BatchedShipEnv, ScenarioBank  # noqa: E402
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


def weights(n, mode, dev):
    if mode == "equal":
        return torch.ones(n, device=dev)
    rng = np.random.RandomState(0)
    w = np.zeros(n)
    keep = rng.permutation(n)[: n // 2]
    w[keep] = 1.0 / (1.0 + np.arange(len(keep)))
    return torch.tensor(w, device=dev)


def kernel_case(name, env, K, reps, rounds):
    modes = ("off", "equal", "skewed")
    t = {m: [] for m in modes}
    w = {m: weights(env.n_scenarios, m, env.device) for m in modes[1:]}
    for _ in range(rounds):
        for m in modes:
            env.set_scenario_weights(None if m == "off" else w[m])
            t[m].append(launch_ms(env, K, reps))
    env.set_scenario_weights(None)
    info = env.launch_info()
    kern = "window_kernel<T=%d>" % info["steps_in_flight"] if info["steps_in_flight"] > 1 else "step_kernel<G=%d>" % info["lanes_per_env"]
    med = {m: float(np.median(v)) for m, v in t.items()}
    print("%-26s %-20s %s" % (name, kern, "  ".join("%s %.4f ms [%.4f-%.4f] (x%.4f)" % (m, med[m], min(t[m]), max(t[m]), med[m] / med["off"])
                                                   for m in modes)), flush=True)


def build_case(env, reps, rounds):
    w = weights(env.n_scenarios, "skewed", env.device)
    env.set_scenario_weights(w)
    torch.cuda.synchronize()
    t = []
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for _ in range(rounds):
        e0.record()
        for _ in range(reps):
            env.set_scenario_weights(w)
        e1.record()
        torch.cuda.synchronize()
        t.append(e0.elapsed_time(e1) / reps * 1e3)
    env.set_scenario_weights(None)
    print("%-26s quantize + table build: %.1f us [%.1f-%.1f] per set_scenario_weights" % (
        "build, %d maps" % env.n_scenarios, np.median(t), min(t), max(t)), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    a = ap.parse_args()
    print("card: %s" % card(), flush=True)
    bank = ScenarioBank.generate(1024, (600, 600), seed=0)
    env = BatchedShipEnv(4096, bank=bank, seed=0, validate_actions=False)
    env.reset()
    kernel_case("headline 4,096 x 1,000", env, 1000, 10, a.rounds)
    build_case(env, 50, a.rounds)
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
    env = BatchedShipEnv(4096, seed=0, scenario_source="device", n_scenarios=65536, validate_actions=False)
    build_case(env, 50, a.rounds)
    env.close()


if __name__ == "__main__":
    main()
