"""-m gpu: bench.py prints the contract line (one JSON object: metric, value, roofline, e2e through the C ABI with host
buffers, launch count = steps, clocks) and its self-check against the oracle passes; --dump-outputs writes the last
timed rollout, the same in every run with the same arguments."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BENCH_ARGS = ["--steps", "4", "--warmup", "3", "--no-extra", "--no-cpu-baseline"]
NAMES = ("obs", "reward", "done")


def _bench(dump):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + BENCH_ARGS + ["--dump-outputs", str(dump)],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1
    return json.loads(lines[0]), {name: np.load(str(dump / (name + ".npy"))) for name in NAMES}


@pytest.fixture(scope="module")
def first_run(tmp_path_factory):
    dump = tmp_path_factory.mktemp("bench") / "outputs"
    d, arrays = _bench(dump)
    return d, arrays, dump


def test_bench_line_on_one_gpu(first_run):
    d, arrays, dump = first_run
    assert d["metric"] == "env-steps/sec" and d["unit"] == "env-steps/s" and d["n_gpus"] == 1 and d["steps"] == 4 and d["warmup"] == 3
    assert d["higher_is_better"] is True and d["scaling"] == "weak" and d["dtype"] == "f32" and d["data"] == "synthetic" and d["vs_baseline"] is None
    assert d["value"] > 1e9 and abs(d["value"] - 4096 * 1000 / (d["ms_per_step"] * 1e-3)) < 1e-6 * d["value"]
    assert d["gpu_launches"] == 4                                  # one fused launch of ours per bench step
    r = d["roofline"]
    assert r["bound"] == "hbm" and r["unit"] == "GB/s" and abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-9 and 0.05 < r["frac"] < 1.0
    assert "window_kernel" in r["kernel"] and r["bytes_per_env_step"] == pytest.approx(137.188)
    e = d["e2e"]
    assert 0 < e["value"] < d["value"] and e["h2d_bytes_per_step"] == 4096 * 1000 * 4 and e["d2h_bytes_per_step"] > 4096 * 1000 * 16
    assert d["self_check"]["env_steps_compared"] > 30000 and d["self_check"]["excluded_frac"] < 0.05
    assert d["config"]["envs_per_gpu"] == 4096 and d["config"]["rollout_steps"] == 1000 and "workload" in d["config"]
    assert d["clocks"] is None or "sm_mhz" in d["clocks"]
    # --dump-outputs: the last timed rollout's outputs, float32, 64 MB at most
    assert sorted(p.name for p in dump.iterdir()) == ["done.npy", "obs.npy", "reward.npy"]
    assert sum(p.stat().st_size for p in dump.iterdir()) <= 64 << 20
    assert all(a.dtype == np.float32 and np.isfinite(a).all() for a in arrays.values())
    assert arrays["obs"].shape == (1000, 192, 32) and arrays["reward"].shape == arrays["done"].shape == (1000, 4096)
    assert set(np.unique(arrays["done"])) <= {0.0, 1.0} and arrays["done"].any()


def test_dump_repeats_and_is_the_last_timed_rollout(first_run, tmp_path):
    """A second run with the same arguments dumps identical arrays, and they are the 7th rollout (3 warm-up + 4 timed)
    of bench.py's workload replayed here, not the one before or after it."""
    import torch
    from ship_sim_gym_b200 import BatchedShipEnv, ScenarioBank
    _, first, _ = first_run
    _, second = _bench(tmp_path / "outputs")
    for name in NAMES:
        assert np.array_equal(first[name], second[name]), name

    dev = torch.device("cuda", 0)
    bank = ScenarioBank.generate(1024, (600, 600), seed=0)
    env = BatchedShipEnv(4096, bank=bank, seed=0, auto_reset=True, device=dev, validate_actions=False)
    env.reset()
    gen = torch.Generator(device=dev).manual_seed(0)
    actions = torch.randint(0, 3, (1000, 4096), dtype=torch.int32, device=dev, generator=gen)
    envs = np.sort(np.random.RandomState(0).choice(4096, 192, replace=False))
    replay = []
    for _ in range(8):
        obs, rew, done = env.rollout(actions)
        replay.append({"obs": obs[:, envs].float().cpu().numpy(), "reward": rew.float().cpu().numpy(),
                       "done": done.float().cpu().numpy()})
    env.close()
    for name in NAMES:
        assert np.array_equal(first[name], replay[6][name]), name
    assert not np.array_equal(first["obs"], replay[5]["obs"]) and not np.array_equal(first["obs"], replay[7]["obs"])
