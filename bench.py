#!/usr/bin/env python
"""bench.py -- env-steps/sec of the fused ShipEnv step on B200, with roofline, CPU baseline and e2e numbers.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

One bench "step" = one pass of the hot path over one batch: a rollout of ROLLOUT (1000) consecutive env-steps of
ENVS (4096) environments in ONE persistent kernel launch, with synthetic uniform{0,1,2} actions resident in HBM
(BASELINE.json configs[1]: "default map, 4,096 batched envs on 1xB200, random actions, 1,000 steps").
N > 1 (torchrun, one rank per GPU): every rank runs that same workload on its own shard of global env ids
(weak scaling) plus ONE all-reduce of the 16-double episode-statistics vector per rollout -- the only collective
the path has.  Rank 0 prints one JSON line.
"""
import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

# Rank 0 prints ONE JSON line on stdout.  Libraries write there too (NCCL's version banner), so file descriptor 1 is
# pointed at stderr for the duration of the run and the line goes to the real stdout at the end.
_REAL_STDOUT = os.dup(1)
os.dup2(2, 1)


if os.environ.get("SHIPSIM_BENCH_WATCHDOG"):        # debugging aid: dump every thread's stack if the run is still going after N seconds
    import faulthandler
    faulthandler.dump_traceback_later(float(os.environ["SHIPSIM_BENCH_WATCHDOG"]), exit=True)


def emit(line):
    sys.stdout.flush()
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())

ENVS = 4096          # BASELINE.json configs[1]
ROLLOUT = 1000       # env-steps per launch ("1,000 steps")
N_SCENARIOS = 1024   # SURVEY.md §8(d) config 2
SEED = 0
DUMP_OBS_ENVS = 192  # --dump-outputs: observation rows of this many envs (the whole obs tensor is 524 MB)
METRIC = "env-steps/sec"
UNIT = "env-steps/s"


def b_alg(K):
    """Algorithmic HBM bytes per env-step for a K-step fused launch (SURVEY.md §8d): mandatory I/O
    action 4 + obs 128 + reward 4 + done 1 = 137, plus state read 116 + write 72 = 188 once per launch."""
    return 137.0 + 188.0 / K


def kernel_name(info):
    """The kernel the last launch ran: the time-parallel window kernel (small batches) or the serial-in-time one."""
    if info.get("steps_in_flight", 1) > 1:
        return "window_kernel<T=%d>" % info["steps_in_flight"]
    return "step_kernel<G=%d>" % info["lanes_per_env"]


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """Samples SM clock + throttle reasons with NVML while the timed region runs."""

    def __init__(self, index, period=0.002):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._halt = threading.Event()
        self._armed = False          # samples count only from arm() on (the thread starts before the barrier)
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._halt.is_set():
            if not self._armed:
                time.sleep(0.0005)
                continue
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    r = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def arm(self):
        self._armed = True

    def armed_samples(self):
        return len(self.samples)

    def stop(self):
        self._halt.set()
        self.join(timeout=2)
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ---------------------------------------------------------------------------------------------- CPU arms
def cpu_port_rate(n_envs, budget_s, threads):
    """Time the float64 C restatement of the reference (oracle/, kind "port") on the host cores: same workload
    (default map, random Philox actions, auto-reset), a bounded number of env-steps."""
    import oracle
    from ship_sim_gym_b200 import ScenarioBank
    bank = ScenarioBank.generate(N_SCENARIOS, (600, 600), seed=SEED).as_dict()
    env = oracle.OracleEnv(n_envs, bank, auto_reset=True, seed=SEED, n_threads=threads)
    env.reset()
    want = ("obs", "reward", "done")
    env.step(None, K=4, want=want)                      # warm-up + calibration
    t0 = time.perf_counter()
    env.step(None, K=8, want=want)
    per_step = (time.perf_counter() - t0) / 8
    K = max(8, min(4000, int(budget_s / max(per_step, 1e-9))))
    t0 = time.perf_counter()
    env.step(None, K=K, want=want)
    dt = time.perf_counter() - t0
    return n_envs * K / dt, K, dt


def probe_real_reference():
    """BASELINE.md section 2: is the real reference runnable here?  Needs pymunk < 6, pygame and gym importable and the
    reference package `ship_gym` on the path (`baseline/_ref/`, a driver-written install; SHIPSIM_REF_PATH overrides it
    for local experiments).  Returns (module dict, label) or (None, why-not)."""
    for d in (os.environ.get("SHIPSIM_REF_PATH"), os.path.join(ROOT, "baseline", "_ref")):
        if d and os.path.isdir(d) and d not in sys.path:
            sys.path.insert(0, d)
    os.environ.setdefault("SDL_VIDEODRIVER", "dummy")
    try:
        import pymunk
        import pygame  # noqa: F401
        import gym  # noqa: F401
        ver = str(getattr(pymunk, "version", "0"))
        if int(ver.split(".")[0]) >= 6:
            return None, "pymunk %s is >= 6 (the reference mutates a Vec2d, ship_gym/models.py:146)" % ver
        from ship_gym.config import EnvConfig, GameConfig
        from ship_gym.ship_env import ShipEnv
        return dict(ShipEnv=ShipEnv, GameConfig=GameConfig, EnvConfig=EnvConfig), "reference(pymunk %s)" % ver
    except Exception as exc:        # ModuleNotFoundError in this image
        return None, "%s: %s" % (type(exc).__name__, exc)


def _real_env_worker(conn, mods_path, seconds, stub_render, fps, speed):
    """One process = one reference ShipEnv (the SubprocVecEnv pattern of train/stable_baselines/ppo.py:122-123)."""
    mods, _ = probe_real_reference()
    gc, ec = mods["GameConfig"], mods["EnvConfig"]
    gc.SPEED, gc.FPS, gc.DEBUG = speed, fps, False
    env = mods["ShipEnv"](gc, ec)
    if stub_render:
        env.game.render = lambda *a, **k: None
    env.reset()
    n, t_end = 0, time.perf_counter() + 1.0
    while time.perf_counter() < t_end:                       # 1 s warm-up
        if env.step(env.action_space.sample())[2]:
            env.reset()
    t0 = time.perf_counter()
    while time.perf_counter() - t0 < seconds:
        if env.step(env.action_space.sample())[2]:
            env.reset()
        n += 1
    conn.send((n, time.perf_counter() - t0))


def real_reference_rates(seconds=10.0):
    """BASELINE.md section 3 rows C2-C4 with the real reference: one env uncapped (FPS=100000, train/rllib/ppo.py:13),
    the same with ShipGame.render stubbed, and one env per host core.  Only called when probe_real_reference succeeds."""
    import multiprocessing as mp
    ctx = mp.get_context("fork")

    def run(n_proc, stub):
        pipes, procs = [], []
        for _ in range(n_proc):
            a, b = ctx.Pipe()
            pr = ctx.Process(target=_real_env_worker, args=(b, None, seconds, stub, 100000, 10))
            pr.start()
            pipes.append(a)
            procs.append(pr)
        res = [c.recv() for c in pipes]
        for pr in procs:
            pr.join()
        return sum(n / dt for n, dt in res)

    cores = os.cpu_count() or 1
    return {"C2_single_uncapped": run(1, False), "C3_single_render_stubbed": run(1, True), "C4_all_cores": run(cores, False),
            "cores": cores}


def run_reference_arm(args, rank, world):
    """--impl reference: the reference's own CPU implementation of the path on the box's host cores, rank 0 only.
    When the real reference is importable (probe_real_reference) it is timed through its own public API, one ShipEnv per
    core (kind "reference"); in this image it is not (pymunk / pygame / gym absent), and the arm times the float64 C
    restatement in oracle/ (kind "port") with every host thread, on the WHOLE job's envs (ENVS x world), each step being
    a bounded sample of the rollout."""
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    mods, label = probe_real_reference()
    if mods is not None:
        per = max(2.0, min(20.0, 60.0 / max(1, args.steps + args.warmup)))
        rates = real_reference_rates(per)
        value = rates["C4_all_cores"]
        line = {
            "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": None, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic", "config": workload_config(world),
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference", "label": label,
                             "sample": "one real ShipEnv per core, %.0f s each, FPS=100000, random actions" % per,
                             "rows": rates},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
        }
        emit(line)
        return
    import oracle
    from ship_sim_gym_b200 import ScenarioBank
    n_envs = ENVS * world                       # the whole job: what `global_envs` says
    bank = ScenarioBank.generate(N_SCENARIOS, (600, 600), seed=SEED).as_dict()
    env = oracle.OracleEnv(n_envs, bank, auto_reset=True, seed=SEED, n_threads=cores)
    env.reset()
    want = ("obs", "reward", "done")
    t0 = time.perf_counter()
    env.step(None, K=4, want=want)
    per_env_step = (time.perf_counter() - t0) / 4
    total = max(1, args.steps + args.warmup)
    sample_K = max(1, min(ROLLOUT, int(60.0 / total / max(per_env_step, 1e-9))))
    for _ in range(args.warmup):
        env.step(None, K=sample_K, want=want)
    t0 = time.perf_counter()
    for _ in range(args.steps):
        env.step(None, K=sample_K, want=want)
    dt = time.perf_counter() - t0
    value = n_envs * sample_K * args.steps / dt
    sample = "%d envs x %d env-steps per bench step (of %d), auto-reset, Philox random actions" % (n_envs, sample_K, ROLLOUT)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "label": "restated-reference (no pymunk in image: %s)" % label},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "note": "reference = pure Python over pymunk/Chipmunk (not installable here); timed arm is the un-optimised float64 C "
                "restatement in oracle/ (it rebuilds the bank planes every step, but has no cffi, no pygame, no "
                "clock.tick sleep: faster than the real Python env, i.e. a conservative baseline)",
    }
    emit(line)


def workload_config(world):
    return {"workload": "default map 600x600, SPEED=10, %d envs/GPU, random actions, %d env-steps per launch "
                        "(BASELINE configs[1])" % (ENVS, ROLLOUT),
            "envs_per_gpu": ENVS, "global_envs": ENVS * world, "rollout_steps": ROLLOUT, "n_scenarios": N_SCENARIOS,
            "history": 2, "auto_reset": True, "parallelism": "env-shard x%d" % world,
            "l2": "rollout buffers (%.0f MB per launch) exceed the 126 MB L2; no explicit flush"
                  % ((ENVS * ROLLOUT * 137) / 1e6)}


# ---------------------------------------------------------------------------------------------- GPU arm
def oracle_self_check(env, actions, obs, rew, done, state0, rank, steps=64, n_check=512):
    """The headline launch itself against the float64 oracle: the first `steps` steps of the K = ROLLOUT launch that
    started from `state0`, for the first `n_check` envs (tests/parity.py tolerances: pose / lidar 1e-4 relative, reward
    and done exact away from grazing decisions).  Raises on mismatch -- a fast kernel with different results is not a
    result."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import numpy as np
    import oracle
    import parity
    n = min(n_check, env.num_envs)
    bank = env.bank.as_dict()
    orc = oracle.OracleEnv(n, bank, auto_reset=True, seed=SEED, env_id_offset=rank * ENVS)
    orc.reset()
    st = [state0[k][:n] for k in ("pose", "ints", "lidar", "goals", "ep_return")]
    parity.load_oracle_state(orc, st[0].astype(np.float64), st[1], st[2].astype(np.float64),
                             st[3].reshape(n, 10).astype(np.float64), st[4].astype(np.float64))
    a = actions[:steps, :n].cpu().numpy()
    ref = orc.step(a)
    rep = parity.compare_steps(ref, obs[:steps, :n].cpu().numpy(), rew[:steps, :n].cpu().numpy(),
                               done[:steps, :n].cpu().numpy(), margin_thr=1e-3, label="bench self-check")
    if rep["excluded_frac"] > 0.05:
        raise AssertionError("bench self-check: %.3f of the env-steps excluded as grazing" % rep["excluded_frac"])
    return {"env_steps_compared": rep["compared"], "of": rep["total"], "excluded_frac": rep["excluded_frac"],
            "max_rel_err": rep["max_rel_err"], "checker": "oracle/ (float64 C restatement), first %d steps x %d envs of a "
            "K=%d launch" % (steps, n, ROLLOUT)}


class OutputDump(object):
    """--dump-outputs: what the last timed rollout returned, as float32 .npy files (57 MB in all), so that two builds can
    be compared output for output: reward.npy and done.npy [ROLLOUT, ENVS] in full, obs.npy [ROLLOUT, DUMP_OBS_ENVS, 32]
    for a fixed, seeded sample of env indices (in increasing order).  The device buffers are allocated, and the copy
    kernels used once, before the timed region; after it take() only queues copies into them, so that nothing
    allocates, loads or waits while the clock sampler still counts; write() runs after the sampler has stopped."""

    def __init__(self, out):
        import numpy as np
        import torch
        obs, rew, done = out
        idx = np.sort(np.random.RandomState(SEED).choice(obs.shape[1], DUMP_OBS_ENVS, replace=False))
        self.idx = torch.as_tensor(idx, device=obs.device)
        self.bufs = {"obs": obs.new_empty(obs.shape[0], DUMP_OBS_ENVS, obs.shape[2]), "reward": torch.empty_like(rew),
                     "done": torch.empty_like(done)}
        self.take(out)      # the first copies load their kernels (milliseconds): not in the sampled region

    def take(self, out):
        import torch
        obs, rew, done = out
        torch.index_select(obs, 1, self.idx, out=self.bufs["obs"])
        self.bufs["reward"].copy_(rew)
        self.bufs["done"].copy_(done)

    def write(self, dirname):
        import numpy as np
        os.makedirs(dirname, exist_ok=True)
        for name, t in self.bufs.items():
            np.save(os.path.join(dirname, name + ".npy"), t.float().cpu().numpy())


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the other (non-headline) configurations")
    ap.add_argument("--no-self-check", action="store_true")
    ap.add_argument("--lanes", type=int, default=0)
    ap.add_argument("--window", type=int, default=0, help="steps_in_flight (0 = auto)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the last timed rollout's obs "
                    "(a fixed sample of envs), reward and done to DIR/<name>.npy (rank 0's envs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    args.warmup = max(args.warmup, 3 if args.impl == "ours" else 0)

    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    from ship_sim_gym_b200 import BatchedShipEnv, ScenarioBank, dist as sdist

    rank, world, local = sdist.init("nccl")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)

    bank = ScenarioBank.generate(N_SCENARIOS, (600, 600), seed=SEED)
    env = BatchedShipEnv(ENVS, bank=bank, seed=SEED, auto_reset=True, device=dev, env_id_offset=rank * ENVS,
                         lanes_per_env=args.lanes, steps_in_flight=args.window, validate_actions=False)
    env.reset()
    gen = torch.Generator(device=dev).manual_seed(SEED + rank)
    actions = torch.randint(0, 3, (ROLLOUT, ENVS), dtype=torch.int32, device=dev, generator=gen)
    out = env.alloc_rollout(ROLLOUT)
    dump = OutputDump(out) if args.dump_outputs and rank == 0 else None
    reducer = sdist.StatsReducer(dev)
    reduce_mode = os.environ.get("SHIPSIM_BENCH_REDUCE", "full")

    def one_step():
        env.rollout(actions, out=out)
        if world > 1:       # one all-reduce of the (cumulative) episode statistics per rollout; it overlaps the next rollout's kernel
            if reduce_mode == "full":
                env.stats_tensor(clear=False, out=reducer.next_buffer())
                reducer.reduce()
            elif reduce_mode == "local":
                env.stats_tensor(clear=False)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # NVML is initialised and the sampler thread started BEFORE the barrier (nvmlInit takes milliseconds, a different
    # number in every process: done after the barrier it made the ranks enter the timed region milliseconds apart)
    sampler = ClockSampler(local)
    sampler.start()
    for _ in range(args.warmup):
        one_step()
    reducer.wait_all()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = env.launch_info()["launches"]
    barrier()
    sampler.arm()
    ev0.record()
    for _ in range(args.steps):
        one_step()
    reducer.wait_all()                      # the last all-reduce belongs to the timed region
    ev1.record()
    barrier()
    ms = ev0.elapsed_time(ev1)
    launches = env.launch_info()["launches"] - l0
    # this rank's statistics as of the last all-reduced rollout (taken before anything else steps the envs)
    local_stats = env.stats_tensor(clear=False).clone()
    if dump is not None:                    # stream-ordered before anything below launches into `out` again
        dump.take(out)
    if sampler.nv is not None and sampler.armed_samples() < 5:    # region too short for NVML: extend, untimed
        t_end = time.time() + 0.5
        while time.time() < t_end:          # no collective in here: ranks run different numbers of these
            env.rollout(actions, out=out)
        torch.cuda.synchronize()
    clocks = sampler.stop()
    if dump is not None:
        dump.write(args.dump_outputs)
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item())
    env_steps = float(ENVS) * ROLLOUT * args.steps * world
    value = env_steps / (ms * 1e-3)

    # ---- the only collective of the path, checked on the GPUs: the all-reduced vector of the last rollout must equal
    # the sum of the all-gathered per-rank vectors; the printed statistics are the GLOBAL ones
    collective = None
    if world > 1 and reduce_mode == "full":
        reduced = reducer.latest().clone()
        torch.cuda.synchronize()
        ok, err, mat = sdist.verify_all_reduce(local_stats, reduced)
        collective = {"op": "all_reduce(SUM) f64[16] per rollout, NCCL", "verified": ok, "max_rel_err": err,
                      "ranks_seen": int(mat.shape[0]), "per_rank_episodes": [float(x) for x in mat[:, 0].tolist()],
                      "reducer_depth": len(reducer.bufs)}
        if not ok:
            raise AssertionError("statistics all-reduce differs from the sum of the per-rank vectors: %r" % collective)
        global_stats = reduced
    else:
        global_stats = local_stats
    stats = dict(zip(sdist_names(), [float(x) for x in global_stats.tolist()]))
    stats["steps"] = float(ENVS) * ROLLOUT * (args.steps + args.warmup) * world
    stats["scope"] = "global (all ranks)" if world > 1 else "single rank"

    # ---- roofline of the dominant kernel (the fused step kernel is the only kernel of ours in the timed region)
    peak, peak_src = load_peaks()
    launch_ms = ms / args.steps
    achieved = b_alg(ROLLOUT) * ENVS * ROLLOUT / (launch_ms * 1e-3) / 1e9
    traffic, traffic_src = None, None
    tp = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tp):
        with open(tp) as f:
            tj = json.load(f)
        traffic, traffic_src = tj.get("dram_bytes_per_launch"), "profiles/traffic.json <- " + str(tj.get("source", "ncu --set full capture"))
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "traffic": traffic,
                "traffic_source": traffic_src, "peak_source": peak_src, "kernel": kernel_name(env.launch_info()),
                "bytes_per_env_step": b_alg(ROLLOUT), "launch_ms": launch_ms}

    # ---- the headline launch against the oracle (rank 0; after the timed region)
    self_check = None
    if rank == 0 and not args.no_self_check:
        torch.cuda.synchronize()
        state0 = env.get_state()
        env.rollout(actions, out=out)
        torch.cuda.synchronize()
        self_check = oracle_self_check(env, actions, out[0], out[1], out[2], state0, rank)

    # ---- end to end through the C ABI with HOST buffers (copies inside the timed region)
    e2e = None
    pin = lambda *shape, dtype: torch.empty(*shape, dtype=dtype).pin_memory()   # noqa: E731
    h_act = pin(ROLLOUT, ENVS, dtype=torch.int32)
    h_act.copy_(actions.cpu())
    h_obs, h_rew, h_done = pin(ROLLOUT, ENVS, 32, dtype=torch.float32), pin(ROLLOUT, ENVS, dtype=torch.float32), pin(ROLLOUT, ENVS, dtype=torch.uint8)
    host_out = (h_obs.numpy(), h_rew.numpy(), h_done.numpy())
    e2e_steps = max(3, min(args.steps, 20))
    for _ in range(8):          # untimed: staging buffers, host threads, and the DMA / host-thread split settles
        env.step_host(h_act.numpy(), K=ROLLOUT, out=host_out)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        env.step_host(h_act.numpy(), K=ROLLOUT, out=host_out)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    h2d_b, d2h_b = env.host_traffic()
    e2e = {"value": float(ENVS) * ROLLOUT * e2e_steps * world / float(t.item()), "unit": UNIT,
           # counted by shipsim_step_host from the copies it issues
           "h2d_bytes_per_step": int(h2d_b), "d2h_bytes_per_step": int(d2h_b),
           "host_obs_bytes_per_step": int(h_obs.numel() * 4),
           "steps": e2e_steps, "api": "BatchedShipEnv.step_host -> shipsim_step_host (pinned host buffers)",
           "host_threads": env.host_threads()}

    # ---- other BASELINE configurations (not the headline; same kernels)
    extra = {}
    if not args.no_extra:
        extra = extra_configs(torch, dev, rank, world)
        roofline["other_configs"] = {k: {kk: v[kk] for kk in v if kk in ("env_steps_per_s", "launch_ms", "K", "roofline_frac",
                                                                        "roofline_frac_per_gpu", "kernel", "rollout_ms")}
                                     for k, v in extra.items()}

    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline:
            cores = os.cpu_count() or 1
            mods, label = probe_real_reference()
            v_all, K_all, dt_all = cpu_port_rate(ENVS, 10.0, cores)
            v_one, K_one, dt_one = cpu_port_rate(ENVS, 5.0, 1)
            cpu = {"value": v_all, "unit": UNIT, "cores": cores, "kind": "port",
                   "label": "restated-reference (%s)" % label,
                   "sample": "%d envs x %d env-steps (%.1f s), all host threads; single thread: %.3g env-steps/s "
                             "(%d env-steps, %.1f s)" % (ENVS, K_all, dt_all, v_one, K_one, dt_one),
                   "single_thread_value": v_one}
            if mods is not None:            # BASELINE.md section 3 rows C2-C4 with the real thing
                rates = real_reference_rates(10.0)
                cpu.update({"value": rates["C4_all_cores"], "kind": "reference", "label": label, "rows": rates,
                            "port_value": v_all,
                            "sample": "one real ShipEnv per core (SubprocVecEnv pattern), 10 s each, FPS=100000"})
        info = env.launch_info()
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": launch_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic", "config": workload_config(world), "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e,
            "gpu_launches": int(launches), "clocks": clocks,
            "launch_shape": {k: info[k] for k in ("lanes_per_env", "threads_per_cta", "ctas", "steps_in_flight")},
            "stats": stats, "collective": collective, "self_check": self_check, "extra": extra,
        }
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def sdist_names():
    from ship_sim_gym_b200 import _abi
    return _abi.STAT_NAMES


def extra_configs(torch, dev, rank, world):
    """Other BASELINE.json configurations, timed with the same kernels (reported under "extra" and
    roofline.other_configs, never as the headline): configs[1] stepped gym-style (K = 1, a policy in the loop cannot
    hand over 1,000 actions up front); configs[2] hard map 65,536 envs; configs[3] 1,048,576 envs sharded over the
    ranks; configs[4] policy + 16,384 envs."""
    import torch.distributed as dist
    from ship_sim_gym_b200 import BatchedShipEnv, ScenarioBank, dist as sdist
    from ship_sim_gym_b200.config import EnvConfig, GameConfig
    peak, _ = load_peaks()
    res = {}

    def timed(env, K, reps, with_allreduce):
        acts = torch.randint(0, 3, (K, env.num_envs), dtype=torch.int32, device=dev)
        out = env.alloc_rollout(K)
        reducer = sdist.StatsReducer(dev)

        def go():
            env.rollout(acts, out=out)
            if with_allreduce and world > 1:    # asynchronous: the reduction of rollout i overlaps rollout i + 1
                env.stats_tensor(clear=False, out=reducer.next_buffer())
                reducer.reduce()
        for _ in range(3):
            go()
        reducer.wait_all()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(reps):
            go()
        reducer.wait_all()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t.item()) / reps
        return ms

    bank = ScenarioBank.generate(N_SCENARIOS, (600, 600), seed=SEED)
    if rank == 0:
        # configs[1] as a gym caller sees it: one launch per env-step (the serial-in-time kernel; B_alg(1) = 325 B)
        env = BatchedShipEnv(ENVS, bank=bank, seed=SEED, device=dev, validate_actions=False)
        env.reset()
        ms = _single_rank_timed(torch, dev, env, 1, 200)
        rate = ENVS / (ms * 1e-3)
        res["default_4096_K1"] = {"env_steps_per_s": rate, "launch_ms": ms, "K": 1, "kernel": kernel_name(env.launch_info()),
                                  "roofline_frac": rate * b_alg(1) / 1e9 / peak}
        env.close()
        del env
        # configs[0] as the reference's own caller sees it: ONE env behind the gym facade (train/random.py:4-27), host in / host out
        from ship_sim_gym_b200 import ShipEnv
        fenv = ShipEnv()
        fenv.reset()
        import numpy as _np
        acts = _np.random.RandomState(SEED).randint(0, 3, 2200)
        t0 = None
        for i, a in enumerate(acts):
            if i == 200:
                t0 = time.perf_counter()
            if fenv.step(int(a))[2]:
                fenv.reset()
        dt = time.perf_counter() - t0
        res["gym_facade_1_env"] = {"env_steps_per_s": 2000 / dt, "us_per_step": dt / 2000 * 1e6,
                                   "api": "ShipEnv.step(a) -> numpy obs, float reward, bool done (shipsim_step_host, K = 1)"}
        fenv.close()
        del fenv
        # configs[1] with a new map for every episode (SURVEY section 8 f2; game.py:271-272): the device-generated bank is
        # regenerated slice by slice on a side stream, one period per 1,000-step rollout
        env = BatchedShipEnv(ENVS, n_scenarios=N_SCENARIOS, seed=SEED, device=dev, scenario_source="device", fresh_maps=True,
                             validate_actions=False)
        env.reset()
        ms = _single_rank_timed(torch, dev, env, ROLLOUT, 10)
        rate = ENVS * ROLLOUT / (ms * 1e-3)
        res["default_4096_fresh_maps"] = {"env_steps_per_s": rate, "launch_ms": ms, "K": ROLLOUT, "kernel": kernel_name(env.launch_info()),
                                          "roofline_frac": rate * b_alg(ROLLOUT) / 1e9 / peak, "fresh": env.fresh_info()}
        env.close()
        del env
        # configs[2]: builder-defined "max difficulty" map (SURVEY.md section 8d): 1000x1000, N=30, width_frac=0.9, 180 deg fan
        class GC(GameConfig):
            BOUNDS = (1000, 1000)
        hbank = ScenarioBank.generate(256, (1000, 1000), seed=SEED, map_N=30, width_frac=0.9)
        env = BatchedShipEnv(65536, GC, EnvConfig, bank=hbank, seed=SEED, honour_lidar_config=True, device=dev, validate_actions=False)
        env.reset()
        K = 100
        ms = _single_rank_timed(torch, dev, env, K, 10)
        rate = 65536 * K / (ms * 1e-3)
        res["hard_map_65536"] = {"env_steps_per_s": rate, "launch_ms": ms, "K": K, "kernel": kernel_name(env.launch_info()),
                                 "roofline_frac": rate * b_alg(K) / 1e9 / peak}
        env.close()
        del env
    # configs[3]: 1,048,576 envs sharded over the ranks, 128-step rollouts, one stats all-reduce per rollout
    total = 1048576
    off, cnt = sdist.shard(total, rank, world)
    env = BatchedShipEnv(cnt, bank=bank, seed=SEED, device=dev, env_id_offset=off, validate_actions=False)
    env.reset()
    K = 128 if world > 1 else 32       # one GPU: 1M envs x 128 steps of obs would be 17 GB; keep it modest
    ms = timed(env, K, 5, True)
    rate = total * K / (ms * 1e-3)
    res["sharded_1048576"] = {"env_steps_per_s": rate, "launch_ms": ms, "K": K, "envs_per_gpu": cnt,
                              "kernel": kernel_name(env.launch_info()),
                              "roofline_frac_per_gpu": rate / world * b_alg(K) / 1e9 / peak}
    # K=1 gym-style stepping of the same batch (one launch per env-step)
    ms1 = timed(env, 1, 50, False)
    rate1 = total / (ms1 * 1e-3)
    res["sharded_1048576_K1"] = {"env_steps_per_s": rate1, "launch_ms": ms1, "K": 1, "kernel": kernel_name(env.launch_info()),
                                 "roofline_frac_per_gpu": rate1 / world * b_alg(1) / 1e9 / peak}
    env.close()
    # configs[4]: MLP policy + 16,384 envs on the same GPU, 128-step rollouts replayed from ONE CUDA graph: no host
    # round-trip per step (rank 0 only; nothing here is the headline)
    if rank == 0:
        from ship_sim_gym_b200.rollout import MlpPolicy, RolloutCollector
        n, T = 16384, 128
        env = BatchedShipEnv(n, bank=bank, seed=SEED, device=dev, validate_actions=False)
        torch.manual_seed(SEED)
        col = RolloutCollector(env, MlpPolicy().to(dev), T=T, use_graph=True)
        col.collect()
        col.collect()
        torch.cuda.synchronize()
        reps = 5
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            col.collect()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / reps
        res["policy_rollout_16384"] = {"env_steps_per_s": n * T / (ms * 1e-3), "rollout_ms": ms, "T": T,
                                       "policy": "MlpPolicy 32-64-64 tanh (pi, vf), Gumbel-max sampling, GAE on device",
                                       "host_syncs_per_rollout": 0, "cuda_graph": True}
        env.close()
    return res


def _single_rank_timed(torch, dev, env, K, reps):
    acts = torch.randint(0, 3, (K, env.num_envs), dtype=torch.int32, device=dev)
    out = env.alloc_rollout(K)
    for _ in range(3):
        env.rollout(acts, out=out)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        env.rollout(acts, out=out)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


if __name__ == "__main__":
    main()
