"""BatchedShipEnv -- N ShipEnvs resident on one B200, stepped by the fused CUDA kernel through the C ABI.

Mirrors the reference interface for the path (ship_gym/ship_env.py:16-184): `reset()`, `step(actions)`,
`seed()`, `render()`, `action_space` / `observation_space` / `reward_range` / `metadata`, `n_states`,
`states_history`, the `GameConfig` / `EnvConfig` knobs, the same exceptions for the same mistakes
(AssertionError for an action outside Discrete(3), ValueError for HISTORY_SIZE < 1).  PyTorch is used only to
own device memory and streams; all arithmetic happens in libshipsim.so.
"""
import ctypes as C
import math

import numpy as np
import torch

from . import _abi
from .config import BASE_DT, SPACE_DAMPING, snapshot
from .scenario import ScenarioBank

STEP_PENALTY = -0.01          # ship_env.py:13
DEFAULT_STATE_VAL = -1        # ship_env.py:12


class Discrete(object):
    """Stand-in for gym.spaces.Discrete (gym is not a dependency): ship_env.py:19."""

    def __init__(self, n):
        self.n = n
        self.shape = ()
        self.dtype = np.int64
        self._rng = np.random.RandomState()

    def seed(self, seed=None):
        self._rng = np.random.RandomState(seed)

    def sample(self):
        return int(self._rng.randint(self.n))

    def contains(self, x):
        if isinstance(x, (int, np.integer)) and not isinstance(x, bool):
            return 0 <= int(x) < self.n
        if isinstance(x, np.ndarray) and x.shape == () and x.dtype.kind in "iu":
            return 0 <= int(x) < self.n
        return False

    def __repr__(self):
        return "Discrete(%d)" % self.n


class Box(object):
    """Stand-in for gym.spaces.Box as the reference declares it (ship_env.py:48).  Note the reference declares
    uint8 in [0, max(bounds)] but returns float64 values including -1 (SURVEY.md App. B Q15); we keep the
    declaration and return float32."""

    def __init__(self, low, high, shape, dtype):
        self.low = np.full(shape, low, dtype=np.float32)
        self.high = np.full(shape, high, dtype=np.float32)
        self.shape = tuple(shape)
        self.dtype = np.dtype(dtype)

    def __repr__(self):
        return "Box%s" % (self.shape,)


def _dtype_code(t):
    if t.dtype == torch.int32:
        return _abi.ACTION_I32
    if t.dtype == torch.int64:
        return _abi.ACTION_I64
    if t.dtype == torch.uint8:
        return _abi.ACTION_U8
    raise TypeError("actions must be int32, int64 or uint8, got %s" % t.dtype)


# why an episode ended, in the order of the outcome table's columns (END_GOAL only says a goal was taken on the last step)
END_REASONS = (_abi.END_COLLISION, _abi.END_ALL_GOALS, _abi.END_OOB, _abi.END_TIMEOUT)
_END_REASON_BITS = _abi.END_COLLISION | _abi.END_ALL_GOALS | _abi.END_OOB | _abi.END_TIMEOUT


def end_truncated(end):
    """Episode-log end bits (column _abi.EP_END; numpy or torch integer array) -> truncated: the episode ended on the step
    cap alone (SHIPSIM_END_TIMEOUT; a goal taken on that step does not change it)."""
    return (end & _END_REASON_BITS) == _abi.END_TIMEOUT


class EpisodeLog(object):
    """The episode log's buffers (BatchedShipEnv.enable_episode_log): the kernels append terminal rows `rows` and metadata
    `meta` (columns _abi.EP_*) and count the records in the device int32 `count` (those past `capacity` are lost).
    HISTORY_SIZE > 2: the kernel logs terminal frames, and `term` holds the terminal rows assembled from them."""

    def __init__(self, rows, meta, count, capacity, term=None):
        self.rows, self.meta, self.count, self.capacity, self.term = rows, meta, count, capacity, term

    def clear(self):
        """Empty the log: zero the device count, in order on the current stream."""
        self.count.zero_()


def episode_dict(meta, rows, env_id_offset=0):
    """Episode-log records -> the dict `BatchedShipEnv.episodes()` returns, sorted by (call, k, env).

    meta: int32 [n, 8] (columns _abi.EP_*), rows: float32 [n, D] terminal observations.  Pure torch, any device.
    `truncated` = end_truncated, `terminated` = everything else: collision, out of bounds or all goals taken."""
    meta = meta.to(torch.int32).contiguous()
    order = torch.arange(meta.shape[0], device=meta.device)
    for col in (_abi.EP_ENV, _abi.EP_K, _abi.EP_CALL):          # least significant key first, stable sorts
        order = order[torch.sort(meta[order, col], stable=True).indices]
    m = meta[order]
    end = m[:, _abi.EP_END]
    truncated = end_truncated(end)
    col = lambda c: m[:, c].long()      # noqa: E731
    return {
        "env": col(_abi.EP_ENV), "global_env": col(_abi.EP_ENV) + int(env_id_offset), "k": col(_abi.EP_K), "call": col(_abi.EP_CALL),
        "length": col(_abi.EP_LENGTH), "return": m[:, _abi.EP_RETURN].contiguous().view(torch.float32),
        "terminated": ~truncated, "truncated": truncated, "collision": (end & _abi.END_COLLISION) != 0,
        "oob": (end & _abi.END_OOB) != 0, "all_goals": (end & _abi.END_ALL_GOALS) != 0, "goal": (end & _abi.END_GOAL) != 0,
        "scenario": col(_abi.EP_SCENARIO), "episode": col(_abi.EP_EPISODE), "terminal_obs": rows[order],
    }


# columns of the per-scenario outcome table (fold_episode_log, BatchedShipEnv.scenario_outcomes)
OUTCOME_COLUMNS = ("episodes", "return_sum", "length_sum", "collision", "all_goals", "oob", "timeout")


def fold_episode_log(meta, count, n_scenarios, out=None):
    """Per-scenario sums of the episode-log records meta[:count] (int32 [cap, 8], columns _abi.EP_*; `count` a 1-element
    tensor, records past the capacity are lost): float64 [n_scenarios, len(OUTCOME_COLUMNS)] -- episodes, return sum,
    length sum and the episodes that ended by collision, all goals, out of bounds and the step cap.  Added into `out`
    when given.  Pure torch on meta's device, masked by the device-side count: no host synchronisation."""
    cap = meta.shape[0]
    dev = meta.device
    valid = torch.arange(cap, device=dev) < count.to(dev)
    end = meta[:, _abi.EP_END]
    cols = torch.stack([torch.ones(cap, dtype=torch.float64, device=dev),
                        meta[:, _abi.EP_RETURN].contiguous().view(torch.float32).double(),
                        meta[:, _abi.EP_LENGTH].double()] +
                       [((end & bit) != 0).double() for bit in END_REASONS], 1)
    cols = torch.where(valid[:, None], cols, torch.zeros((), dtype=torch.float64, device=dev))
    scen = meta[:, _abi.EP_SCENARIO].long().clamp(0, n_scenarios - 1)      # (rows past the count hold anything)
    if out is None:
        out = torch.zeros(n_scenarios, len(OUTCOME_COLUMNS), dtype=torch.float64, device=dev)
    return out.index_add_(0, scen, cols)


def quantize_scenario_weights(w):
    """Float pick weights -> the uint32 weights shipsim_scenario_weights reads (as int32: every value is below 2^31), on
    w's device with no host synchronisation: NaN and negative weights count as 0, +inf as the largest finite weight; the
    weights are scaled so that their sum stays at most 2^31, and a positive weight is never rounded to 0 (it becomes at
    least 1).  Equal weights stay equal (so the picks are the uniform ones), and all-zero weights stay zero (uniform
    picks as well)."""
    w = torch.nan_to_num(w.to(torch.float64), nan=0.0, posinf=torch.finfo(torch.float64).max, neginf=0.0).clamp_min(0.0)
    n = w.numel()
    w = w / w.amax().clamp_min(torch.finfo(torch.float64).tiny)            # in [0, 1], the largest is 1: no overflow below
    # 2n of headroom: the rounding of the float64 sum (far below n) and the floor of positive weights at 1 (at most n)
    q = torch.floor(w * ((2.0 ** 31 - 2 * n) / w.sum().clamp_min(1.0)))
    return torch.where(w > 0, q.clamp_min(1.0), q).to(torch.int32)


def long_history_rows(prev_rows, frames, done, auto_reset):
    """HISTORY_SIZE > 2 (SURVEY App. A, N2): the rows [frame t-H+1 | ... | frame t] of K steps, put together from the
    steps' frames and the rows before them, with -1 for everything older than an env's latest reset (under auto-reset the
    frame of a done step IS the reset frame: ship_env.py:180-184).  Copies and -1 fills only.
    prev_rows [N, H*F], frames [K, N, F], done [K, N] -> [K, N, H*F]."""
    K, N, F = frames.shape
    H = prev_rows.shape[1] // F
    prev = prev_rows.view(N, H, F).permute(1, 0, 2)            # [H][N][F], oldest first
    allf = torch.cat([prev, frames], dim=0)                   # frame of step k sits at index H + k
    rows = allf.unfold(0, H, 1)[1:].permute(0, 1, 3, 2)       # [K][N][H][F]: rows[k] = frames k-H+1 .. k
    if auto_reset:
        k_idx = torch.arange(K, device=frames.device)[:, None]
        last_reset = torch.where(done.bool(), k_idx, torch.full_like(k_idx, -(1 << 30))).cummax(dim=0).values      # [K][N]
        slot_time = k_idx[:, :, None] - torch.arange(H - 1, -1, -1, device=frames.device)[None, None, :]           # [K][1][H]
        rows = torch.where((slot_time < last_reset[:, :, None])[..., None], torch.full_like(rows, -1.0), rows)
    return rows.reshape(K, N, H * F).contiguous()


def long_history_terminal_rows(prev_rows, rows, k, env, frame):
    """HISTORY_SIZE > 2: the kernel logs the terminal FRAME; the terminal row is the env's row before the done step
    (`rows[k - 1]`, or `prev_rows` -- the rows before the call -- for k = 0) moved on by one frame, then that frame, i.e.
    the H - 1 frames before the done step with -1 beyond the env's previous reset, as long_history_rows builds rows.
    prev_rows [N, H*F], rows [K, N, H*F], k / env [n] int64, frame [n, F] -> [n, H*F]."""
    F = frame.shape[1]
    before = torch.where((k > 0)[:, None], rows[(k - 1).clamp(min=0), env], prev_rows[env])
    return torch.cat([before[:, F:], frame], dim=1)


class BatchedShipEnv(object):
    """`num_envs` independent ShipEnvs on one GPU.

    step(actions) -> (obs [N,F*H] f32, reward [N] f32, done [N] bool, info {})      one env-step per call
    rollout(actions [K,N] | None, K) -> (obs [K,N,F*H], reward [K,N], done [K,N])   K steps in ONE launch
    F = n_states = 6 + n_beams floats per frame: 16 with the reference's 10-beam lidar; with `honour_lidar_config=True`
    LidarConfig.N_BEAMS (1..32) sets the fan.
    With auto_reset (default, the SubprocVecEnv worker semantics behind train/stable_baselines/ppo.py:123) a
    done env is reset inside the kernel and the obs returned for that step is the reset obs.
    """

    metadata = {"render.modes": ["human", "rgb_array"]}       # ship_env.py:18
    reward_range = (-1, 1)                                    # ship_env.py:20

    def __init__(self, num_envs, game_config=None, env_config=None, device=None, seed=0, n_scenarios=1024,
                 bank=None, map_N=10, map_width_frac=0.5, auto_reset=True, honour_lidar_config=False,
                 env_id_offset=0, lanes_per_env=0, validate_actions=True, scenario_source="host", steps_in_flight=0,
                 host_threads=0, fresh_maps=False):
        self.knobs = snapshot(game_config, env_config, honour_lidar_config)
        self.n_beams = self.knobs["lidar"]["N_BEAMS"]         # 1..32 (shipsim_create checks the range)
        self.num_envs = int(num_envs)
        self.device = torch.device("cuda") if device is None else torch.device(device)
        if self.device.type != "cuda":
            raise _abi.ShipsimError("BatchedShipEnv needs a CUDA device: there is no CPU fallback")
        if self.device.index is None:          # 'cuda' = the CURRENT device, not device 0: handle and buffers must agree
            self.device = torch.device("cuda", torch.cuda.current_device())
        self.L = _abi.load()
        self._needs_reset = True
        self.action_space = Discrete(3)                        # ship_env.py:19
        self.history = self.knobs["history"]
        self.n_states = 2 + 1 + 1 + 2 + self.n_beams           # ship_env.py:43: floats per frame
        self.states_history = self.n_states * self.history     # ship_env.py:44
        self.observation_space = Box(0, max(self.knobs["W"], self.knobs["H"]), (self.states_history,), np.uint8)
        self.bounds = (self.knobs["W"], self.knobs["H"])
        self.auto_reset = bool(auto_reset)
        self.validate_actions = bool(validate_actions)
        self.seed_value = int(seed)

        dt = BASE_DT * self.knobs["speed"]                     # game.py:194
        cfg = _abi.default_config()
        cfg.num_envs = self.num_envs
        cfg.env_id_offset = int(env_id_offset)
        cfg.seed = self.seed_value & 0xFFFFFFFFFFFFFFFF
        cfg.bounds_w, cfg.bounds_h = self.knobs["W"], self.knobs["H"]
        cfg.dt = dt
        cfg.damping = math.pow(SPACE_DAMPING, dt)              # cpSpaceStep: pow(space.damping, dt), in double
        cfg.max_steps = self.knobs["max_steps"]
        cfg.history = self.history if self.history <= 2 else 1         # longer rows are assembled here from frames
        cfg.auto_reset = int(self.auto_reset)
        cfg.lidar_spread_deg = self.knobs["lidar"]["ANGULAR_SPREAD"]
        cfg.lidar_distance = self.knobs["lidar"]["DISTANCE"]
        cfg.lidar_beams = self.n_beams
        cfg.lanes_per_env = int(lanes_per_env)
        cfg.steps_in_flight = int(steps_in_flight)     # 0 auto, 1 serial-in-time kernel, 4/8/16/32 time-parallel window
        if not host_threads:
            # step_host's row-assembly pool: the box's cores are shared by the ranks torchrun started on it
            import os
            ranks_here = max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1")))
            host_threads = max(1, min(16, (os.cpu_count() or 1) // ranks_here))
        cfg.host_threads = int(host_threads)
        self.cfg = cfg
        self.reset_epoch = 0
        self.last_reset_obs = None
        self.params_epoch = 0                  # bumped whenever kernel parameters change (captured CUDA graphs go stale)
        self.graph_safe = True                 # False: kernel parameters change between launches (no CUDA-graph replay)
        self._pick_w = None                    # scenario weights (set_scenario_weights): the quantized device copy, or None
        self._n_generated = 0
        self._hist = None                      # HISTORY_SIZE > 2: the latest rows [N, H*F] (long_history_rows)
        self.total_steps = 0
        self._calls = 0                        # shipsim_step / shipsim_step_host calls (mirrors the handle's SHIPSIM_EP_CALL)
        self.episode_log = None                # EpisodeLog while the log is on (enable_episode_log)
        self._np_bufs = None                   # step_np's page-locked buffers
        # back-to-back rollouts may overlap (shipsim_step_chained): each env's next launch starts as soon as its own
        # previous one is done.  False: every launch waits for the whole previous launch (shipsim_step).
        self.chain_launches = True
        self._chain_prev = None                # (stream, actions, their _version) of the last _launch while it is the env's last device work
        self._h = C.c_void_p()
        _abi.check(self.L.shipsim_create(C.byref(cfg), self.device.index, C.byref(self._h)))
        self._obs_dim_kernel = self.n_states * cfg.history

        if scenario_source not in ("host", "device"):
            raise ValueError("scenario_source must be 'host' or 'device'")
        if bank is None and scenario_source == "device":
            # maps generated by the GPU itself (shipsim_generate_scenarios): no host loop over resets
            self.generate_scenarios(n_scenarios, seed=self.seed_value, map_N=map_N, map_width_frac=map_width_frac)
        else:
            if bank is None:
                bank = ScenarioBank.generate(n_scenarios, self.bounds, seed=self.seed_value, map_N=map_N,
                                             width_frac=map_width_frac)
            self.load_scenarios(bank)

        with torch.cuda.device(self.device):
            nbytes = self.L.shipsim_state_bytes(self._h)
            # planes [0, 8) as for every fan, then ceil((n - 10) / 4) planes of lidar[10 ..] for fans of more than 10 beams
            self.state = torch.zeros(nbytes // 4, dtype=torch.float32, device=self.device).view(nbytes // (16 * self.num_envs), self.num_envs, 4)
            self._stats_slots = torch.zeros(self.L.shipsim_stats_bytes(self._h) // 8, dtype=torch.float64, device=self.device)
            self._stats_out = torch.zeros(_abi.STATS_LEN, dtype=torch.float64, device=self.device)
            _abi.check(self.L.shipsim_bind_state(self._h, self.state.data_ptr(), self._stats_slots.data_ptr(), self._stream()))
        if fresh_maps:
            self.fresh_maps(True)

    # ------------------------------------------------------------------------------------------ plumbing
    def _stream(self):
        """The current stream of the env's device, for a call that enqueues work through the handle: such work ends a
        chain of launches (_chains_on)."""
        self._chain_prev = None
        return C.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self.L.shipsim_destroy(self._h)
            self._h = C.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def load_scenarios(self, bank):
        """Upload a ScenarioBank (curriculum changes call this between rollouts).  On a live batch every env is then
        RESET: its stored scenario id and goals belong to the old bank (ShipGame.reset builds level and goals together,
        game.py:271-272); `last_reset_obs` holds the reset observations."""
        if tuple(bank.bounds) != tuple(self.bounds):
            raise ValueError("scenario bank was generated for bounds %s, env has %s" % (bank.bounds, self.bounds))
        self._chain_prev = None
        with torch.cuda.device(self.device):
            _abi.check(self.L.shipsim_load_scenarios(self._h, bank.hull_xy.ctypes.data, bank.hull_n.ctypes.data,
                                                     bank.goals.ctypes.data, len(bank), bank.maxv))
        self._new_bank(bank, len(bank))
        if not self._needs_reset:
            self.reset()

    def generate_scenarios(self, n_scenarios, seed=0, map_N=10, map_width_frac=0.5):
        """Replace the scenario bank by `n_scenarios` maps generated on the device (river banks, hulls, goal paths;
        SURVEY.md §8 f2).  Envs keep the goals of the scenario they started with until their next reset, so call it
        where all envs are reset (e.g. followed by `reset()`)."""
        with torch.cuda.device(self.device):
            _abi.check(self.L.shipsim_generate_scenarios(self._h, int(n_scenarios), int(seed) & 0xFFFFFFFFFFFFFFFF, int(map_N),
                                                         float(map_width_frac), self._stream()))
        self._n_generated = int(n_scenarios)
        self._new_bank(None, self._n_generated)
        self._needs_reset = True

    def _new_bank(self, bank, n_scenarios):
        """Host-side state of a newly installed bank (`bank` None: generated on the device).  A new bank leaves fresh-maps
        mode and drops the scenario weights (shipsim_load_scenarios / shipsim_generate_scenarios)."""
        self.bank = bank
        self._n_scen = n_scenarios
        self.params_epoch += 1
        self.graph_safe = True
        self._pick_w = None

    def fresh_maps(self, enable=True):
        """A new map for every episode, as ShipGame.reset builds one (game.py:271-272): the device-generated bank
        (`scenario_source="device"` or `generate_scenarios`; 4 * 2^k scenarios) is regenerated slice by slice on a side
        stream behind the envs, and resets only pick from the newest slice (shipsim_fresh_maps).  Needs auto_reset."""
        self._chain_prev = None
        with torch.cuda.device(self.device):
            _abi.check(self.L.shipsim_fresh_maps(self._h, int(bool(enable))))
        self.graph_safe = not enable
        self.params_epoch += 1

    @property
    def n_scenarios(self):
        """Size of the scenario bank the resets pick from."""
        return self._n_scen

    def set_scenario_weights(self, weights):
        """Resets (automatic ones and reset() without explicit scenarios) pick map i with probability w[i] / sum(w)
        instead of uniformly (shipsim_scenario_weights).  `weights`: n_scenarios floats (numpy, list or tensor); None
        returns to uniform picks.  Weight 0 holds a map out; all-zero device weights fall back to uniform picks.  The
        weights are quantized on the device (quantize_scenario_weights) and the pick table is rebuilt there: no host
        synchronisation for device input, so the call may sit between the replays of a captured rollout graph, which
        picks up the new weights (changing weights leaves `params_epoch` alone; turning them on or off moves it).  A new
        bank drops the weights; fresh maps and weights exclude each other (ShipsimError)."""
        if weights is None:
            with torch.cuda.device(self.device):
                _abi.check(self.L.shipsim_scenario_weights(self._h, None, self._stream()))
            if self._pick_w is not None:
                self._pick_w = None
                self.params_epoch += 1
            return
        n = self._n_scen
        if not (isinstance(weights, torch.Tensor) and weights.is_cuda):
            a = np.asarray(weights.numpy() if isinstance(weights, torch.Tensor) else weights, dtype=np.float64)
            if a.shape != (n,):
                raise ValueError("scenario weights: need %d weights (one per scenario), got shape %s" % (n, a.shape))
            if not (np.nan_to_num(a, nan=0.0) > 0).any():
                raise ValueError("scenario weights: no positive weight (None returns to uniform picks)")
            weights = torch.from_numpy(a)
        elif tuple(weights.shape) != (n,):
            raise ValueError("scenario weights: need %d weights (one per scenario), got shape %s" % (n, tuple(weights.shape)))
        turning_on = self._pick_w is None
        with torch.cuda.device(self.device):
            q = quantize_scenario_weights(weights.to(self.device, non_blocking=True))
            buf = torch.empty_like(q) if turning_on else self._pick_w
            buf.copy_(q)                       # a fixed buffer: the table build reads it later in stream order
            _abi.check(self.L.shipsim_scenario_weights(self._h, buf.data_ptr(), self._stream()))
        self._pick_w = buf
        if turning_on:
            self.params_epoch += 1

    def fresh_info(self):
        """dict(enabled, period, pick_base, pick_count, generation[4]) of the fresh-maps rotation."""
        a = (C.c_int32 * 8)()
        _abi.check(self.L.shipsim_fresh_info(self._h, a))
        return {"enabled": bool(a[0]), "period": a[1], "pick_base": a[2], "pick_count": a[3], "generation": list(a[4:8])}

    def read_scenarios(self):
        """The device-generated bank as a host ScenarioBank (validation / inspection)."""
        S = self._n_generated
        hull_xy = np.zeros((S, 2, _abi.MAX_HULL, 2))
        hull_n = np.zeros((S, 2), dtype=np.int32)
        goals = np.zeros((S, 5, 2))
        self._chain_prev = None
        with torch.cuda.device(self.device):
            _abi.check(self.L.shipsim_read_scenarios(self._h, hull_xy.ctypes.data, hull_n.ctypes.data, goals.ctypes.data))
        return ScenarioBank(hull_xy, hull_n, goals, self.bounds)

    def set_max_steps(self, max_steps):
        """Change EnvConfig.MAX_STEPS (config.py:16) of the live batch -- a curriculum knob."""
        _abi.check(self.L.shipsim_set_max_steps(self._h, int(max_steps)))
        self.knobs["max_steps"] = int(max_steps)
        self.params_epoch += 1

    def seed(self, seed=None):
        """ship_env.py:52-60 seeds numpy only; here it also re-keys the action-space sampler."""
        if seed is None:
            seed = int(np.random.SeedSequence().entropy % (2 ** 31))
        np.random.seed(seed % (2 ** 32))
        self.action_space.seed(seed)
        return [seed]

    def render(self, mode="human", close=False, env_index=0, size=None):
        """ship_env.py:158-168 only prints; `rgb_array` (listed in metadata, ship_env.py:18, never implemented there)
        draws ONE env on the device the way ShipGame.render does (game.py:197-229) and returns a uint8 CUDA tensor
        [height, width, 3] (the gym convention); `size` = (width, height), default = BOUNDS."""
        if mode != "rgb_array":
            return None
        if self._needs_reset:
            raise _abi.ShipsimError("call reset() before render()")
        w, h = (int(self.knobs["W"]), int(self.knobs["H"])) if size is None else (int(size[0]), int(size[1]))
        img = torch.empty(h, w, 3, dtype=torch.uint8, device=self.device)
        with torch.cuda.device(self.device):
            _abi.check(self.L.shipsim_render(self._h, int(env_index), w, h, img.data_ptr(), self._stream()))
        return img

    def get_screen(self, env_index=0):
        """ShipGame.get_screen (game.py:133-138): pygame.surfarray.array3d layout, [width, height, 3]."""
        return self.render("rgb_array", env_index=env_index).permute(1, 0, 2).contiguous()

    # ------------------------------------------------------------------------------------------ reset / step
    def reset(self, mask=None, scenario=None):
        """Reset all envs (or those where `mask` is true).  Returns the observation of ALL envs is not
        available for a partial reset -- rows of envs that were not reset are left as zeros."""
        N = self.num_envs
        obs = torch.zeros(N, self._obs_dim_kernel, dtype=torch.float32, device=self.device)
        m = None if mask is None else mask.to(device=self.device, dtype=torch.uint8).contiguous()
        sc = None if scenario is None else torch.as_tensor(scenario, device=self.device).to(torch.int32).contiguous()
        if sc is not None:
            if sc.numel() != N:
                raise ValueError("scenario must hold one id per env")
            lo, hi = int(sc.min()), int(sc.max())
            if lo < 0 or hi >= self._n_scen:
                raise ValueError("scenario ids must be in [0, %d), got [%d, %d]" % (self._n_scen, lo, hi))
        first = 1 if (mask is None and self._needs_reset) else 0
        with torch.cuda.device(self.device):
            _abi.check(self.L.shipsim_reset(self._h, None if m is None else m.data_ptr(), None if sc is None else sc.data_ptr(),
                                            first, obs.data_ptr(), self._stream()))
        self._needs_reset = False
        self.reset_epoch += 1
        self.last_reset_obs = obs if mask is None else None
        if self.history > 2:                   # obs holds the reset frames: rows [-1 ... -1 | frame]
            fresh = torch.full((N, self.states_history), -1.0, dtype=torch.float32, device=self.device)
            fresh[:, -self.n_states:] = obs
            self._hist = fresh if mask is None or self._hist is None else torch.where(m.bool()[:, None], fresh, self._hist)
            return self._hist.clone()
        return obs

    def _check_actions(self, actions):
        if self.validate_actions:
            bad = ((actions < 0) | (actions > 2)).any()
            assert not bool(bad), "%r invalid" % (actions,)       # ship_env.py:143

    def step(self, actions):
        """One env-step for every env.  `actions`: int tensor [N] on the env's device (or anything
        torch.as_tensor accepts; host data is copied)."""
        a = torch.as_tensor(actions)
        if a.device != self.device:
            a = a.to(self.device)
        if a.dtype not in (torch.int32, torch.int64, torch.uint8):
            a = a.to(torch.int64)
        a = a.contiguous().view(-1)
        assert a.numel() == self.num_envs, "expected %d actions" % self.num_envs
        self._check_actions(a)
        obs, rew, done = self._step_long(a, 1) if self.history > 2 else self._launch(a, 1)
        return obs[0], rew[0], done[0].bool(), {}

    def rollout(self, actions=None, K=None, out=None):
        """K consecutive env-steps in one kernel launch.  actions: int tensor [K,N] on device, or None for the
        in-kernel random agent (train/random.py:18).  `out` = (obs, reward, done) preallocated tensors."""
        if self.history > 2 and out is not None:
            raise NotImplementedError("rollout(out=...) supports HISTORY_SIZE <= 2 (longer rows are assembled from frames here)")
        if actions is not None:
            a = actions
            if a.device != self.device:
                a = a.to(self.device)
            a = a.contiguous()
            assert a.dim() == 2 and a.shape[1] == self.num_envs
            K = a.shape[0]
            self._check_actions(a)
        else:
            assert K is not None
            a = None
        if self.history > 2:
            return self._step_long(a, K)
        return self._launch(a, K, out)

    def _step_long(self, a, K):
        """HISTORY_SIZE > 2: one launch in the kernel's one-frame mode; the rows come from long_history_rows, and the
        records the launch logged get their terminal rows (no host sync).  -> rows [K, N, H*F], reward, done."""
        frames, rew, done = self._launch(a, K)
        rows = long_history_rows(self._hist, frames, done, self.auto_reset)
        log = self.episode_log
        if log is not None:
            new = (torch.arange(log.capacity, device=self.device) < log.count) & (log.meta[:, _abi.EP_CALL] == self._calls - 1)
            k = log.meta[:, _abi.EP_K].long().clamp(0, K - 1)
            env = log.meta[:, _abi.EP_ENV].long().clamp(0, self.num_envs - 1)
            log.term = torch.where(new[:, None], long_history_terminal_rows(self._hist, rows, k, env, log.rows), log.term)
        self._hist = rows[-1].clone()
        return rows, rew, done

    def alloc_rollout(self, K):
        N = self.num_envs
        return (torch.empty(K, N, self._obs_dim_kernel, dtype=torch.float32, device=self.device),
                torch.empty(K, N, dtype=torch.float32, device=self.device),
                torch.empty(K, N, dtype=torch.uint8, device=self.device))

    def _launch(self, a, K, out=None):
        if self._needs_reset:
            raise _abi.ShipsimError("call reset() before step()")
        obs, rew, done = out if out is not None else self.alloc_rollout(K)
        code = _abi.ACTION_RANDOM if a is None else _dtype_code(a)
        # (no torch.cuda.device() context here: shipsim_step selects the handle's device itself, and on the gym-style K = 1
        # path the two extra cudaSetDevice calls were a fifth of the per-launch host time)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        step = self.L.shipsim_step_chained if self._chains_on(a, stream) else self.L.shipsim_step
        rc = step(self._h, None if a is None else a.data_ptr(), code, K, obs.data_ptr(), rew.data_ptr(), done.data_ptr(), stream)
        if rc:
            _abi.check(rc)
        self._calls += 1
        self.total_steps += K * self.num_envs
        return obs, rew, done

    def _chains_on(self, a, stream):
        """Whether this launch may chain onto the previous one (shipsim_step_chained, which checks the rest): that launch
        was the env's last device work, on the same stream, with the same actions -- the same tensor, not modified in place
        since (its _version), or the in-kernel random agent both times -- and rows are at most two frames long (longer
        ones are assembled by torch ops between the launches)."""
        prev, self._chain_prev = self._chain_prev, (stream, a, None if a is None else a._version)
        if not self.chain_launches or self.history > 2 or prev is None:
            return False
        return prev[0] == stream and prev[1] is a and (a is None or prev[2] == a._version)

    def step_host(self, actions, K=1, out=None):
        """The CPU-caller path: numpy/pinned int32 actions [K,N] in, numpy obs/reward/done out, with the
        host<->device copies inside (shipsim_step_host)."""
        a = np.ascontiguousarray(actions, dtype=np.int32).reshape(K, self.num_envs)
        if out is None:
            out = (np.empty((K, self.num_envs, self.states_history), dtype=np.float32),
                   np.empty((K, self.num_envs), dtype=np.float32), np.empty((K, self.num_envs), dtype=np.uint8))
        obs, rew, done = out           # any of them may be None: that output is then not copied back
        self._step_host(a, K, obs, rew, done)
        return obs, rew, done

    def step_np(self, actions):
        """One env-step for a caller on the CPU (the gym facade, the vector-env adapters): numpy int actions [N] in,
        (obs [N, n_states * history] float32, reward [N] float32, done [N] bool) out -- ONE call into shipsim_step_host with
        page-locked buffers kept on the env; no torch ops, one stream wait.  The returned arrays are the env's buffers:
        valid until the next call (copy them to keep them)."""
        if self._np_bufs is None:
            pin = lambda *shape, dtype: torch.empty(*shape, dtype=dtype).pin_memory()      # noqa: E731
            self._np_keep = (pin(1, self.num_envs, dtype=torch.int32), pin(1, self.num_envs, self.states_history, dtype=torch.float32),
                             pin(1, self.num_envs, dtype=torch.float32), pin(1, self.num_envs, dtype=torch.uint8))
            self._np_bufs = tuple(t.numpy() for t in self._np_keep)
        a, obs, rew, done = self._np_bufs
        a[0, :] = actions
        self._step_host(a, 1, obs, rew, done)
        return obs[0], rew[0], done[0].view(np.bool_)

    def _step_host(self, a, K, obs, rew, done):
        """step_host / step_np: int32 actions a [K, N] and numpy outputs (None: not copied back) through shipsim_step_host."""
        if self.validate_actions:
            assert ((a >= 0) & (a <= 2)).all(), "%r invalid" % (a,)       # ship_env.py:143
        if self.history > 2:          # (rows assembled on the device, then copied: this path is not tuned for long histories)
            for dst, src in zip((obs, rew, done), self._step_long(torch.from_numpy(a).to(self.device), K)):
                if dst is not None:
                    dst[...] = src.cpu().numpy()
            return
        with torch.cuda.device(self.device):
            _abi.check(self.L.shipsim_step_host(self._h, a.ctypes.data, K, None if obs is None else obs.ctypes.data, None if rew is None
                                                else rew.ctypes.data, None if done is None else done.ctypes.data, self._stream()))
        self._calls += 1
        self.total_steps += K * self.num_envs

    def host_threads(self):
        """Host threads step_host() uses to rebuild observation rows (0 before its first call)."""
        n = C.c_int32()
        _abi.check(self.L.shipsim_host_threads(self._h, C.byref(n)))
        return n.value

    def host_traffic(self):
        """(host->device, device->host) bytes the last step_host() moved over PCIe."""
        a, b = C.c_int64(), C.c_int64()
        _abi.check(self.L.shipsim_host_traffic(self._h, C.byref(a), C.byref(b)))
        return a.value, b.value

    # ------------------------------------------------------------------------------------------ episode log
    def enable_episode_log(self, capacity=None, pinned=False):
        """Record every finished episode (shipsim_episode_log_bind): its terminal observation -- the row an auto_reset=False
        batch would have returned for the done step, which the auto-reset replaces by the reset row -- why it ended, its
        return and length.  Read the records with episodes().  `capacity` = records kept between two episodes() calls
        (default num_envs: one K = 1 step); 0 turns the log off.  `pinned`: rows and metadata in page-locked host memory
        (written over PCIe by the kernel: a numpy caller reads them after step_np's own wait, with no copy).  Needs
        auto_reset."""
        capacity = self.num_envs if capacity is None else int(capacity)
        self._chain_prev = None
        self.params_epoch += 1                 # (the buffers' addresses travel in the kernel parameters: captured graphs go stale)
        if capacity == 0:
            _abi.check(self.L.shipsim_episode_log_bind(self._h, None, None, 0, None))
            self.episode_log = None
            return
        term = None
        if self.history > 2:                   # the kernel logs frames: the terminal rows are assembled in _step_long
            if pinned:
                raise ValueError("pinned episode logs need HISTORY_SIZE <= 2 (longer terminal rows are assembled on the device)")
            term = torch.full((capacity, self.states_history), -1.0, dtype=torch.float32, device=self.device)
        where = dict(pin_memory=True) if pinned else dict(device=self.device)
        rows = torch.zeros(capacity, self._obs_dim_kernel, dtype=torch.float32, **where)
        meta = torch.zeros(capacity, _abi.EPISODE_META, dtype=torch.int32, **where)
        count = torch.zeros(1, dtype=torch.int32, device=self.device)
        with torch.cuda.device(self.device):
            _abi.check(self.L.shipsim_episode_log_bind(self._h, rows.data_ptr(), meta.data_ptr(), capacity, count.data_ptr()))
        self.episode_log = EpisodeLog(rows, meta, count, capacity, term)

    def episodes(self, clear=True):
        """The records of the episodes that finished since the log was last cleared, as a dict of device tensors sorted by
        (call, k, env): env, global_env (+ env_id_offset: shard logs concatenate), k (step within the call), call (sequence
        number of the step call), length, return, terminated, truncated (step cap alone), collision, oob, all_goals, goal,
        scenario, episode (of the finished episode) and terminal_obs.  `clear` empties the log.  Raises ShipsimError when
        more episodes finished than the log could hold."""
        log = self.episode_log
        if log is None:
            raise _abi.ShipsimError("no episode log: call enable_episode_log() first")
        n, cap = int(log.count.item()), log.capacity       # (waits for the stream: the records of every launch so far are in place)
        if clear:
            log.clear()
            self._chain_prev = None
        if n > cap:
            raise _abi.ShipsimError("episode log overflow: %d episodes finished, capacity %d: %d records lost" % (n, cap, n - cap))
        r = log.rows[:n].to(self.device) if log.term is None else log.term[:n]
        return episode_dict(log.meta[:n].to(self.device), r, self.cfg.env_id_offset)

    def scenario_outcomes(self, out=None, clear=True):
        """Per-map outcomes of the episodes the log holds (fold_episode_log): float64 [n_scenarios, 7] device tensor with
        columns OUTCOME_COLUMNS (episodes, return_sum, length_sum, collision, all_goals, oob, timeout), added into `out`
        when given -- "which maps does the policy fail on".  `clear` empties the log.  No host synchronisation (an
        overflowing log is not reported here: its lost records are simply missing)."""
        log = self.episode_log
        if log is None:
            raise _abi.ShipsimError("no episode log: call enable_episode_log() first")
        out = fold_episode_log(log.meta.to(self.device, non_blocking=True), log.count, self._n_scen, out)
        if clear:
            log.clear()
            self._chain_prev = None
        return out

    # ------------------------------------------------------------------------------------------ stats / state
    def stats_tensor(self, clear=False, out=None):
        """float64[16] device tensor (see shipsim_stat); ready to be all-reduced.  `out`: write into this tensor
        (e.g. StatsReducer.next_buffer()) instead of the env's own."""
        dst = self._stats_out if out is None else out
        assert dst.dtype == torch.float64 and dst.numel() >= _abi.STATS_LEN and dst.is_contiguous()
        with torch.cuda.device(self.device):
            _abi.check(self.L.shipsim_stats_read(self._h, dst.data_ptr(), int(clear), self._stream()))
        return dst

    def stats(self, clear=False):
        v = self.stats_tensor(clear).cpu().tolist()
        d = dict(zip(_abi.STAT_NAMES, v))
        d["steps"] = float(self.total_steps)
        return d

    def get_state(self):
        """dict of numpy arrays: pose [N,6] (x y angle vx vy w), ints [N,5] (rudder, alive_mask, step_count,
        scenario, episode), lidar [N,n_beams], goals [N,5,2], ep_return [N]."""
        N = self.num_envs
        pose = np.zeros((N, 6), dtype=np.float32)
        ints = np.zeros((N, 5), dtype=np.int32)
        lidar = np.zeros((N, self.n_beams), dtype=np.float32)
        goals = np.zeros((N, 5, 2), dtype=np.float32)
        ret = np.zeros(N, dtype=np.float32)
        self._chain_prev = None
        with torch.cuda.device(self.device):
            _abi.check(self.L.shipsim_get_state(self._h, pose.ctypes.data, ints.ctypes.data, lidar.ctypes.data,
                                                goals.ctypes.data, ret.ctypes.data))
        return dict(pose=pose, ints=ints, lidar=lidar, goals=goals, ep_return=ret)

    def set_state(self, pose, ints, lidar, goals, ep_return):
        N = self.num_envs
        pose = np.ascontiguousarray(pose, dtype=np.float32).reshape(N, 6)
        ints = np.ascontiguousarray(ints, dtype=np.int32).reshape(N, 5)
        lidar = np.ascontiguousarray(lidar, dtype=np.float32).reshape(N, self.n_beams)
        goals = np.ascontiguousarray(goals, dtype=np.float32).reshape(N, 10)
        ret = np.ascontiguousarray(ep_return, dtype=np.float32).reshape(N)
        self._chain_prev = None
        with torch.cuda.device(self.device):
            _abi.check(self.L.shipsim_set_state(self._h, pose.ctypes.data, ints.ctypes.data, lidar.ctypes.data,
                                                goals.ctypes.data, ret.ctypes.data))
        self._needs_reset = False

    def launch_info(self):
        """Launches issued so far, of which `chained` overlapped their predecessor (shipsim_step_chained), and the shape of
        the last one."""
        n, chained = C.c_int64(), C.c_int64()
        lanes, thr, ctas = C.c_int32(), C.c_int32(), C.c_int32()
        _abi.check(self.L.shipsim_launch_count(self._h, C.byref(n)))
        _abi.check(self.L.shipsim_launch_shape(self._h, C.byref(lanes), C.byref(thr), C.byref(ctas)))
        win = C.c_int32()
        _abi.check(self.L.shipsim_launch_window(self._h, C.byref(win)))
        _abi.check(self.L.shipsim_chained_count(self._h, C.byref(chained)))
        return dict(launches=n.value, lanes_per_env=lanes.value, threads_per_cta=thr.value, ctas=ctas.value,
                    steps_in_flight=win.value, chained=chained.value)


class ShipEnv(object):
    """Single-env facade with the reference constructor and numpy in/out: `ShipEnv(game_config, env_config)`
    (ship_env.py:23) -- what train/random.py:9-26 and the `make_env()` thunks construct.  It is a batch of one;
    like the reference, `step` does NOT auto-reset."""

    metadata = BatchedShipEnv.metadata
    reward_range = BatchedShipEnv.reward_range
    action_space = Discrete(3)

    def __init__(self, game_config=None, env_config=None, **kw):
        kw.setdefault("n_scenarios", 64)
        kw["auto_reset"] = False
        self.batch = BatchedShipEnv(1, game_config, env_config, **kw)
        self.env_config = env_config
        self.n_states = self.batch.n_states
        self.states_history = self.batch.states_history
        self.observation_space = self.batch.observation_space
        self.last_action = None
        self.reward = 0
        self.cumulative_reward = 0
        self.step_count = 0
        self.episodes_count = -1                               # ship_env.py:33

    def seed(self, seed=None):
        return self.batch.seed(seed)

    def reset(self):
        obs = self.batch.reset(mask=None if self.episodes_count < 0 else torch.ones(1, dtype=torch.uint8))
        self.last_action = None
        self.reward = 0
        self.cumulative_reward = 0
        self.step_count = 0
        self.episodes_count += 1
        return obs[0].cpu().numpy()

    def step(self, action):
        assert self.action_space.contains(action), "%r (%s) invalid" % (action, type(action))   # ship_env.py:143
        obs, rew, done = self.batch.step_np(int(action))
        self.last_action = action
        self.reward = float(rew[0])
        self.cumulative_reward += self.reward
        self.step_count += 1
        return obs[0].copy(), self.reward, bool(done[0]), {}

    def render(self, mode="human", close=False):
        if mode == "rgb_array":
            return self.batch.render("rgb_array").cpu().numpy()
        import sys
        if self.last_action is not None:
            sys.stdout.write("action=%s, cumm_reward=%s" % (self.last_action, self.cumulative_reward))

    def close(self):
        self.batch.close()
