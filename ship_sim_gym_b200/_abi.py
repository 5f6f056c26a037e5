"""ctypes binding of libshipsim.so (include/shipsim.h).

This is the only door to the compute path: there is NO CPU or PyTorch fallback.  If the shared library has
not been built (`python -c "import __graft_entry__ as g; g.build()"` or `make -C ship_sim_gym_b200/csrc`)
importing the symbols raises, and every entry point fails with an error when no sm_100 GPU is usable.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SHIPSIM_LIB") or os.path.join(HERE, "libshipsim.so")   # override: kernel-variant experiments

ACTION_I32, ACTION_I64, ACTION_U8, ACTION_RANDOM = 0, 1, 2, 3
STATS_LEN = 16
STAT_NAMES = ("episodes", "return_sum", "length_sum", "goal_steps", "collision", "oob", "timeout", "all_goals", "steps")
N_GOALS, N_BEAMS, FRAME, STATE_PLANES, MAX_HULL = 5, 10, 16, 8, 32       # (N_BEAMS, FRAME: the default 10-beam fan)
MAX_BEAMS = 32                  # lidar_beams in [1, MAX_BEAMS]; a frame is 6 + lidar_beams floats
# episode log (shipsim_episode_log_bind): columns of a record's metadata, and the SHIPSIM_END_* bits
EPISODE_META = 8
EP_K, EP_ENV, EP_LENGTH, EP_RETURN, EP_END, EP_SCENARIO, EP_EPISODE, EP_CALL = range(8)
END_COLLISION, END_ALL_GOALS, END_OOB, END_TIMEOUT, END_GOAL = 1, 2, 4, 8, 16
# level scores (shipsim_gae_scored): columns of a map's row; the table has one more row for steps of no known map
SCORE_STEPS, SCORE_POS_ADV, SCORE_ABS_ADV, SCORE_COLS = range(4)

# every symbol include/shipsim.h declares (tests check the library exports all of them)
SYMBOLS = (
    "shipsim_abi_version", "shipsim_last_error", "shipsim_config_default", "shipsim_create", "shipsim_destroy",
    "shipsim_load_scenarios", "shipsim_state_bytes", "shipsim_stats_bytes", "shipsim_bind_state", "shipsim_reset",
    "shipsim_step", "shipsim_step_host", "shipsim_stats_read", "shipsim_set_state", "shipsim_get_state",
    "shipsim_launch_count", "shipsim_launch_shape", "shipsim_launch_window", "shipsim_set_max_steps",
    "shipsim_generate_scenarios", "shipsim_read_scenarios", "shipsim_render", "shipsim_assemble_history", "shipsim_expand_delta", "shipsim_host_traffic", "shipsim_host_threads",
    "shipsim_fresh_maps", "shipsim_fresh_info", "shipsim_mlp_policy_forward", "shipsim_gae", "shipsim_episode_log_bind",
    "shipsim_scenario_weights", "shipsim_step_chained", "shipsim_chained_count", "shipsim_gae_scored",
)


class ShipsimError(RuntimeError):
    pass


class Config(C.Structure):
    """struct shipsim_config (include/shipsim.h)."""
    _fields_ = [
        ("struct_size", C.c_int32), ("num_envs", C.c_int32), ("env_id_offset", C.c_int64), ("seed", C.c_uint64),
        ("bounds_w", C.c_float), ("bounds_h", C.c_float), ("dt", C.c_float), ("damping", C.c_float),
        ("max_steps", C.c_int32), ("history", C.c_int32), ("auto_reset", C.c_int32), ("lidar_beams", C.c_int32),
        ("lidar_spread_deg", C.c_float), ("lidar_distance", C.c_float), ("ship_w", C.c_float), ("ship_h", C.c_float),
        ("mass", C.c_float), ("thrust", C.c_float), ("goal_radius", C.c_float), ("step_penalty", C.c_float),
        ("spawn_y", C.c_float), ("lanes_per_env", C.c_int32), ("steps_in_flight", C.c_int32), ("host_threads", C.c_int32),
    ]


_lib = None


def load():
    """dlopen libshipsim.so and declare the prototypes.  Raises if the library is missing: no fallback."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ShipsimError("libshipsim.so not found at %s -- build it with `make -C %s` (needs nvcc); there is no "
                           "CPU fallback" % (LIB_PATH, os.path.join(HERE, "csrc")))
    L = C.CDLL(LIB_PATH)
    vp, i32, i64 = C.c_void_p, C.c_int32, C.c_int64
    L.shipsim_abi_version.restype = C.c_int
    L.shipsim_abi_version.argtypes = []
    L.shipsim_last_error.restype = C.c_char_p
    L.shipsim_last_error.argtypes = []
    L.shipsim_config_default.argtypes = [C.POINTER(Config)]
    L.shipsim_create.argtypes = [C.POINTER(Config), C.c_int, C.POINTER(vp)]
    L.shipsim_destroy.argtypes = [vp]
    L.shipsim_load_scenarios.argtypes = [vp, vp, vp, vp, i32, i32]
    L.shipsim_state_bytes.restype = C.c_size_t
    L.shipsim_state_bytes.argtypes = [vp]
    L.shipsim_stats_bytes.restype = C.c_size_t
    L.shipsim_stats_bytes.argtypes = [vp]
    L.shipsim_bind_state.argtypes = [vp, vp, vp, vp]
    L.shipsim_reset.argtypes = [vp, vp, vp, C.c_int, vp, vp]
    L.shipsim_step.argtypes = [vp, vp, C.c_int, i32, vp, vp, vp, vp]
    L.shipsim_step_chained.argtypes = [vp, vp, C.c_int, i32, vp, vp, vp, vp]
    L.shipsim_step_host.argtypes = [vp, vp, i32, vp, vp, vp, vp]
    L.shipsim_stats_read.argtypes = [vp, vp, C.c_int, vp]
    L.shipsim_set_state.argtypes = [vp, vp, vp, vp, vp, vp]
    L.shipsim_get_state.argtypes = [vp, vp, vp, vp, vp, vp]
    L.shipsim_set_max_steps.argtypes = [vp, i32]
    L.shipsim_generate_scenarios.argtypes = [vp, i32, C.c_uint64, i32, C.c_float, vp]
    L.shipsim_read_scenarios.argtypes = [vp, vp, vp, vp]
    L.shipsim_render.argtypes = [vp, i32, i32, i32, vp, vp]
    L.shipsim_assemble_history.argtypes = [vp, vp, vp, i64, i64]
    L.shipsim_expand_delta.argtypes = [vp, vp, vp, vp, vp, vp, vp, i32, i64, C.c_float, i32, i32]
    L.shipsim_host_traffic.argtypes = [vp, C.POINTER(i64), C.POINTER(i64)]
    L.shipsim_host_threads.argtypes = [vp, C.POINTER(i32)]
    L.shipsim_fresh_maps.argtypes = [vp, i32]
    L.shipsim_fresh_info.argtypes = [vp, C.POINTER(i32)]
    L.shipsim_scenario_weights.argtypes = [vp, vp, vp]
    L.shipsim_mlp_policy_forward.argtypes = [vp, i32, vp, vp, vp, vp, vp, vp, vp, vp, vp, vp]
    L.shipsim_gae.argtypes = [vp, vp, vp, i32, i32, C.c_float, C.c_float, vp, vp, vp]
    L.shipsim_gae_scored.argtypes = [vp, vp, vp, vp, i32, C.c_float, C.c_float, i32, i32, vp, vp, vp, vp, vp]
    L.shipsim_episode_log_bind.argtypes = [vp, vp, vp, i32, vp]
    L.shipsim_launch_count.argtypes = [vp, C.POINTER(i64)]
    L.shipsim_chained_count.argtypes = [vp, C.POINTER(i64)]
    L.shipsim_launch_shape.argtypes = [vp, C.POINTER(i32), C.POINTER(i32), C.POINTER(i32)]
    L.shipsim_launch_window.argtypes = [vp, C.POINTER(i32)]
    for name in SYMBOLS:
        fn = getattr(L, name)
        if name not in ("shipsim_last_error", "shipsim_state_bytes", "shipsim_stats_bytes", "shipsim_abi_version"):
            fn.restype = C.c_int
    _lib = L
    return L


def check(rc):
    """Map a shipsim_status to the exception the reference would raise for the same mistake."""
    if rc == 0:
        return
    msg = load().shipsim_last_error().decode("utf-8", "replace")
    if rc == -1:
        raise ValueError(msg)           # e.g. "history_size must be greater than zero" (ship_env.py:46-47)
    if rc == -4:
        raise NotImplementedError(msg)
    raise ShipsimError("libshipsim error %d: %s" % (rc, msg))


def default_config():
    cfg = Config()
    check(load().shipsim_config_default(C.byref(cfg)))
    return cfg
