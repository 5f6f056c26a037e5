"""ship_sim_gym_b200 -- B200-native batched drop-in for the CapAI/ship-sim-gym environment step.

Host layer (Python, torch tensors for device memory) over libshipsim.so (hand-written sm_100a CUDA kernels
behind the C ABI in include/shipsim.h).  There is no CPU fallback: constructing an env without the built
library or without a B200 raises.
"""
from .config import EnvConfig, GameConfig, LidarConfig  # noqa: F401
from .curriculum import Curriculum, CurriculumDriver, Lesson, LessonCondition, LevelReplay  # noqa: F401
from .scenario import ScenarioBank  # noqa: F401


def __getattr__(name):
    # torch is imported lazily so that config / scenario / curriculum stay usable in light-weight tools
    if name in ("BatchedShipEnv", "ShipEnv", "Discrete", "Box"):
        from . import env
        return getattr(env, name)
    raise AttributeError(name)
