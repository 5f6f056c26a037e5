"""Configuration knobs of the batched ShipEnv.

Attribute names and defaults are the reference's (ship_gym/config.py:8-24) so that its training scripts can
keep doing ``gc = GameConfig; gc.SPEED = 30`` (train/stable_baselines/ppo.py:65-69, train/random.py:4-7):
the classes are used as mutable singletons there.  Unlike the reference, values are SNAPSHOTTED when an env
is constructed (`snapshot()`), so later mutation of the class does not reach into a live batch.
"""


class LidarConfig(object):
    """config.py:8-11.  The reference never reads it -- LiDAR is built with its constructor defaults
    (10 beams / 90 degrees / 100 units, models.py:29,149-150).  BatchedShipEnv honours it only when asked
    (`honour_lidar_config=True`); N_BEAMS may then be 1 to 32 (a frame is 6 + N_BEAMS values)."""
    N_BEAMS = 10
    DISTANCE = 100
    ANGULAR_SPREAD = 180


class EnvConfig(object):
    """config.py:14-17"""
    HISTORY_SIZE = 2
    MAX_STEPS = 1000
    LIDAR_CONFIG = LidarConfig


class GameConfig(object):
    """config.py:20-24.  FPS and DEBUG only drive pygame sleeping / drawing in the reference (game.py:195,
    200-204); they are accepted and ignored."""
    DEBUG = False
    FPS = 1000
    SPEED = 10
    BOUNDS = (600, 600)


# what LiDAR actually uses in the reference (models.py:29)
REFERENCE_LIDAR = dict(N_BEAMS=10, DISTANCE=100, ANGULAR_SPREAD=90)

BASE_DT = 0.1          # game.py:27
SPACE_DAMPING = 0.4    # game.py:270


def snapshot(game_config=None, env_config=None, honour_lidar_config=False):
    """Freeze the knob values (class or instance, attributes looked up like the reference does)."""
    gc = GameConfig if game_config is None else game_config
    ec = EnvConfig if env_config is None else env_config
    bounds = tuple(getattr(gc, "BOUNDS", GameConfig.BOUNDS))
    if len(bounds) != 2:
        raise ValueError("BOUNDS must be (width, height)")
    lidar = dict(REFERENCE_LIDAR)
    if honour_lidar_config:
        lc = getattr(ec, "LIDAR_CONFIG", LidarConfig)
        lidar = dict(N_BEAMS=int(lc.N_BEAMS), DISTANCE=float(lc.DISTANCE), ANGULAR_SPREAD=float(lc.ANGULAR_SPREAD))
    history = int(getattr(ec, "HISTORY_SIZE", EnvConfig.HISTORY_SIZE))
    if history < 1:
        raise ValueError("history_size must be greater than zero")         # ship_env.py:46-47
    return dict(
        W=float(bounds[0]), H=float(bounds[1]),
        speed=float(getattr(gc, "SPEED", GameConfig.SPEED)),
        fps=getattr(gc, "FPS", GameConfig.FPS), debug=bool(getattr(gc, "DEBUG", GameConfig.DEBUG)),
        history=history, max_steps=int(getattr(ec, "MAX_STEPS", EnvConfig.MAX_STEPS)),
        lidar=lidar,
    )
