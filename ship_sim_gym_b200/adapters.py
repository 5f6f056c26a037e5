"""Vector-env adapters for the reference's callers (SURVEY.md §8 f1).

`ShipVecEnv` duck-types the stable-baselines 2.x `VecEnv` protocol that `SubprocVecEnv([make_env() ...])` provides
in train/stable_baselines/ppo.py:122-123 (`num_envs`, `observation_space`, `action_space`, `reset()`,
`step_async(actions)`, `step_wait() -> (obs [N,32], rews [N], dones [N], infos)`, `close()`), including its worker
semantics: the observation returned on a done step is already the reset observation.

`ShipVectorEnv` duck-types the RLlib 0.6 `VectorEnv` protocol (`vector_reset()`, `reset_at(i)`,
`vector_step(actions)`, `get_unwrapped()`) used by `tune.register_env(..., env_creator)` in train/rllib/ppo.py:21-24.

Neither library is a dependency (neither is installable here); the classes only implement the methods those
libraries call.  Both sit on one `BatchedShipEnv`, i.e. one GPU; numpy in / numpy out by default, CUDA tensors when
`as_tensors=True` (a policy that lives on the same GPU then never touches the host).
"""
import numpy as np
import torch

from . import _abi
from .env import BatchedShipEnv, end_truncated


def tile_images(images):
    """n pictures [h, w, c] -> one [rows * h, cols * w, c] picture, row-major, black where the grid has no picture
    (the layout of stable-baselines' tile_images: a near-square grid)."""
    imgs = np.stack(list(images))
    n, h, w, c = imgs.shape
    rows = int(np.ceil(np.sqrt(n)))
    cols = int(np.ceil(n / rows))
    pad = np.zeros((rows * cols - n, h, w, c), dtype=imgs.dtype)
    grid = np.concatenate([imgs, pad]).reshape(rows, cols, h, w, c).transpose(0, 2, 1, 3, 4)
    return grid.reshape(rows * h, cols * w, c)


def episode_infos(base, env, ret, length, truncated, rows):
    """The per-env info dicts of one step, as `Monitor` and the stable-baselines workers fill them: an env whose episode
    ended gets {'episode': {'r': return, 'l': length}, 'terminal_observation': row, 'TimeLimit.truncated': ended on the
    step cap alone}; the others keep their entry of `base` ({}).  env / ret / length / truncated: lists with one entry per
    finished episode (plain Python numbers: this runs once per step on the caller's critical path), rows: its terminal
    observations."""
    infos = list(base)
    for e, r, ln, tr, row in zip(env, ret, length, truncated, rows):
        infos[e] = {"episode": {"r": r, "l": ln}, "terminal_observation": row, "TimeLimit.truncated": tr}
    return infos


def log_infos(base, meta, rows):
    """episode_infos from raw episode-log records (int32 meta [n, 8], rows [n, D]; numpy; the rows are copied)."""
    meta = np.asarray(meta, dtype=np.int32)
    return episode_infos(base, meta[:, _abi.EP_ENV].tolist(), meta[:, _abi.EP_RETURN].view(np.float32).tolist(),
                         meta[:, _abi.EP_LENGTH].tolist(), end_truncated(meta[:, _abi.EP_END]).tolist(), np.array(rows, dtype=np.float32))


class ShipVecEnv(object):
    """stable-baselines `VecEnv` over a BatchedShipEnv (auto-reset on, like a SubprocVecEnv worker).

    episode_info=True: the info of an env whose episode ended on this step carries what `Monitor` and the later
    stable-baselines workers put there -- `episode` {r, l}, `terminal_observation`, `TimeLimit.truncated` -- from the
    kernels' episode log (BatchedShipEnv.enable_episode_log)."""

    def __init__(self, num_envs, game_config=None, env_config=None, as_tensors=False, episode_info=False, **kw):
        kw["auto_reset"] = True
        self.batch = BatchedShipEnv(num_envs, game_config, env_config, **kw)
        self.num_envs = self.batch.num_envs
        self.observation_space = self.batch.observation_space
        self.action_space = self.batch.action_space
        self.as_tensors = bool(as_tensors)
        self._pending = None
        self._infos = [{} for _ in range(self.num_envs)]       # ShipEnv.step's info is always {} (ship_env.py:156)
        self.episode_info = bool(episode_info)
        if self.episode_info:
            # numpy callers: the log lives in page-locked host memory, written by the kernel during the step; the step's
            # own wait makes it readable, and the number of new records is the number of done flags (one per finished
            # episode), so nothing else is read from the device.  The count is reset only when the log is nearly full.
            self._np_log = not self.as_tensors and self.batch.history <= 2
            self._log_cap = 64 * self.num_envs if self._np_log else self.num_envs
            self.batch.enable_episode_log(self._log_cap, pinned=self._np_log)
            self._log_used = 0
            if self._np_log:
                log = self.batch.episode_log
                self._log_np = (log.rows.numpy(), log.meta.numpy())

    def _out(self, t):
        return t if self.as_tensors else t.cpu().numpy()

    def reset(self):
        return self._out(self.batch.reset())

    def step_async(self, actions):
        if self._pending is not None:
            raise RuntimeError("step_async called twice without step_wait")
        if not self.as_tensors and not torch.is_tensor(actions) and self.batch.history <= 2:
            # a numpy caller: one call into the C ABI's host-buffer path (no torch ops; the work is done here)
            if self.episode_info and self._log_used + self.num_envs > self._log_cap:
                self.batch.episode_log.clear()             # (enqueued ahead of the step on the same stream)
                self._log_used = 0
            obs, rew, done = self.batch.step_np(np.asarray(actions))
            infos = None
            if self.episode_info:
                n = int(np.count_nonzero(done))
                rows, meta = self._log_np
                lo = self._log_used
                infos = log_infos(self._infos, meta[lo:lo + n], rows[lo:lo + n]) if n else self._infos
                self._log_used += n
            self._pending = (obs.copy(), rew.copy(), done.copy(), infos)
            return
        a = torch.as_tensor(np.asarray(actions) if not torch.is_tensor(actions) else actions)
        self._pending = self.batch.step(a)       # enqueued on the GPU; nothing is waited for here

    def step_wait(self):
        if self._pending is None:
            raise RuntimeError("step_wait called before step_async")
        obs, rew, done, infos = self._pending
        self._pending = None
        if isinstance(obs, np.ndarray):
            return obs, rew, done, infos if infos is not None else self._infos
        infos = self._infos
        if self.episode_info:                   # (tensor path: the records are read back from the device once per step)
            ep = self.batch.episodes()
            self._log_used = 0
            if ep["env"].numel():
                rows = ep["terminal_obs"] if self.as_tensors else ep["terminal_obs"].cpu().numpy()
                infos = episode_infos(self._infos, *(ep[k].tolist() for k in ("env", "return", "length", "truncated")), rows)
        return self._out(obs), self._out(rew), self._out(done), infos

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    def close(self):
        self.batch.close()

    # the rest of the VecEnv surface stable-baselines touches
    def get_images(self, max_envs=16, size=(150, 150)):
        """VecEnv.get_images: one RGB picture per env (uint8 [h, w, 3] numpy arrays), drawn on the device by
        shipsim_render the way ShipGame.render does (game.py:197-229).  At most `max_envs` pictures of `size` pixels: a
        batch of thousands is not something to look at."""
        n = min(self.num_envs, int(max_envs))
        return [self.batch.render("rgb_array", env_index=i, size=size).cpu().numpy() for i in range(n)]

    def render(self, mode="human", **kw):
        """VecEnv.render: the pictures of get_images tiled into one (stable-baselines' tile_images layout: a near-square
        grid, row-major) for mode 'rgb_array'; 'human' has no window to draw into and returns None."""
        if mode != "rgb_array":
            return None
        return tile_images(self.get_images(**kw))

    def seed(self, seed=None):
        return self.batch.seed(seed)

    @property
    def unwrapped(self):
        return self


class ShipVectorEnv(object):
    """RLlib `VectorEnv` over a BatchedShipEnv.  RLlib resets sub-envs itself (`reset_at`), so auto-reset is off."""

    def __init__(self, num_envs, game_config=None, env_config=None, **kw):
        kw["auto_reset"] = False
        self.batch = BatchedShipEnv(num_envs, game_config, env_config, **kw)
        self.num_envs = self.batch.num_envs
        self.observation_space = self.batch.observation_space
        self.action_space = self.batch.action_space

    def vector_reset(self):
        obs = self.batch.reset().cpu().numpy()
        return [obs[i] for i in range(self.num_envs)]

    def reset_at(self, index):
        mask = torch.zeros(self.num_envs, dtype=torch.uint8)
        mask[int(index)] = 1
        obs = self.batch.reset(mask=mask)
        return obs[int(index)].cpu().numpy()

    def vector_step(self, actions):
        obs, rew, done = self.batch.step_np(np.asarray(actions, dtype=np.int64))
        obs = obs.copy()
        n = self.num_envs
        return [obs[i] for i in range(n)], [float(rew[i]) for i in range(n)], [bool(done[i]) for i in range(n)], [{} for _ in range(n)]

    def get_unwrapped(self):
        return []

    def close(self):
        self.batch.close()
