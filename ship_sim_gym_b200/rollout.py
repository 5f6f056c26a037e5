"""On-device rollout collection: policy and envs on the same GPU, no host round-trip per step (BASELINE.json
configs[4], SURVEY.md §8d config 5).

The policy is the reference's: stable-baselines `MlpPolicy` as used at train/stable_baselines/ppo.py:88 -- two tanh
layers of 64 units each for the policy and for the value function -- here as a plain torch module.  One rollout =
T x (policy forward -> categorical sample -> fused env step); the env kernel reads the int64 action tensor the sampler
produced and writes obs / reward / done straight into the rollout buffers.  Because `shipsim_step` allocates nothing
and never synchronises, the whole rollout is captured once in a CUDA graph and replayed.
"""
import torch
import torch.nn as nn

from . import _abi
from .env import BatchedShipEnv


def score_levels(adv, dones, meta, count, scenario_now, call0, n_scenarios, steps_per_call=1, scenarios=None, scores=None):
    """The map of every rollout step and Prioritized Level Replay's value-loss sums per map -- shipsim_gae_scored's rule, in
    torch, on any device, with no host synchronisation.

    adv float [T, N], dones [T, N]; meta int32 [cap, 8] episode-log records (columns _abi.EP_*) of which the first `count`
    (a 1-element tensor) are valid; scenario_now int [N]: the map each env plays after the rollout.  The record of call c,
    step k is rollout step t = (c - call0) * steps_per_call + k; records whose t, env or scenario are out of range are
    ignored.  Walking backwards from step T - 1, an env's steps after its last done belong to scenario_now, and a done at
    t switches to the scenario of the record of (t, env) -- -1 if that record was lost.  Returns (scenarios int32 [T, N],
    scores float64 [n_scenarios + 1, 3]); the columns are _abi.SCORE_STEPS / SCORE_POS_ADV / SCORE_ABS_ADV, row
    n_scenarios collects the steps of no known map, and the sums are added into `scores` when given."""
    T, N = adv.shape
    dev = adv.device
    meta = meta.to(dev)
    k, env, scen = meta[:, _abi.EP_K].long(), meta[:, _abi.EP_ENV].long(), meta[:, _abi.EP_SCENARIO].long()
    t = (meta[:, _abi.EP_CALL].long() - call0) * steps_per_call + k
    ok = ((torch.arange(meta.shape[0], device=dev) < count.to(dev)) & (k >= 0) & (k < steps_per_call) & (t >= 0) & (t < T)
          & (env >= 0) & (env < N) & (scen >= 0) & (scen < n_scenarios))
    ended = torch.full((T * N + 1,), -1, dtype=torch.int32, device=dev)       # last slot: where the skipped records land
    ended.scatter_(0, torch.where(ok, t * N + env, T * N), torch.where(ok, scen, -1).to(torch.int32))
    ended = ended[:T * N].view(T, N)
    if scenarios is None:
        scenarios = torch.empty(T, N, dtype=torch.int32, device=dev)
    done = dones.bool()
    torch.where(done[T - 1], ended[T - 1], scenario_now.to(device=dev, dtype=torch.int32), out=scenarios[T - 1])
    for s in range(T - 2, -1, -1):
        torch.where(done[s], ended[s], scenarios[s + 1], out=scenarios[s])
    row = torch.where((scenarios >= 0) & (scenarios < n_scenarios), scenarios, n_scenarios).long().reshape(-1)
    a = adv.double().reshape(-1)
    cols = torch.stack([torch.ones_like(a), a.clamp_min(0.0), a.abs()], 1)
    if scores is None:
        scores = torch.zeros(n_scenarios + 1, _abi.SCORE_COLS, dtype=torch.float64, device=dev)
    scores.index_add_(0, row, cols)
    return scenarios, scores


class MlpPolicy(nn.Module):
    """stable-baselines MlpPolicy: pi 32 -> 64 -> 64 -> 3, vf 32 -> 64 -> 64 -> 1, tanh (separate trunks)."""

    def __init__(self, obs_dim=32, n_actions=3, hidden=64, obs_scale=1.0 / 600.0):
        super().__init__()
        self.obs_scale = obs_scale

        def trunk(out):
            return nn.Sequential(nn.Linear(obs_dim, hidden), nn.Tanh(), nn.Linear(hidden, hidden), nn.Tanh(), nn.Linear(hidden, out))
        self.pi = trunk(n_actions)
        self.vf = trunk(1)

    def forward(self, obs):
        x = obs * self.obs_scale
        return self.pi(x), self.vf(x).squeeze(-1)


class RolloutCollector(object):
    """Collects T-step rollouts of a BatchedShipEnv under a policy, entirely on the device.

    The loop is launch bound (16,384 envs: every kernel in it runs for a few microseconds), so it is written to launch
    as little as possible per step.  For an `MlpPolicy` the two trunks run as ONE three-layer network -- layer 1
    side by side (the observation scale folded into its weights), layers 2 and 3 block-diagonal -- through `addmm`
    into preallocated buffers: 3 GEMMs + 2 tanh per step instead of 6 + 4 + 1; the Gumbel noise of the whole rollout is
    drawn once; log-probabilities, values and the GAE deltas are computed for all steps at once after the loop, which
    leaves one fused multiply-add per step for the GAE recurrence.  Per step: 7 torch kernels + the env kernel -- or, for
    the reference's own shape (32 -> 64 -> 64 -> 3 | 1), ONE launch of the library's policy kernel (both trunks, heads and
    the Gumbel-max sample: `shipsim_mlp_policy_forward`) + the env kernel.
    Any other policy module (`forward(obs) -> (logits, value)`) takes the generic per-step path.

    episode_log=True: the env's episode log (BatchedShipEnv.enable_episode_log, room for T * N records: every env-step
    could end an episode) is emptied at the start of every rollout, inside the graph; episodes() returns the rollout's
    finished episodes with `t` = the rollout step -- what a PPO loop logs as ep_reward_mean / ep_len_mean.

    level_scores=True (implies episode_log=True): after every rollout `scenarios` (int32 [T, N]) holds the map every step
    played, and `level_scores` (float64 [n_scenarios + 1, 3], zeroed at the start of every rollout) per map the steps, the
    sum of max(advantage, 0) and the sum of |advantage| (columns _abi.SCORE_*; the last row: steps whose episode record was
    lost) -- Prioritized Level Replay's value-loss scores, for LevelReplay(score="positive_value_loss").  The kernel path
    computes them inside its GAE launch (shipsim_gae_scored), the generic path with score_levels."""

    def __init__(self, env, policy, T=128, gamma=0.99, lam=0.95, use_graph=True, use_kernel=True, episode_log=False, level_scores=False):
        assert isinstance(env, BatchedShipEnv) and env.history <= 2
        self.env, self.policy, self.T, self.gamma, self.lam = env, policy, int(T), gamma, lam
        N, D, dev = env.num_envs, env.states_history, env.device
        f32 = dict(dtype=torch.float32, device=dev)
        self.obs = torch.empty(T + 1, N, D, **f32)              # obs[t] is what the policy sees at step t
        self.actions = torch.empty(T, N, dtype=torch.int64, device=dev)
        self.logp = torch.empty(T, N, **f32)
        self.values = torch.empty(T + 1, N, **f32)
        self.rewards = torch.empty(T, N, **f32)
        self.dones = torch.empty(T, N, dtype=torch.uint8, device=dev)
        self.adv = torch.empty(T, N, **f32)
        self.returns = torch.empty(T, N, **f32)
        self.use_graph = bool(use_graph)
        self._graph = None
        self._graph_epoch = -1
        self._fused = isinstance(policy, MlpPolicy)
        self._kernel = False
        if self._fused:
            lin = [policy.pi[0], policy.pi[2], policy.pi[4], policy.vf[0], policy.vf[2], policy.vf[4]]
            H, A = lin[0].out_features, lin[2].out_features
            assert lin[0].in_features == D and lin[3].out_features == H and lin[5].out_features == 1
            self._alloc_fused(N, D, H, A, T, f32)
            self._z = torch.empty(N, A, **f32)
            # the library's fused policy kernel (shipsim_mlp_policy_forward) has the reference's shape built in
            self._kernel = bool(use_kernel) and (D, H, A) == (32, 64, 3)
        self._noise = torch.empty(T, N, policy.pi[4].out_features if self._fused else 3, **f32)
        self._a_spare = torch.empty(N, dtype=torch.int64, device=dev)
        self._nonterm = torch.empty(T, N, **f32)
        self._coef = torch.empty(T, N, **f32)
        self._delta = torch.empty(T, N, **f32)
        env.validate_actions = False                            # the range check would need a host sync per step
        self._scored = bool(level_scores)
        self.episode_log = bool(episode_log) or self._scored
        self._call0 = 0                                         # the env's step-call number of the rollout's first launch
        self.scenarios = self.level_scores = None
        if self._scored:
            self.scenarios = torch.empty(T, N, dtype=torch.int32, device=dev)
            self._alloc_scores()
        if self.episode_log:
            env.enable_episode_log(self.T * N)
        self.obs[0].copy_(env.reset())
        self._seen_reset_epoch = env.reset_epoch

    def _alloc_scores(self):
        """The level-score table of the env's current bank (a bank of another size replaces it)."""
        self.level_scores = torch.zeros(self.env.n_scenarios + 1, _abi.SCORE_COLS, dtype=torch.float64, device=self.env.device)

    def _alloc_fused(self, N, D, H, A, T, f32):
        self._H, self._A = H, A
        self._W1, self._b1 = torch.empty(D, 2 * H, **f32), torch.empty(2 * H, **f32)             # [pi | vf] side by side
        self._W2, self._b2 = torch.zeros(2 * H, 2 * H, **f32), torch.empty(2 * H, **f32)           # block-diagonal
        self._W2p = torch.empty(2, H, H, **f32)                                                    # the two blocks, packed (policy kernel)
        self._W3, self._b3 = torch.zeros(2 * H, A + 1, **f32), torch.empty(A + 1, **f32)           # pi -> columns 0..A-1, vf -> column A
        self._h1, self._h2 = torch.empty(N, 2 * H, **f32), torch.empty(N, 2 * H, **f32)
        self._out = torch.empty(T + 1, N, A + 1, **f32)         # logits | value of every step

    def _refresh_fused(self):
        """The policy's current parameters, laid out as one network (weights transposed for x @ W)."""
        pi, vf, H, A = self.policy.pi, self.policy.vf, self._H, self._A
        self._W1[:, :H].copy_(pi[0].weight.t()); self._W1[:, H:].copy_(vf[0].weight.t())
        self._W1.mul_(self.policy.obs_scale)
        self._b1[:H].copy_(pi[0].bias); self._b1[H:].copy_(vf[0].bias)
        self._W2[:H, :H].copy_(pi[2].weight.t()); self._W2[H:, H:].copy_(vf[2].weight.t())
        self._W2p[0].copy_(pi[2].weight.t()); self._W2p[1].copy_(vf[2].weight.t())
        self._b2[:H].copy_(pi[2].bias); self._b2[H:].copy_(vf[2].bias)
        self._W3[:H, :A].copy_(pi[4].weight.t()); self._W3[H:, A:].copy_(vf[4].weight.t())
        self._b3[:A].copy_(pi[4].bias); self._b3[A:].copy_(vf[4].bias)

    def _forward_fused(self, t):
        """Three GEMMs and two tanh for both trunks.  (Two-entry batched GEMMs for layers 2 and 3, which skip the zero
        blocks, were measured and are slower at 16,384 envs: 8.8 against 8.5 ms per 128-step rollout.)"""
        torch.addmm(self._b1, self.obs[t], self._W1, out=self._h1).tanh_()
        torch.addmm(self._b2, self._h1, self._W2, out=self._h2).tanh_()
        torch.addmm(self._b3, self._h2, self._W3, out=self._out[t])

    def _forward_kernel(self, t):
        """Both trunks, the heads and the Gumbel-max sample of step t in ONE launch of the library's policy kernel
        (csrc/shipsim_policy.cu): logits | value -> _out[t], action -> actions[t] (t = T: values only, sample discarded)."""
        from . import _abi
        env = self.env
        act = self.actions[t] if t < self.T else self._a_spare
        nz = self._noise[t] if t < self.T else self._noise[0]
        with torch.cuda.device(env.device):
            _abi.check(env.L.shipsim_mlp_policy_forward(self.obs[t].data_ptr(), env.num_envs, self._W1.data_ptr(), self._b1.data_ptr(),
                                                        self._W2p.data_ptr(), self._b2.data_ptr(), self._W3.data_ptr(), self._b3.data_ptr(),
                                                        nz.data_ptr(), self._out[t].data_ptr(), act.data_ptr(), env._stream()))

    @torch.no_grad()
    def _collect(self):
        env, T = self.env, self.T
        if self.episode_log:
            env.episode_log.clear()
            # (a replayed graph repeats the call numbers of its capture: this value is the capture's, like the records')
            self._call0 = env._calls
        if self._scored:
            self.level_scores.zero_()
        # categorical sampling by Gumbel-max (no host sync, graph-capturable): the noise of the whole rollout at once
        self._noise.uniform_().clamp_(1e-10, 1.0).log_().neg_().log_().neg_()
        if self._fused:
            A = self._A
            self._refresh_fused()
            for t in range(T):
                if self._kernel:                            # 2 launches per step: policy + sample, env step
                    self._forward_kernel(t)
                else:
                    self._forward_fused(t)
                    torch.add(self._out[t, :, :A], self._noise[t], out=self._z)
                    torch.argmax(self._z, dim=-1, out=self.actions[t])
                env.rollout(self.actions[t:t + 1], out=(self.obs[t + 1:t + 2], self.rewards[t:t + 1], self.dones[t:t + 1]))
            if self._kernel:
                self._forward_kernel(T)
            else:
                self._forward_fused(T)
            self.values.copy_(self._out[:, :, A])
            self.logp.copy_(torch.log_softmax(self._out[:T, :, :A], dim=-1).gather(-1, self.actions[:, :, None]).squeeze(-1))
        else:
            for t in range(T):
                logits, v = self.policy(self.obs[t])
                a = torch.argmax(logits + self._noise[t], dim=-1)
                self.actions[t].copy_(a)
                self.logp[t].copy_(torch.log_softmax(logits, dim=-1).gather(-1, a[:, None]).squeeze(-1))
                self.values[t].copy_(v)
                env.rollout(self.actions[t:t + 1], out=(self.obs[t + 1:t + 2], self.rewards[t:t + 1], self.dones[t:t + 1]))
            _, v = self.policy(self.obs[T])
            self.values[T].copy_(v)
        if self._kernel and self._scored:               # GAE + the map of every step + the per-map sums, one GAE launch
            with torch.cuda.device(env.device):
                _abi.check(env.L.shipsim_gae_scored(env._h, self.rewards.data_ptr(), self.values.data_ptr(), self.dones.data_ptr(), T,
                                                    float(self.gamma), float(self.lam), self._call0, 1, self.adv.data_ptr(),
                                                    self.returns.data_ptr(), self.scenarios.data_ptr(), self.level_scores.data_ptr(),
                                                    env._stream()))
        elif self._kernel:                              # one launch (shipsim_gae) instead of ~T + 8 elementwise kernels
            with torch.cuda.device(env.device):
                _abi.check(env.L.shipsim_gae(self.rewards.data_ptr(), self.values.data_ptr(), self.dones.data_ptr(), T, env.num_envs,
                                             float(self.gamma), float(self.lam), self.adv.data_ptr(), self.returns.data_ptr(), env._stream()))
        else:
            self._gae()
            if self._scored:
                log = env.episode_log
                score_levels(self.adv, self.dones, log.meta, log.count, env.state[4, :, 2].view(torch.int32), self._call0, env.n_scenarios,
                             scenarios=self.scenarios, scores=self.level_scores)

    def _gae(self):
        """GAE(lambda), as PPO2 computes it: adv[t] = delta[t] + gamma * lam * nonterminal[t] * adv[t + 1], with the deltas
        of all steps computed at once."""
        T = self.T
        torch.sub(1.0, self.dones, out=self._nonterm)
        torch.mul(self._nonterm, self.gamma * self.lam, out=self._coef)
        torch.mul(self.values[1:], self._nonterm, out=self._delta)
        self._delta.mul_(self.gamma).add_(self.rewards).sub_(self.values[:T])
        self.adv[T - 1].copy_(self._delta[T - 1])
        for t in range(T - 2, -1, -1):
            torch.addcmul(self._delta[t], self._coef[t], self.adv[t + 1], out=self.adv[t])
        torch.add(self.adv, self.values[:T], out=self.returns)

    def episodes(self):
        """The episodes that finished during the last rollout (BatchedShipEnv.episodes), plus `t` = the rollout step at
        which each ended (0 .. T-1)."""
        if not self.episode_log:
            raise RuntimeError("RolloutCollector(episode_log=True) keeps the episode log")
        ep = self.env.episodes(clear=False)
        ep["t"] = ep["call"] - self._call0
        return ep

    def collect(self):
        """One rollout; the buffers (obs, actions, logp, values, rewards, dones, adv, returns) hold the result.
        The captured graph freezes the kernel parameters (StepParams travels by value: episode cap, scenario-bank
        pointers, ...), so it is dropped and captured again whenever the env's `params_epoch` has moved -- after
        set_max_steps / load_scenarios / generate_scenarios, e.g. from a CurriculumDriver between rollouts."""
        if self._seen_reset_epoch != self.env.reset_epoch:
            # the batch was reset behind the collector's back (a bank swap resets every env): go on from that observation
            if self.env.last_reset_obs is not None:
                self.obs[0].copy_(self.env.last_reset_obs)
            self._seen_reset_epoch = self.env.reset_epoch
        if self._scored and self.level_scores.shape[0] != self.env.n_scenarios + 1:
            self._alloc_scores()                        # (a new bank also moved params_epoch: the graph is captured again)
        if not self.use_graph or not self.env.graph_safe:     # (fresh maps: the pick slice moves between launches)
            self._collect()
        else:
            if self._graph is not None and self._graph_epoch != self.env.params_epoch:
                self._graph = None
            if self._graph is None:
                self._graph_epoch = self.env.params_epoch
                steps_before = self.env.total_steps
                s = torch.cuda.Stream(device=self.env.device)
                s.wait_stream(torch.cuda.current_stream(self.env.device))
                with torch.cuda.stream(s):
                    self._collect()                             # warm-up outside capture (cuBLAS handles, allocator)
                    self.obs[0].copy_(self.obs[self.T])
                torch.cuda.current_stream(self.env.device).wait_stream(s)
                call0 = self._call0
                self._graph = torch.cuda.CUDAGraph()
                with torch.cuda.graph(self._graph):
                    self._collect()
                    self.obs[0].copy_(self.obs[self.T])         # next rollout continues where this one ended
                # the capture pass enqueued nothing: only the warm-up rollout ran
                self.env.total_steps = steps_before + self.T * self.env.num_envs
                self._graph_call0, self._call0 = self._call0, call0
                return self
            self._graph.replay()
            self._call0 = self._graph_call0
            self.env.total_steps += self.T * self.env.num_envs
            return self
        self.obs[0].copy_(self.obs[self.T])
        return self
