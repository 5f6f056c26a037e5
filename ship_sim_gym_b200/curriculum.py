"""Scalar lesson schedule with the semantics of the reference helper (ship_gym/curriculum.py:23-50), which
nothing in the reference imports.  Here `progress()` is meant to be fed the all-reduced mean episode return
(BatchedShipEnv.stats()) and `int(c)` / `float(c)` to select e.g. MAX_STEPS or a scenario-bank tier.

Kept quirks (SURVEY.md App. B Q27): the pass test is strict (`val > condition`), the counter is NOT reset
by a failing call, so a lesson advances on the (repeat_condition + 1)-th passing call, consecutive or not.
"""
import enum


class LessonCondition(enum.Enum):
    STEPS = 0
    REWARD = 1


class Lesson(object):
    """A bundle of thresholds; passed when every tracked value reaches its threshold (curriculum.py:7-20)."""

    def __init__(self, param_dict):
        self.param_dict = dict(param_dict)

    def pass_lesson(self, val_dict):
        return all(val_dict[k] >= v for k, v in self.param_dict.items())


class Curriculum(object):
    def __init__(self, values, conditions, repeat_condition=1):
        self.values = list(values)
        self.conditions = list(conditions)
        self.repeat_condition = repeat_condition
        self.lesson = 0
        self.repeat_reached = 0

    def __int__(self):
        return int(self.values[self.lesson])

    def __float__(self):
        return float(self.values[self.lesson])

    @property
    def value(self):
        return self.values[self.lesson]

    def progress(self, val):
        """Feed one measurement; returns True when it moved the curriculum to the next lesson."""
        if self.lesson >= len(self.conditions) or not (val > self.conditions[self.lesson]):
            return False
        self.repeat_reached += 1
        if self.repeat_reached <= self.repeat_condition:
            return False
        self.lesson += 1
        self.repeat_reached = 0
        return True


class CurriculumDriver(object):
    """Wires a `Curriculum` to a batched env (SURVEY.md §8 f3; the reference defines the helper but never uses it).

    After every rollout call `update()`: the episode statistics of all ranks are summed (one all-reduce of 16 doubles),
    the global mean episode return is fed to `Curriculum.progress`, and when that advances the lesson the new lesson's
    value is applied:
      * `knob="max_steps"`: the value is the new EnvConfig.MAX_STEPS (config.py:16);
      * `knob="bank"`: the value indexes `banks`, a list of ScenarioBank difficulty tiers, which is uploaded.
    Lessons only advance when at least `min_episodes` episodes finished since the last update (otherwise the mean is
    noise and the statistics keep accumulating).
    """

    def __init__(self, env, curriculum, knob="max_steps", banks=None, min_episodes=1, all_reduce=None):
        if knob not in ("max_steps", "bank"):
            raise ValueError("knob must be 'max_steps' or 'bank'")
        if knob == "bank" and not banks:
            raise ValueError("knob='bank' needs the list of scenario-bank tiers")
        self.env, self.curriculum, self.knob, self.banks = env, curriculum, knob, banks
        self.min_episodes = min_episodes
        self.all_reduce = all_reduce
        self.history = []
        self._apply()

    def _apply(self):
        if self.knob == "max_steps":
            self.env.set_max_steps(int(self.curriculum))
        else:
            self.env.load_scenarios(self.banks[int(self.curriculum)])

    def update(self):
        """Returns (advanced, mean_return or None)."""
        stats = self.env.stats_tensor(clear=False)
        if self.all_reduce is not None:
            stats = self.all_reduce(stats.clone())
        v = stats.tolist()
        episodes, return_sum = float(v[0]), float(v[1])
        if episodes < self.min_episodes:
            return False, None
        self.env.stats_tensor(clear=True)
        mean_return = return_sum / episodes
        advanced = self.curriculum.progress(mean_return)
        self.history.append((self.curriculum.lesson, mean_return, episodes))
        if advanced:
            self._apply()
        return advanced, mean_return


def replay_distribution(score, played, last, clock, rho=0.1, beta=0.1):
    """Prioritized Level Replay's replay distribution (Jiang et al., 2021) over the maps of a bank, as torch tensors on any
    device: P = (1 - rho) * P_score + rho * P_stale, with P_score proportional to (1 / rank) ** (1 / beta) -- rank 1 = the
    highest `score`; maps not `played` yet all share rank 1, ahead of every played map -- and P_stale proportional to
    clock - last (the episodes played since the map was last played; uniform while that is 0 everywhere)."""
    import torch
    n = score.numel()
    key = torch.where(played, score.double(), torch.full_like(score, float("inf"), dtype=torch.float64))
    order = torch.sort(key, descending=True, stable=True).indices
    pos = torch.empty(n, dtype=torch.float64, device=score.device)
    pos.scatter_(0, order, torch.arange(1, n + 1, dtype=torch.float64, device=score.device))
    rank = torch.where(played, pos, torch.ones_like(pos))
    p_score = rank.pow(-1.0 / beta)
    p_score = p_score / p_score.sum()
    stale = (clock - last).double().clamp_min(0.0)
    total = stale.sum()
    p_stale = torch.where(total > 0, stale / total.clamp_min(1.0), torch.full_like(stale, 1.0 / n))
    return (1.0 - rho) * p_score + rho * p_stale


class LevelReplay(object):
    """Prioritized Level Replay (Jiang et al., 2021) over the env's scenario bank: the maps the policy still does badly on
    are replayed more often, through the env's scenario weights (BatchedShipEnv.set_scenario_weights).

    After every rollout call `update()`: the env's episode log is folded into per-map outcomes
    (BatchedShipEnv.scenario_outcomes, which empties the log), optionally summed over ranks by `all_reduce` (a callable
    that takes a float64 table -- the [n_scenarios, 7] outcomes, and for the value-loss scores also the [n_scenarios + 1,
    3] level scores -- and returns the global one, e.g. an all-reduce(SUM) -- so that every rank holds the same weights
    and the picks stay independent of the sharding), and the replay distribution (replay_distribution) becomes the env's
    pick weights.  No host synchronisation: with a captured RolloutCollector graph the next replay plays the new weights.

    The score of a map is the exponential moving average (factor `alpha`) of a per-rollout score, chosen by `score`:
      * "positive_value_loss": PLR's default, the mean over the map's steps of max(GAE advantage, 0) -- high where the
        value function still underestimates what the policy achieves, i.e. where there is still something to learn;
      * "l1_value_loss": the mean over the map's steps of |GAE advantage|;
      * "return": minus the mean return of the map's finished episodes -- low returns, high priority.
    The value-loss scores read `update(scores)`, the `level_scores` table of a RolloutCollector(level_scores=True), which
    attributes every step of the rollout to its map, so a map played only by an episode that has not finished yet is
    scored too.  Whether a map has been played, and its staleness, count finished episodes for every score.
    `table` accumulates the global per-map outcomes of every update (columns env.OUTCOME_COLUMNS)."""

    SCORES = ("return", "positive_value_loss", "l1_value_loss")

    def __init__(self, env, rho=0.1, beta=0.1, alpha=0.5, all_reduce=None, score="return"):
        import torch
        if env.episode_log is None:
            raise ValueError("LevelReplay reads the episode log: call env.enable_episode_log() or use RolloutCollector(episode_log=True)")
        if not (0.0 <= rho <= 1.0 and beta > 0.0 and 0.0 < alpha <= 1.0):
            raise ValueError("need 0 <= rho <= 1, beta > 0 and 0 < alpha <= 1")
        if score not in self.SCORES:
            raise ValueError("score must be one of %s" % (self.SCORES,))
        self.env, self.rho, self.beta, self.alpha, self.all_reduce = env, rho, beta, alpha, all_reduce
        self.score_name = score
        n, f64 = env.n_scenarios, dict(dtype=torch.float64, device=env.device)
        self.table = torch.zeros(n, 7, **f64)
        self.score = torch.zeros(n, **f64)
        self.scored = torch.zeros(n, dtype=torch.bool, device=env.device)     # `score` holds a value for the map
        self.played = torch.zeros(n, dtype=torch.bool, device=env.device)
        self.last = torch.zeros(n, **f64)              # value of `clock` when the map was last played
        self.clock = torch.zeros((), **f64)            # episodes played so far (all ranks)

    def observe(self, outcomes, scores=None):
        """Fold one global per-map outcome table (float64 [n_scenarios, 7]) and, for the value-loss scores, one global
        level-score table (float64 [n_scenarios + 1, 3], RolloutCollector.level_scores) into the scores and staleness."""
        import torch
        from . import _abi
        self.table += outcomes
        ep = outcomes[:, 0]
        hit = ep > 0
        if self.score_name == "return":
            new, s = hit, -outcomes[:, 1] / ep.clamp_min(1.0)
        else:
            steps = scores[:ep.numel(), _abi.SCORE_STEPS]
            col = _abi.SCORE_POS_ADV if self.score_name == "positive_value_loss" else _abi.SCORE_ABS_ADV
            new, s = steps > 0, scores[:ep.numel(), col] / steps.clamp_min(1.0)
        self.score = torch.where(new, torch.where(self.scored, (1.0 - self.alpha) * self.score + self.alpha * s, s), self.score)
        self.scored |= new
        self.played |= hit
        self.clock += ep.sum()
        self.last = torch.where(hit, self.clock, self.last)

    def probabilities(self):
        return replay_distribution(self.score, self.played, self.last, self.clock, self.rho, self.beta)

    def update(self, scores=None):
        """Fold the rollout's episodes -- and for the value-loss scores `scores`, the collector's level_scores -- and set
        the env's scenario weights; returns the replay distribution (device tensor)."""
        if self.score_name == "return":
            scores = None
        elif scores is None:
            raise ValueError("score=%r needs the rollout's level scores: update(RolloutCollector(level_scores=True).level_scores)"
                             % self.score_name)
        outcomes = self.env.scenario_outcomes(clear=True)
        if self.all_reduce is not None:
            outcomes = self.all_reduce(outcomes)
            if scores is not None:
                scores = self.all_reduce(scores.clone())    # (an in-place all-reduce leaves the collector's table alone)
        self.observe(outcomes, scores)
        p = self.probabilities()
        self.env.set_scenario_weights(p)
        return p
