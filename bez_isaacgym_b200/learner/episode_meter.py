"""``EpisodeMeter`` -- rl_games' ``game_rewards`` / ``game_lengths`` meters (rl_games/algos_torch/torch_ext.py ``AverageMeter``,
v1.1.3, RECALLED) kept on the device and fed by the fused step's episode partials (``KickEnv.set_rollout_targets(
episode_returns=..., episode_lengths=..., episode_partials=...)``), so that the per-step bookkeeping needs no ``nonzero()`` and no
host synchronisation.  The meters of one pair share one (2,) buffer: ``update`` folds T steps of partials into both with one
launch (``bezk_episode_meter_update``)."""
import torch

from .. import ops


class EpisodeMeter:
    """``AverageMeter(1, games_to_track)``: mean of the last ``games_to_track`` finished episodes' values, in fp32 on the device.
    ``get_mean()`` is one device-to-host read and returns a numpy array of shape (1,) as rl_games does."""

    def __init__(self, games_to_track=100, device="cuda", _store=None, _index=0):
        if int(games_to_track) <= 0:
            raise ValueError("games_to_track must be positive")
        self.max_size = int(games_to_track)
        self.device = torch.device(device)
        if _store is None:
            _store = (torch.zeros(2, dtype=torch.float32, device=self.device), torch.zeros(2, dtype=torch.int64, device=self.device))
        self._mean2, self._size2 = _store
        self._index = _index

    @classmethod
    def pair(cls, games_to_track=100, device="cuda"):
        """(game_rewards, game_lengths) sharing one buffer: the returns and lengths meters one fold updates together."""
        rewards = cls(games_to_track, device)
        return rewards, cls(games_to_track, device, _store=(rewards._mean2, rewards._size2), _index=1)

    def update(self, partials, num_envs):
        """Fold (T, 3, ceil(num_envs/32)) float64 episode partials -- T consecutive steps -- into BOTH meters of the pair, step by
        step in order (rl_games calls ``update`` once per env step)."""
        w = (int(num_envs) + 31) // 32
        ops.episode_meter_update(partials, num_envs, self.max_size, self._mean2, self._size2, steps=partials.numel() // (3 * w))

    @property
    def current_size(self):
        return int(self._size2[self._index])

    def get_mean(self):
        return self._mean2[self._index:self._index + 1].cpu().numpy()

    def clear(self):
        """Both meters of the pair: they are only ever updated together."""
        self._mean2.zero_()
        self._size2.zero_()


class OutcomeMeter:
    """``AverageMeter(K, games_to_track)`` fed with one one-hot row per finished episode, over the outcome classes ``names`` (the
    env's ``OUTCOMES``): the share of the last ``games_to_track`` episodes that ended through each termination rule.  Kept on the
    device and fed by the fused step's outcome partials (``KickEnv.set_rollout_targets(episode_outcomes=...)``) with
    ``EpisodeMeter``'s recurrence and step order, so after the same updates ``current_size`` equals the game meters'."""

    def __init__(self, names, games_to_track=100, device="cuda"):
        from ..tasks import KickEnv, WalkEnv
        if int(games_to_track) <= 0:
            raise ValueError("games_to_track must be positive")
        self.names = tuple(names)
        # the fold takes the task whose classes these are (walk and orient share theirs)
        tasks = {KickEnv.OUTCOMES: KickEnv.TASK, WalkEnv.OUTCOMES: WalkEnv.TASK}
        if self.names not in tasks:
            raise ValueError(f"names must be the OUTCOMES of an env: {KickEnv.OUTCOMES} or {WalkEnv.OUTCOMES}")
        self.task = tasks[self.names]
        self.max_size = int(games_to_track)
        self.device = torch.device(device)
        self._mean = torch.zeros(len(self.names), dtype=torch.float32, device=self.device)
        self._size = torch.zeros(1, dtype=torch.int64, device=self.device)

    def update(self, partials, num_envs):
        """Fold (T, K, ceil(num_envs/32)) int32 outcome partials -- T consecutive steps -- step by step in order, one launch."""
        k, w = len(self.names), (int(num_envs) + 31) // 32
        ops.outcome_meter_update(partials, num_envs, self.task, self.max_size, self._mean, self._size,
                                 steps=partials.numel() // (k * w))

    @property
    def current_size(self):
        return int(self._size[0])

    def get_mean(self):
        """numpy (K,): the share of each class among the tracked episodes."""
        return self._mean.cpu().numpy()

    def as_dict(self):
        """name -> share, one device-to-host read."""
        return dict(zip(self.names, (float(x) for x in self.get_mean())))

    def clear(self):
        self._mean.zero_()
        self._size.zero_()


class RewardTerms:
    """The mean per env-step of each reward term ``names`` (the env's ``REWARD_TERMS``) over the last folded rollout, an fp64 (K,)
    vector on the device: ``update`` folds the fused step's per-warp term sums (``KickEnv.set_rollout_targets(reward_terms=...)``)
    of T steps over N envs into sum / (T * N) with one launch and no host synchronisation.  Summed over the terms it is the
    rollout's mean unshaped reward."""

    def __init__(self, names, device="cuda"):
        from ..tasks import KickEnv, OrientEnv, WalkEnv
        self.names = tuple(names)
        # the fold takes the task whose terms these are
        tasks = {env.REWARD_TERMS: env.TASK for env in (KickEnv, WalkEnv, OrientEnv)}
        if self.names not in tasks:
            raise ValueError(f"names must be the REWARD_TERMS of an env: {', '.join(map(str, tasks))}")
        self.task = tasks[self.names]
        self.device = torch.device(device)
        self._mean = torch.zeros(len(self.names), dtype=torch.float64, device=self.device)

    def update(self, partials, num_envs):
        """Fold (T, K, ceil(num_envs/32)) float64 term partials -- T consecutive steps -- into the means, replacing the last ones."""
        ops.reward_terms_update(partials, num_envs, self.task, self._mean)

    @property
    def mean(self):
        """(K,) float64 on the device."""
        return self._mean

    def as_dict(self):
        """name -> mean per env-step, one device-to-host read."""
        return dict(zip(self.names, self._mean.tolist()))


class GameTermMeter:
    """``AverageMeter(K, games_to_track)`` fed with one K-row per finished episode: that episode's return in each reward term
    ``names`` (the env's ``REWARD_TERMS``), so the means say what the last ``games_to_track`` games' mean return is made of.  Kept
    on the device and fed by the fused step's game term partials (``KickEnv.set_rollout_targets(game_term_returns=...,
    game_term_partials=...)``) together with the episode partials (their done counts), with ``EpisodeMeter``'s recurrence and step
    order, so after the same updates ``current_size`` equals the game meters'.  Summed over the terms the means are the mean game
    return up to fp32 rounding."""

    def __init__(self, names, games_to_track=100, device="cuda"):
        from ..tasks import KickEnv, OrientEnv, WalkEnv
        if int(games_to_track) <= 0:
            raise ValueError("games_to_track must be positive")
        self.names = tuple(names)
        # the fold takes the task whose terms these are
        tasks = {env.REWARD_TERMS: env.TASK for env in (KickEnv, WalkEnv, OrientEnv)}
        if self.names not in tasks:
            raise ValueError(f"names must be the REWARD_TERMS of an env: {', '.join(map(str, tasks))}")
        self.task = tasks[self.names]
        self.max_size = int(games_to_track)
        self.device = torch.device(device)
        self._mean = torch.zeros(len(self.names), dtype=torch.float32, device=self.device)
        self._size = torch.zeros(1, dtype=torch.int64, device=self.device)

    def update(self, ep_partials, term_partials, num_envs):
        """Fold (T, 3, W) float64 episode partials and (T, K, W) float64 game term partials, W = ceil(num_envs/32) -- T consecutive
        steps -- step by step in order, one launch."""
        k, w = len(self.names), (int(num_envs) + 31) // 32
        ops.game_terms_meter_update(ep_partials, term_partials, num_envs, self.task, self.max_size, self._mean, self._size,
                                    steps=term_partials.numel() // (k * w))

    @property
    def current_size(self):
        return int(self._size[0])

    def get_mean(self):
        """numpy (K,): each term's mean return per tracked game."""
        return self._mean.cpu().numpy()

    def as_dict(self):
        """name -> mean per game, one device-to-host read."""
        return dict(zip(self.names, (float(x) for x in self.get_mean())))

    def clear(self):
        self._mean.zero_()
        self._size.zero_()
