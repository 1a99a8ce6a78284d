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
