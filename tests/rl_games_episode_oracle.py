"""torch-CPU restatement of rl_games==1.1.3's episode statistics (TEST INFRASTRUCTURE ONLY; RECALLED, not vendored, so parity is
unpinned): ``rl_games/algos_torch/torch_ext.py`` ``AverageMeter`` and the per-step bookkeeping of
``rl_games/common/a2c_common.py`` ``play_steps``.  The library's fused step (``bezk_post_physics_rollout_ep``) and meter fold
(``bezk_episode_meter_update``) are tested against it."""
import torch


class AverageMeter:
    """torch_ext.AverageMeter(in_shape=1, max_size): fp32 mean buffer, python-int current_size."""

    def __init__(self, in_shape=1, max_size=100):
        self.max_size = max_size
        self.current_size = 0
        self.mean = torch.zeros(in_shape, dtype=torch.float32)

    def clear(self):
        self.current_size = 0
        self.mean.fill_(0)

    def update(self, values):
        size = values.size()[0]
        if size == 0:
            return
        new_mean = torch.mean(values.float(), dim=0)
        self.update_from_mean(new_mean, size)

    def update_from_mean(self, new_mean, size):
        """The recurrence with ``new_mean`` given (fp32): what the fold does with the fp64 sum / count rounded to fp32."""
        size = max(0, min(size, self.max_size))
        old_size = min(self.max_size - size, self.current_size)
        size_sum = old_size + size
        self.current_size = size_sum
        self.mean = (self.mean * old_size + new_mean * size) / size_sum

    def get_mean(self):
        return self.mean.squeeze(0).cpu().numpy()


def episode_bookkeeping(current_rewards, current_lengths, rewards, dones, game_rewards, game_lengths, num_agents=1):
    """One env step of play_steps' episode statistics.  ``rewards``: the env's UNSHAPED rew_buf (N,); ``dones``: reset_buf (N,).
    ``current_rewards`` (N, 1) / ``current_lengths`` (N,) float32.  Returns the new (current_rewards, current_lengths)."""
    current_rewards = current_rewards + rewards.view(-1, 1)
    current_lengths = current_lengths + 1
    done_indices = dones.nonzero()[::num_agents]
    game_rewards.update(current_rewards[done_indices])
    game_lengths.update(current_lengths[done_indices])
    not_dones = 1.0 - dones.float()
    current_rewards = current_rewards * not_dones.unsqueeze(1)
    current_lengths = current_lengths * not_dones
    return current_rewards, current_lengths
