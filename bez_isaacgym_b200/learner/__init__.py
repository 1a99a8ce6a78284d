"""rl_games-shaped learner math on the B200 kernels: RunningMeanStd, discount_values (GAE), advantage
normalisation and the fused PPO loss (forward + backward), and the player that scores a checkpoint.  Same names / argument meaning as rl_games==1.1.3 so
an ``A2CAgent`` can call them in place of its own (see INTEGRATION.md)."""
from .running_mean_std import RunningMeanStd
from .a2c_common import discount_values, normalize_advantages, swap_and_flatten01
from .losses import ppo_loss, PPOLossConfig
from .experience import ExperienceBuffer, PPODataset, SlabDataset
from .policy_head import policy_head
from .agent import A2CAgent, A2CNetwork, AdaptiveScheduler
from .episode_meter import EpisodeMeter, OutcomeMeter, RewardTerms
from .player import PpoPlayerContinuous

__all__ = ["RunningMeanStd", "discount_values", "normalize_advantages", "swap_and_flatten01",
           "ppo_loss", "PPOLossConfig", "ExperienceBuffer", "PPODataset", "SlabDataset", "policy_head", "A2CAgent", "A2CNetwork",
           "AdaptiveScheduler", "EpisodeMeter", "OutcomeMeter", "RewardTerms", "PpoPlayerContinuous"]
