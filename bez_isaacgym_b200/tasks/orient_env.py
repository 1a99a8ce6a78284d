"""``OrientEnv`` -- drop-in for the reference's turn-to-heading task (``bez_isaacgym/tasks/orient_env.py:37-620``).

Layout, reset and goal redraw as ``WalkEnv`` (one actor, 52-wide observation, 10 s episodes).  What differs:

* the heading columns are ``compute_off_angle`` = (cos, sin) of ``goal_angle - normalize_angle(yaw)``
  (``orient_env.py:719-733``) with a per-env ``goal_angle`` (N,1) tensor initialised from ``goalState.goal_angle``
  (``orient_env.py:145``);
* the reward (``orient_env.py:845-1014``): ``-0.5 |angle|`` while turning, posture terms once the SIGNED angle is below 0.05
  (the reference compares the signed value, kept), win state, out of bound = more than 0.3 m from the START position (so, unlike
  walk, ``bez_init_state`` is NOT zeroed), -5 penalty.

Kernel side: the ``BEZK_TASK_ORIENT`` instantiation of the tile kernel (``csrc/bezk_task.cu``, ``include/bezk.h``).
"""
import torch

from .walk_env import WalkEnv


class OrientEnv(WalkEnv):
    TASK = "orient"
    #: heading (|ang| * -0.5, not close), uprightness (-dist_h), body velocity (-vel_s, close only), posture (-pos_s close,
    #: -(0.05 * pos_s) not close), termination
    REWARD_TERMS = ("heading", "uprightness", "body_velocity", "posture", "termination")

    def _init_task_tensors(self, env_cfg, n, f32):
        super()._init_task_tensors(env_cfg, n, f32)
        self.goal_angle = torch.tensor([[float(env_cfg["goalState"]["goal_angle"])]], **f32).repeat((n, 1))    # orient_env.py:145

    def _zero_start_for_out_of_bound(self):
        """orient_env.py:985-999 measures the out-of-bound distance from the configured start: nothing is zeroed."""
