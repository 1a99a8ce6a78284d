"""``WalkEnv`` -- drop-in for the reference's walking task (``bez_isaacgym/tasks/walk_env.py:37-620``) on the B200 kernels.

Same skeleton as ``KickEnv`` (K0 + ONE fused post-physics launch; GPU and host pipelines); what differs:

* layout -- the robot is the only actor: ``root_states`` is ``(N,13)``, 21 bodies (29 with cleats), the observation is 52 wide
  ``[dof_pos 18, dof_vel 18, imu 6, off_orn 2, feet 8]`` (``walk_env.py:1032-1050``), episodes last 10 s;
* the reward (``walk_env.py:827-997``): forward velocity towards the goal while far, posture terms once within 5 cm, fall
  (up-vector projection < 0.7), win state (4 conditions at once), out of bound (angle start->goal vs robot->goal > 1.5708);
  ``compute_bez_reward`` ZEROES ``bez_init_state`` in place (``:966-967``), so the out-of-bound angle is measured from the origin;
* reset -- ``reset_idx`` additionally redraws the goal: ``goal_x, goal_y = U(-2, 2)`` drawn per reset env but assigned as
  ``self.goal[env_ids, 0] = goal_x[0]`` (``walk_env.py:566-574``), i.e. EVERY env of a reset batch receives the batch's FIRST
  draw.  Kept bug for bug: one draw per step (Philox keyed (seed, step) alone, ``bezk_goal_uniforms``), written by the masked
  reset inside the fused kernel and by ``bezk_reset_idx_task`` for explicit id lists.

The kernel side is the ``BEZK_TASK_WALK`` instantiation of the tile kernel (``csrc/bezk_task.cu``, ``include/bezk.h``).
"""
import torch

from .kick_env import KickEnv


class WalkEnv(KickEnv):
    TASK = "walk"
    #: fell (up-vector projection < 0.7), reached (win state), out (out of bounds), timeout -- OrientEnv shares them
    OUTCOMES = ("fell", "reached", "out", "timeout")
    #: the fused step's reward terms (``set_rollout_targets(reward_terms=...)``): goal velocity (vel_fwd * 10, not close),
    #: uprightness (-dist_h), body velocity (-vel_s, close only), posture (-pos_s close, -(5 * pos_s) not close), termination
    REWARD_TERMS = ("goal_velocity", "uprightness", "body_velocity", "posture", "termination")

    def _read_task_cfg(self, env_cfg):
        """No ball actor (walk_env.py:146-149); the yaml carries no ``ballInitState``."""
        if "ballInitState" in env_cfg:
            raise ValueError("bez_walk / bez_orient have a single actor: remove env.ballInitState (or use KickEnv)")

    def _init_task_tensors(self, env_cfg, n, f32):
        self.initial_root_states = torch.tensor([self.bez_init_state], **f32).repeat((n, 1))      # walk_env.py:146-149
        self._zero_start_for_out_of_bound()

    def _zero_start_for_out_of_bound(self):
        """walk_env.py:966-967: the reward function zeroes ``bez_init_state`` in place before measuring the out-of-bound angle."""
        self.bez_init_xy.zero_()

    def _init_task_views(self, n):
        """No ball views (the reference's ``root_pos_ball`` etc. do not exist in walk_env.py)."""

    def _reset_goal_tensor(self):
        """``reset_idx`` redraws ``self.goal`` rows (walk_env.py:566-574)."""
        return self.goal
