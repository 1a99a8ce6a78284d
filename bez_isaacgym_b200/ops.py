"""torch-facing shims over the C ABI: validate dtype / device / contiguity, pass raw device pointers and the
current CUDA stream to libbezk.so.  Every function launches hand-written sm_100a kernels; none has a
CPU or torch fallback (CPU tensors raise)."""
import ctypes as C
import math

import torch

from . import _lib
from . import bez_model as bm
from ._lib import BezkNoiseCfg, BezkPpoCfg, BezkRolloutCfg, BezkTaskCfg, BezkError


def _stream(t: torch.Tensor):
    dev = t.device if t.is_cuda else torch.device("cuda", torch.cuda.current_device())
    return C.c_void_p(torch.cuda.current_stream(dev).cuda_stream)


def _p(t, dtype, name, numel=None, allow_none=False):
    if t is None:
        if allow_none:
            return None
        raise BezkError(f"{name} is None")
    if not isinstance(t, torch.Tensor):
        raise BezkError(f"{name} must be a torch.Tensor")
    if not t.is_cuda and not (t.device.type == "cpu" and t.is_pinned()):
        # pinned host memory is device-accessible (UVA): the kernels may gather from / write to it over PCIe
        raise BezkError(f"{name} is on {t.device}: bez_isaacgym_b200 ops run on CUDA only (no CPU fallback); "
                        "host tensors must be pinned")
    if t.dtype != dtype:
        raise BezkError(f"{name} must be {dtype}, got {t.dtype}")
    if not t.is_contiguous():
        raise BezkError(f"{name} must be contiguous")
    if numel is not None and t.numel() != numel:
        raise BezkError(f"{name} has {t.numel()} elements, expected {numel}")
    return C.c_void_p(t.data_ptr())


def make_task_cfg(num_bodies=bm.BODIES_NO_CLEATS, cleats=False, dt=0.01667, max_episode_length=900,
                  clip_actions=3.9, clip_obs=math.inf, default_dof_pos=None, dof_lower=bm.DOF_LOWER,
                  dof_upper=bm.DOF_UPPER, bez_init_xy=(0.0, 0.0), write_contact_filter=True,
                  reset_root_states=True, imu_body=bm.IMU_BODY, left_foot_body=None, right_foot_body=None,
                  imu_max_lin_acc=bm.IMU_MAX_LIN_ACC, imu_max_ang_vel=bm.IMU_MAX_ANG_VEL,
                  reset_pos_noise=0.15, reset_vel_noise=0.1) -> BezkTaskCfg:
    """Build the by-value kernel constant block from the quantities ``KickEnv.__init__`` derives
    (reference ``bez_isaacgym/tasks/kick_env.py:46-238``)."""
    if default_dof_pos is None:
        from .synthetic_gym import READY_POSE
        default_dof_pos = READY_POSE
    c = BezkTaskCfg()
    c.num_bodies = int(num_bodies)
    c.imu_body = int(imu_body)
    if left_foot_body is None:
        left_foot_body = bm.LEFT_CLEATS[0] if cleats else bm.LEFT_FOOT_BODY
    if right_foot_body is None:
        right_foot_body = bm.RIGHT_CLEATS[0] if cleats else bm.RIGHT_FOOT_BODY
    c.left_foot_body, c.right_foot_body = int(left_foot_body), int(right_foot_body)
    c.max_episode_length = int(max_episode_length)
    c.flags = ((_lib.F_CLEATS if cleats else 0) | (_lib.F_WRITE_CONTACT_FILTER if write_contact_filter else 0)
               | (_lib.F_RESET_ROOT_STATES if reset_root_states else 0))
    c.dt = dt
    c.imu_max_lin_acc, c.imu_max_ang_vel = imu_max_lin_acc, imu_max_ang_vel
    c.clip_obs, c.clip_actions = clip_obs, clip_actions
    c.bez_init_xy[0], c.bez_init_xy[1] = bez_init_xy
    # torch_rand_float(lo, hi): (hi - lo) is formed in double, then multiplies an fp32 tensor
    c.reset_pos_lo, c.reset_pos_span = -reset_pos_noise, reset_pos_noise - (-reset_pos_noise)
    c.reset_vel_lo, c.reset_vel_span = -reset_vel_noise, reset_vel_noise - (-reset_vel_noise)
    lo, hi = list(dof_lower), list(dof_upper)
    for j in range(bm.NUM_DOF):
        if lo[j] > hi[j]:                         # kick_env.py:395-397
            lo[j], hi[j] = hi[j], lo[j]
        c.default_dof_pos[j] = float(default_dof_pos[j])
        c.dof_lower[j], c.dof_upper[j] = float(lo[j]), float(hi[j])
    return c


F32, F64, I64, U8 = torch.float32, torch.float64, torch.int64, torch.uint8


def set_l2_fetch_granularity(nbytes=32):
    """cudaLimitMaxL2FetchGranularity hint for the current device; returns the value in effect."""
    got = C.c_int32(0)
    _lib.check(_lib.load().bezk_set_l2_fetch_granularity(int(nbytes), C.byref(got)), "bezk_set_l2_fetch_granularity")
    return got.value


# ------------------------------------------------------------------------------------------- task
def pre_physics(actions, targets, cfg: BezkTaskCfg, actions_out=None):
    n = actions.shape[0]
    lib = _lib.load()
    _lib.check(lib.bezk_pre_physics(_p(actions, F32, "actions", n * 18), _p(actions_out, F32, "actions_out", n * 18, True),
                                    _p(targets, F32, "targets", n * 18), C.byref(cfg), n, _stream(actions)),
               "bezk_pre_physics")
    return targets


def compute_observations(dof_state, rigid_body, root_states, net_contact, goal, ball_init, cfg, obs,
                         prev_lin_vel=None, obs_clipped=None):
    n = obs.shape[0]
    nb = cfg.num_bodies
    lib = _lib.load()
    _lib.check(lib.bezk_compute_observations(
        _p(dof_state, F32, "dof_state", n * 36), _p(rigid_body, F32, "rigid_body", n * nb * 13),
        _p(root_states, F32, "root_states", n * 26), _p(net_contact, F32, "net_contact", n * nb * 3),
        _p(prev_lin_vel, F32, "prev_lin_vel", n * 3, True), _p(goal, F32, "goal", n * 2),
        _p(ball_init, F32, "ball_init", n * 2), C.byref(cfg), _p(obs, F32, "obs", n * 54),
        _p(obs_clipped, F32, "obs_clipped", n * 54, True), n, _stream(obs)), "bezk_compute_observations")
    return obs


def compute_reward(dof_state, rigid_body, root_states, goal, ball_init, reset_in, progress, cfg, rew, reset_out):
    n = rew.shape[0]
    nb = cfg.num_bodies
    lib = _lib.load()
    _lib.check(lib.bezk_compute_reward(
        _p(dof_state, F32, "dof_state", n * 36), _p(rigid_body, F32, "rigid_body", n * nb * 13),
        _p(root_states, F32, "root_states", n * 26), _p(goal, F32, "goal", n * 2),
        _p(ball_init, F32, "ball_init", n * 2), _p(reset_in, I64, "reset_in", n), _p(progress, I64, "progress", n),
        C.byref(cfg), _p(rew, F32, "rew", n), _p(reset_out, I64, "reset_out", n), n, _stream(rew)),
        "bezk_compute_reward")
    return rew, reset_out


def reset_idx(env_ids, dof_state, root_states, initial_root_states, progress, reset, cfg, uniforms=None,
              seed=0, step=0):
    k = int(env_ids.numel())
    n = progress.shape[0]
    lib = _lib.load()
    _lib.check(lib.bezk_reset_idx(
        _p(env_ids, I64, "env_ids"), k, _p(uniforms, F32, "uniforms", k * 36, True), seed, step,
        _p(dof_state, F32, "dof_state", n * 36), _p(root_states, F32, "root_states", n * 26, True),
        _p(initial_root_states, F32, "initial_root_states", n * 26, True), _p(progress, I64, "progress", n),
        _p(reset, I64, "reset", n), C.byref(cfg), n, _stream(progress)), "bezk_reset_idx")


def post_physics(dof_state, rigid_body, root_states, net_contact, goal, ball_init, initial_root_states,
                 reset_buf, progress_buf, timeout_buf, cfg, obs, rew, prev_lin_vel=None, uniforms=None,
                 seed=0, step=0, randomize_buf=None, obs_clipped=None, parts=_lib.PART_ALL):
    n = progress_buf.shape[0]
    nb = cfg.num_bodies
    lib = _lib.load()
    _lib.check(lib.bezk_post_physics(
        _p(dof_state, F32, "dof_state", n * 36), _p(rigid_body, F32, "rigid_body", n * nb * 13),
        _p(root_states, F32, "root_states", n * 26), _p(net_contact, F32, "net_contact", n * nb * 3, True),
        _p(prev_lin_vel, F32, "prev_lin_vel", n * 3, True), _p(goal, F32, "goal", n * 2),
        _p(ball_init, F32, "ball_init", n * 2), _p(initial_root_states, F32, "initial_root_states", n * 26, True),
        _p(uniforms, F32, "uniforms", n * 36, True), seed, step, _p(reset_buf, I64, "reset_buf", n),
        _p(progress_buf, I64, "progress_buf", n), _p(timeout_buf, I64, "timeout_buf", n, True),
        _p(randomize_buf, I64, "randomize_buf", n, True), C.byref(cfg), _p(obs, F32, "obs", n * 54, True),
        _p(obs_clipped, F32, "obs_clipped", n * 54, True), _p(rew, F32, "rew", n, True), int(parts), n,
        _stream(progress_buf)), "bezk_post_physics")


_TASK_ID = {"kick": _lib.TASK_KICK, "walk": _lib.TASK_WALK, "orient": _lib.TASK_ORIENT}


def post_physics_task(task, dof_state, rigid_body, root_states, net_contact, goal, initial_root_states, reset_buf,
                      progress_buf, timeout_buf, cfg, obs, rew, goal_angle=None, ball_init=None, prev_lin_vel=None,
                      uniforms=None, goal_uniforms=None, seed=0, step=0, randomize_buf=None, obs_clipped=None,
                      parts=_lib.PART_ALL):
    """``post_physics`` for any of the three tasks (``"kick"``, ``"walk"``, ``"orient"``): see ``bezk_post_physics_task``."""
    n = progress_buf.shape[0] if progress_buf is not None else (obs.shape[0] if obs is not None else rew.shape[0])
    nb = cfg.num_bodies
    actors, _, width = bm.task_dims(task)
    lib = _lib.load()
    _lib.check(lib.bezk_post_physics_task(
        _TASK_ID[task], _p(dof_state, F32, "dof_state", n * 36), _p(rigid_body, F32, "rigid_body", n * nb * 13),
        _p(root_states, F32, "root_states", n * actors * 13), _p(net_contact, F32, "net_contact", n * nb * 3, True),
        _p(prev_lin_vel, F32, "prev_lin_vel", n * 3, True), _p(goal, F32, "goal", n * 2),
        _p(goal_angle, F32, "goal_angle", n, True), _p(ball_init, F32, "ball_init", n * 2, True),
        _p(initial_root_states, F32, "initial_root_states", n * actors * 13, True),
        _p(uniforms, F32, "uniforms", n * 36, True), _p(goal_uniforms, F32, "goal_uniforms", 2, True), seed, step,
        _p(reset_buf, I64, "reset_buf", n, True), _p(progress_buf, I64, "progress_buf", n, True),
        _p(timeout_buf, I64, "timeout_buf", n, True), _p(randomize_buf, I64, "randomize_buf", n, True), C.byref(cfg),
        _p(obs, F32, "obs", n * width, True), _p(obs_clipped, F32, "obs_clipped", n * width, True), _p(rew, F32, "rew", n, True),
        int(parts), n, _stream(dof_state)), "bezk_post_physics_task")


def make_rollout_cfg(gamma=0.99, scale_value=0.01, shift_value=0.0, value_bootstrap=True) -> BezkRolloutCfg:
    """rl_games' per-step reward path (``play_steps``; cfg/train/bez_kickPPO.yaml:53-56) as kernel constants."""
    c = BezkRolloutCfg()
    c.scale_value, c.shift_value, c.gamma = float(scale_value), float(shift_value), float(gamma)
    c.value_bootstrap = int(bool(value_bootstrap))
    return c


def post_physics_rollout(task, dof_state, rigid_body, root_states, net_contact, goal, initial_root_states, reset_buf,
                         progress_buf, timeout_buf, cfg, obs, rew, rollout_cfg=None, values=None, shaped_rewards=None,
                         dones_u8=None, goal_angle=None, ball_init=None, prev_lin_vel=None, uniforms=None, goal_uniforms=None,
                         seed=0, step=0, randomize_buf=None, obs_clipped=None, env_base=0):
    """The fused step + rl_games' reward shaping / value bootstrap / uint8 dones in its epilogue (``bezk_post_physics_rollout``)."""
    n = progress_buf.shape[0]
    nb = cfg.num_bodies
    actors, _, width = bm.task_dims(task)
    lib = _lib.load()
    _lib.check(lib.bezk_post_physics_rollout(
        _TASK_ID[task], _p(dof_state, F32, "dof_state", n * 36), _p(rigid_body, F32, "rigid_body", n * nb * 13),
        _p(root_states, F32, "root_states", n * actors * 13), _p(net_contact, F32, "net_contact", n * nb * 3),
        _p(prev_lin_vel, F32, "prev_lin_vel", n * 3, True), _p(goal, F32, "goal", n * 2),
        _p(goal_angle, F32, "goal_angle", n, True), _p(ball_init, F32, "ball_init", n * 2, True),
        _p(initial_root_states, F32, "initial_root_states", n * actors * 13, True),
        _p(uniforms, F32, "uniforms", n * 36, True), _p(goal_uniforms, F32, "goal_uniforms", 2, True), seed, step,
        _p(reset_buf, I64, "reset_buf", n), _p(progress_buf, I64, "progress_buf", n),
        _p(timeout_buf, I64, "timeout_buf", n), _p(randomize_buf, I64, "randomize_buf", n, True), C.byref(cfg),
        _p(obs, F32, "obs", n * width), _p(obs_clipped, F32, "obs_clipped", n * width, True), _p(rew, F32, "rew", n),
        C.byref(rollout_cfg) if rollout_cfg is not None else None, _p(values, F32, "values", n, True),
        _p(shaped_rewards, F32, "shaped_rewards", n, True), _p(dones_u8, U8, "dones_u8", n, True), int(env_base), n,
        _stream(dof_state)), "bezk_post_physics_rollout")


def _cuda(t, dtype, name, numel):
    if not isinstance(t, torch.Tensor) or not t.is_cuda:
        raise BezkError(f"{name} must be a CUDA tensor")
    return _p(t, dtype, name, numel)


def post_physics_rollout_ep(task, dof_state, rigid_body, root_states, net_contact, goal, initial_root_states, reset_buf,
                            progress_buf, timeout_buf, cfg, obs, rew, episode_returns, episode_lengths, episode_partials,
                            rollout_cfg=None, values=None, shaped_rewards=None, dones_u8=None, goal_angle=None, ball_init=None,
                            prev_lin_vel=None, uniforms=None, goal_uniforms=None, seed=0, step=0, randomize_buf=None,
                            obs_clipped=None, env_base=0):
    """``post_physics_rollout`` that also carries rl_games' per-env episode return / length (``episode_returns`` /
    ``episode_lengths``, (N,) float32, CUDA) and writes this step's done-env partials (``episode_partials``, (3, ceil(N/32))
    float64, CUDA; ``bezk_post_physics_rollout_ep``)."""
    n = progress_buf.shape[0]
    nb = cfg.num_bodies
    actors, _, width = bm.task_dims(task)
    ret = _cuda(episode_returns, F32, "episode_returns", n)
    length = _cuda(episode_lengths, F32, "episode_lengths", n)
    part = _cuda(episode_partials, F64, "episode_partials", 3 * ((n + 31) // 32))
    lib = _lib.load()
    _lib.check(lib.bezk_post_physics_rollout_ep(
        _TASK_ID[task], _p(dof_state, F32, "dof_state", n * 36), _p(rigid_body, F32, "rigid_body", n * nb * 13),
        _p(root_states, F32, "root_states", n * actors * 13), _p(net_contact, F32, "net_contact", n * nb * 3),
        _p(prev_lin_vel, F32, "prev_lin_vel", n * 3, True), _p(goal, F32, "goal", n * 2),
        _p(goal_angle, F32, "goal_angle", n, True), _p(ball_init, F32, "ball_init", n * 2, True),
        _p(initial_root_states, F32, "initial_root_states", n * actors * 13, True),
        _p(uniforms, F32, "uniforms", n * 36, True), _p(goal_uniforms, F32, "goal_uniforms", 2, True), seed, step,
        _p(reset_buf, I64, "reset_buf", n), _p(progress_buf, I64, "progress_buf", n),
        _p(timeout_buf, I64, "timeout_buf", n), _p(randomize_buf, I64, "randomize_buf", n, True), C.byref(cfg),
        _p(obs, F32, "obs", n * width), _p(obs_clipped, F32, "obs_clipped", n * width, True), _p(rew, F32, "rew", n),
        C.byref(rollout_cfg) if rollout_cfg is not None else None, _p(values, F32, "values", n, True),
        _p(shaped_rewards, F32, "shaped_rewards", n, True), _p(dones_u8, U8, "dones_u8", n, True), int(env_base), n,
        ret, length, part, _stream(dof_state)), "bezk_post_physics_rollout_ep")


def episode_meter_update(partials, n, games_to_track, mean2, size2, steps=None):
    """Fold ``steps`` consecutive (3, ceil(n/32)) float64 partials of ``post_physics_rollout_ep`` (``partials``: (steps, 3, W) or
    (3, W)) into the two AverageMeters ``mean2`` ((2,) float32: returns, lengths) / ``size2`` ((2,) int64), on the device
    (``bezk_episode_meter_update``)."""
    w = (int(n) + 31) // 32
    if steps is None:
        steps = partials.numel() // (3 * w) if w else 0
    if not isinstance(partials, torch.Tensor) or partials.numel() != int(steps) * 3 * w:
        raise BezkError(f"partials must hold steps x 3 x {w} float64 values")
    lib = _lib.load()
    _lib.check(lib.bezk_episode_meter_update(_cuda(partials, F64, "partials", None), int(steps), int(n), int(games_to_track),
                                             _cuda(mean2, F32, "mean2", 2), _cuda(size2, I64, "size2", 2), _stream(partials)),
               "bezk_episode_meter_update")


def post_physics_rollout_ep_norm(task, dof_state, rigid_body, root_states, net_contact, goal, initial_root_states, reset_buf,
                                 progress_buf, timeout_buf, cfg, obs, rew, episode_returns, episode_lengths, episode_partials,
                                 obs_mean, obs_var, obs_norm, obs_eps=1e-5, rollout_cfg=None, values=None, shaped_rewards=None,
                                 dones_u8=None, goal_angle=None, ball_init=None, prev_lin_vel=None, uniforms=None, goal_uniforms=None,
                                 seed=0, step=0, randomize_buf=None, obs_clipped=None, env_base=0):
    """``post_physics_rollout_ep`` that also writes ``obs_norm`` ((N, obs width) float32, CUDA): the row the step returns through
    ``RunningMeanStd.forward`` in eval mode with ``obs_mean`` / ``obs_var`` ((obs width,) float64, CUDA) and ``obs_eps``
    (``bezk_post_physics_rollout_ep_norm``)."""
    n = progress_buf.shape[0]
    nb = cfg.num_bodies
    actors, _, width = bm.task_dims(task)
    ret = _cuda(episode_returns, F32, "episode_returns", n)
    length = _cuda(episode_lengths, F32, "episode_lengths", n)
    part = _cuda(episode_partials, F64, "episode_partials", 3 * ((n + 31) // 32))
    mean, var = _cuda(obs_mean, F64, "obs_mean", width), _cuda(obs_var, F64, "obs_var", width)
    norm = _cuda(obs_norm, F32, "obs_norm", n * width)
    lib = _lib.load()
    _lib.check(lib.bezk_post_physics_rollout_ep_norm(
        _TASK_ID[task], _p(dof_state, F32, "dof_state", n * 36), _p(rigid_body, F32, "rigid_body", n * nb * 13),
        _p(root_states, F32, "root_states", n * actors * 13), _p(net_contact, F32, "net_contact", n * nb * 3),
        _p(prev_lin_vel, F32, "prev_lin_vel", n * 3, True), _p(goal, F32, "goal", n * 2),
        _p(goal_angle, F32, "goal_angle", n, True), _p(ball_init, F32, "ball_init", n * 2, True),
        _p(initial_root_states, F32, "initial_root_states", n * actors * 13, True),
        _p(uniforms, F32, "uniforms", n * 36, True), _p(goal_uniforms, F32, "goal_uniforms", 2, True), seed, step,
        _p(reset_buf, I64, "reset_buf", n), _p(progress_buf, I64, "progress_buf", n),
        _p(timeout_buf, I64, "timeout_buf", n), _p(randomize_buf, I64, "randomize_buf", n, True), C.byref(cfg),
        _p(obs, F32, "obs", n * width), _p(obs_clipped, F32, "obs_clipped", n * width, True), _p(rew, F32, "rew", n),
        C.byref(rollout_cfg) if rollout_cfg is not None else None, _p(values, F32, "values", n, True),
        _p(shaped_rewards, F32, "shaped_rewards", n, True), _p(dones_u8, U8, "dones_u8", n, True), int(env_base), n,
        ret, length, part, mean, var, float(obs_eps), norm, _stream(dof_state)), "bezk_post_physics_rollout_ep_norm")


def player_tally_update(partials, n, games_num, tally, per_step=None, steps=None):
    """Fold ``steps`` consecutive (3, ceil(n/32)) float64 partials of ``post_physics_rollout_ep`` (``partials``: (steps, 3, W) or
    (3, W)) into rl_games ``BasePlayer.run``'s game tally ``tally`` ((4,) float64: games_played, sum_rewards, sum_steps,
    steps_folded) up to ``games_num`` games; ``per_step`` ((steps, 3) float64, optional) gets each folded step's sums, on the device
    (``bezk_player_tally_update``)."""
    w = (int(n) + 31) // 32
    if steps is None:
        steps = partials.numel() // (3 * w) if w else 0
    if not isinstance(partials, torch.Tensor) or partials.numel() != int(steps) * 3 * w:
        raise BezkError(f"partials must hold steps x 3 x {w} float64 values")
    ps = None if per_step is None else _cuda(per_step, F64, "per_step", int(steps) * 3)
    lib = _lib.load()
    _lib.check(lib.bezk_player_tally_update(_cuda(partials, F64, "partials", None), int(steps), int(n), int(games_num),
                                            _cuda(tally, F64, "tally", 4), ps, _stream(partials)), "bezk_player_tally_update")


I32 = torch.int32


def outcome_classes(task):
    """K, the number of episode outcome classes of ``task`` (5 for ``"kick"``, 4 for ``"walk"`` / ``"orient"``;
    ``bezk_outcome_classes``)."""
    k = _lib.load().bezk_outcome_classes(_TASK_ID[task])
    if k == 10001:                                   # BEZK_E_BADARG
        _lib.check(k, "bezk_outcome_classes")
    return k


def post_physics_rollout_ep_outcome(task, dof_state, rigid_body, root_states, net_contact, goal, initial_root_states, reset_buf,
                                    progress_buf, timeout_buf, cfg, obs, rew, episode_returns, episode_lengths, episode_partials,
                                    outcome_partials, obs_mean=None, obs_var=None, obs_norm=None, obs_eps=1e-5, rollout_cfg=None,
                                    values=None, shaped_rewards=None, dones_u8=None, goal_angle=None, ball_init=None, prev_lin_vel=None,
                                    uniforms=None, goal_uniforms=None, seed=0, step=0, randomize_buf=None, obs_clipped=None, env_base=0):
    """``post_physics_rollout_ep`` (or ``_ep_norm`` when ``obs_mean`` / ``obs_var`` / ``obs_norm`` are given) that also writes the
    per-warp count of done envs per outcome class (``outcome_partials``, (K, ceil(N/32)) int32, CUDA;
    ``bezk_post_physics_rollout_ep_outcome``)."""
    n = progress_buf.shape[0]
    nb = cfg.num_bodies
    actors, _, width = bm.task_dims(task)
    ret = _cuda(episode_returns, F32, "episode_returns", n)
    length = _cuda(episode_lengths, F32, "episode_lengths", n)
    part = _cuda(episode_partials, F64, "episode_partials", 3 * ((n + 31) // 32))
    oc = _cuda(outcome_partials, I32, "outcome_partials", outcome_classes(task) * ((n + 31) // 32))
    norm = (obs_mean, obs_var, obs_norm)
    if any(t is not None for t in norm):
        mean, var = _cuda(obs_mean, F64, "obs_mean", width), _cuda(obs_var, F64, "obs_var", width)
        out = _cuda(obs_norm, F32, "obs_norm", n * width)
    else:
        mean = var = out = None
    lib = _lib.load()
    _lib.check(lib.bezk_post_physics_rollout_ep_outcome(
        _TASK_ID[task], _p(dof_state, F32, "dof_state", n * 36), _p(rigid_body, F32, "rigid_body", n * nb * 13),
        _p(root_states, F32, "root_states", n * actors * 13), _p(net_contact, F32, "net_contact", n * nb * 3),
        _p(prev_lin_vel, F32, "prev_lin_vel", n * 3, True), _p(goal, F32, "goal", n * 2),
        _p(goal_angle, F32, "goal_angle", n, True), _p(ball_init, F32, "ball_init", n * 2, True),
        _p(initial_root_states, F32, "initial_root_states", n * actors * 13, True),
        _p(uniforms, F32, "uniforms", n * 36, True), _p(goal_uniforms, F32, "goal_uniforms", 2, True), seed, step,
        _p(reset_buf, I64, "reset_buf", n), _p(progress_buf, I64, "progress_buf", n),
        _p(timeout_buf, I64, "timeout_buf", n), _p(randomize_buf, I64, "randomize_buf", n, True), C.byref(cfg),
        _p(obs, F32, "obs", n * width), _p(obs_clipped, F32, "obs_clipped", n * width, True), _p(rew, F32, "rew", n),
        C.byref(rollout_cfg) if rollout_cfg is not None else None, _p(values, F32, "values", n, True),
        _p(shaped_rewards, F32, "shaped_rewards", n, True), _p(dones_u8, U8, "dones_u8", n, True), int(env_base), n,
        ret, length, part, mean, var, float(obs_eps), out, oc, _stream(dof_state)), "bezk_post_physics_rollout_ep_outcome")


def _outcome_steps(partials, n, k, steps):
    w = (int(n) + 31) // 32
    if steps is None:
        steps = partials.numel() // (k * w) if w else 0
    if not isinstance(partials, torch.Tensor) or partials.numel() != int(steps) * k * w:
        raise BezkError(f"partials must hold steps x {k} x {w} int32 values")
    return int(steps)


def outcome_meter_update(partials, n, task, games_to_track, mean_k, size, steps=None):
    """Fold ``steps`` consecutive (K, ceil(n/32)) int32 outcome partials (``partials``: (steps, K, W) or (K, W)) into rl_games'
    ``AverageMeter(K, games_to_track)`` ``mean_k`` ((K,) float32) / ``size`` ((1,) int64), on the device
    (``bezk_outcome_meter_update``)."""
    k = outcome_classes(task)
    steps = _outcome_steps(partials, n, k, steps)
    lib = _lib.load()
    _lib.check(lib.bezk_outcome_meter_update(_cuda(partials, I32, "partials", None), steps, int(n), _TASK_ID[task], int(games_to_track),
                                             _cuda(mean_k, F32, "mean_k", k), _cuda(size, I64, "size", 1), _stream(partials)),
               "bezk_outcome_meter_update")


def player_outcome_update(partials, n, task, games_num, counts, per_step=None, steps=None):
    """Fold ``steps`` consecutive (K, ceil(n/32)) int32 outcome partials into ``counts`` ((1 + K,) float64: games_counted, then the
    games per class) up to ``games_num`` games, with ``player_tally_update``'s cutoff; ``per_step`` ((steps, K) float64, optional)
    gets each folded step's counts (``bezk_player_outcome_update``)."""
    k = outcome_classes(task)
    steps = _outcome_steps(partials, n, k, steps)
    ps = None if per_step is None else _cuda(per_step, F64, "per_step", steps * k)
    lib = _lib.load()
    _lib.check(lib.bezk_player_outcome_update(_cuda(partials, I32, "partials", None), steps, int(n), _TASK_ID[task], int(games_num),
                                              _cuda(counts, F64, "counts", 1 + k), ps, _stream(partials)), "bezk_player_outcome_update")


def reward_terms(task):
    """K, the number of reward terms of ``task`` (6 for ``"kick"``, 5 for ``"walk"`` / ``"orient"``; ``bezk_reward_terms``)."""
    k = _lib.load().bezk_reward_terms(_TASK_ID[task])
    if k == 10001:                                   # BEZK_E_BADARG
        _lib.check(k, "bezk_reward_terms")
    return k


def post_physics_rollout_ep_terms(task, dof_state, rigid_body, root_states, net_contact, goal, initial_root_states, reset_buf,
                                  progress_buf, timeout_buf, cfg, obs, rew, episode_returns, episode_lengths, episode_partials,
                                  term_partials, outcome_partials=None, rollout_cfg=None, values=None, shaped_rewards=None,
                                  dones_u8=None, goal_angle=None, ball_init=None, prev_lin_vel=None, uniforms=None, goal_uniforms=None,
                                  seed=0, step=0, randomize_buf=None, obs_clipped=None, env_base=0):
    """``post_physics_rollout_ep`` (or ``_ep_outcome`` when ``outcome_partials`` is given) that also writes the per-warp sum of
    each reward term (``term_partials``, (K, ceil(N/32)) float64, CUDA; ``bezk_post_physics_rollout_ep_terms``)."""
    n = progress_buf.shape[0]
    nb = cfg.num_bodies
    actors, _, width = bm.task_dims(task)
    w = (n + 31) // 32
    ret = _cuda(episode_returns, F32, "episode_returns", n)
    length = _cuda(episode_lengths, F32, "episode_lengths", n)
    part = _cuda(episode_partials, F64, "episode_partials", 3 * w)
    tm = _cuda(term_partials, F64, "term_partials", reward_terms(task) * w)
    oc = None if outcome_partials is None else _cuda(outcome_partials, I32, "outcome_partials", outcome_classes(task) * w)
    lib = _lib.load()
    _lib.check(lib.bezk_post_physics_rollout_ep_terms(
        _TASK_ID[task], _p(dof_state, F32, "dof_state", n * 36), _p(rigid_body, F32, "rigid_body", n * nb * 13),
        _p(root_states, F32, "root_states", n * actors * 13), _p(net_contact, F32, "net_contact", n * nb * 3),
        _p(prev_lin_vel, F32, "prev_lin_vel", n * 3, True), _p(goal, F32, "goal", n * 2),
        _p(goal_angle, F32, "goal_angle", n, True), _p(ball_init, F32, "ball_init", n * 2, True),
        _p(initial_root_states, F32, "initial_root_states", n * actors * 13, True),
        _p(uniforms, F32, "uniforms", n * 36, True), _p(goal_uniforms, F32, "goal_uniforms", 2, True), seed, step,
        _p(reset_buf, I64, "reset_buf", n), _p(progress_buf, I64, "progress_buf", n),
        _p(timeout_buf, I64, "timeout_buf", n), _p(randomize_buf, I64, "randomize_buf", n, True), C.byref(cfg),
        _p(obs, F32, "obs", n * width), _p(obs_clipped, F32, "obs_clipped", n * width, True), _p(rew, F32, "rew", n),
        C.byref(rollout_cfg) if rollout_cfg is not None else None, _p(values, F32, "values", n, True),
        _p(shaped_rewards, F32, "shaped_rewards", n, True), _p(dones_u8, U8, "dones_u8", n, True), int(env_base), n,
        ret, length, part, None, None, 0.0, None, oc, tm, _stream(dof_state)), "bezk_post_physics_rollout_ep_terms")


def reward_terms_update(partials, n, task, mean_k, steps=None):
    """Fold ``steps`` consecutive (K, ceil(n/32)) float64 reward term partials (``partials``: (steps, K, W) or (K, W)) into
    ``mean_k`` ((K,) float64): each term's mean per env-step over the steps x n env-steps, on the device
    (``bezk_reward_terms_update``)."""
    k = reward_terms(task)
    w = (int(n) + 31) // 32
    if steps is None:
        steps = partials.numel() // (k * w) if w else 0
    if not isinstance(partials, torch.Tensor) or partials.numel() != int(steps) * k * w:
        raise BezkError(f"partials must hold steps x {k} x {w} float64 values")
    lib = _lib.load()
    _lib.check(lib.bezk_reward_terms_update(_cuda(partials, F64, "partials", None), int(steps), int(n), _TASK_ID[task],
                                            _cuda(mean_k, F64, "mean_k", k), _stream(partials)), "bezk_reward_terms_update")


def post_physics_rollout_ep_game_terms(task, dof_state, rigid_body, root_states, net_contact, goal, initial_root_states, reset_buf,
                                       progress_buf, timeout_buf, cfg, obs, rew, episode_returns, episode_lengths, episode_partials,
                                       game_term_returns, game_term_partials, outcome_partials=None, term_partials=None, obs_mean=None,
                                       obs_var=None, obs_norm=None, obs_eps=1e-5, rollout_cfg=None, values=None, shaped_rewards=None,
                                       dones_u8=None, goal_angle=None, ball_init=None, prev_lin_vel=None, uniforms=None,
                                       goal_uniforms=None, seed=0, step=0, randomize_buf=None, obs_clipped=None, env_base=0):
    """``post_physics_rollout_ep`` (with the optional normaliser, outcome counts and reward terms of ``_ep_norm`` / ``_ep_outcome``
    / ``_ep_terms``) that also carries each env's per-term episode returns (``game_term_returns``, (K, N) float32, CUDA) and writes
    the per-warp sums of the done envs' per-term returns (``game_term_partials``, (K, ceil(N/32)) float64, CUDA;
    ``bezk_post_physics_rollout_ep_game_terms``)."""
    n = progress_buf.shape[0]
    nb = cfg.num_bodies
    actors, _, width = bm.task_dims(task)
    w = (n + 31) // 32
    k = reward_terms(task)
    ret = _cuda(episode_returns, F32, "episode_returns", n)
    length = _cuda(episode_lengths, F32, "episode_lengths", n)
    part = _cuda(episode_partials, F64, "episode_partials", 3 * w)
    gacc = _cuda(game_term_returns, F32, "game_term_returns", k * n)
    gpart = _cuda(game_term_partials, F64, "game_term_partials", k * w)
    oc = None if outcome_partials is None else _cuda(outcome_partials, I32, "outcome_partials", outcome_classes(task) * w)
    tm = None if term_partials is None else _cuda(term_partials, F64, "term_partials", k * w)
    if any(t is not None for t in (obs_mean, obs_var, obs_norm)):
        mean, var = _cuda(obs_mean, F64, "obs_mean", width), _cuda(obs_var, F64, "obs_var", width)
        out = _cuda(obs_norm, F32, "obs_norm", n * width)
    else:
        mean = var = out = None
    lib = _lib.load()
    _lib.check(lib.bezk_post_physics_rollout_ep_game_terms(
        _TASK_ID[task], _p(dof_state, F32, "dof_state", n * 36), _p(rigid_body, F32, "rigid_body", n * nb * 13),
        _p(root_states, F32, "root_states", n * actors * 13), _p(net_contact, F32, "net_contact", n * nb * 3),
        _p(prev_lin_vel, F32, "prev_lin_vel", n * 3, True), _p(goal, F32, "goal", n * 2),
        _p(goal_angle, F32, "goal_angle", n, True), _p(ball_init, F32, "ball_init", n * 2, True),
        _p(initial_root_states, F32, "initial_root_states", n * actors * 13, True),
        _p(uniforms, F32, "uniforms", n * 36, True), _p(goal_uniforms, F32, "goal_uniforms", 2, True), seed, step,
        _p(reset_buf, I64, "reset_buf", n), _p(progress_buf, I64, "progress_buf", n),
        _p(timeout_buf, I64, "timeout_buf", n), _p(randomize_buf, I64, "randomize_buf", n, True), C.byref(cfg),
        _p(obs, F32, "obs", n * width), _p(obs_clipped, F32, "obs_clipped", n * width, True), _p(rew, F32, "rew", n),
        C.byref(rollout_cfg) if rollout_cfg is not None else None, _p(values, F32, "values", n, True),
        _p(shaped_rewards, F32, "shaped_rewards", n, True), _p(dones_u8, U8, "dones_u8", n, True), int(env_base), n,
        ret, length, part, mean, var, float(obs_eps), out, oc, tm, gacc, gpart, _stream(dof_state)),
        "bezk_post_physics_rollout_ep_game_terms")


def _game_term_steps(ep_partials, term_partials, n, k, steps):
    w = (int(n) + 31) // 32
    if steps is None:
        steps = term_partials.numel() // (k * w) if isinstance(term_partials, torch.Tensor) and w else 0
    if not isinstance(term_partials, torch.Tensor) or term_partials.numel() != int(steps) * k * w:
        raise BezkError(f"term_partials must hold steps x {k} x {w} float64 values")
    if not isinstance(ep_partials, torch.Tensor) or ep_partials.numel() != int(steps) * 3 * w:
        raise BezkError(f"ep_partials must hold steps x 3 x {w} float64 values")
    return int(steps)


def game_terms_meter_update(ep_partials, term_partials, n, task, games_to_track, mean_k, size, steps=None):
    """Fold ``steps`` consecutive (3, ceil(n/32)) episode partials and (K, ceil(n/32)) float64 game term partials (each (steps, ., W)
    or (., W)) into rl_games' ``AverageMeter(K, games_to_track)`` ``mean_k`` ((K,) float32) / ``size`` ((1,) int64), fed one K-row
    of per-term returns per finished game, on the device (``bezk_game_terms_meter_update``)."""
    k = reward_terms(task)
    steps = _game_term_steps(ep_partials, term_partials, n, k, steps)
    lib = _lib.load()
    _lib.check(lib.bezk_game_terms_meter_update(_cuda(ep_partials, F64, "ep_partials", None), _cuda(term_partials, F64, "term_partials", None),
                                                steps, int(n), _TASK_ID[task], int(games_to_track), _cuda(mean_k, F32, "mean_k", k),
                                                _cuda(size, I64, "size", 1), _stream(term_partials)), "bezk_game_terms_meter_update")


def player_game_terms_update(ep_partials, term_partials, n, task, games_num, sums, per_step=None, steps=None):
    """Fold the same partials into ``sums`` ((1 + K,) float64: games_counted, then each term's sum of per-game returns) up to
    ``games_num`` games, with ``player_tally_update``'s cutoff; ``per_step`` ((steps, K) float64, optional) gets each folded step's
    sums (``bezk_player_game_terms_update``)."""
    k = reward_terms(task)
    steps = _game_term_steps(ep_partials, term_partials, n, k, steps)
    ps = None if per_step is None else _cuda(per_step, F64, "per_step", steps * k)
    lib = _lib.load()
    _lib.check(lib.bezk_player_game_terms_update(_cuda(ep_partials, F64, "ep_partials", None), _cuda(term_partials, F64, "term_partials", None),
                                                 steps, int(n), _TASK_ID[task], int(games_num), _cuda(sums, F64, "sums", 1 + k), ps,
                                                 _stream(term_partials)), "bezk_player_game_terms_update")


def reset_idx_task(task, env_ids, dof_state, root_states, initial_root_states, goal, progress, reset, cfg, uniforms=None,
                   goal_uniforms=None, seed=0, step=0, env_base=0):
    k = int(env_ids.numel())
    n = progress.shape[0]
    actors = bm.task_dims(task)[0]
    lib = _lib.load()
    _lib.check(lib.bezk_reset_idx_task(
        _TASK_ID[task], _p(env_ids, I64, "env_ids"), k, _p(uniforms, F32, "uniforms", k * 36, True),
        _p(goal_uniforms, F32, "goal_uniforms", 2, True), seed, step, _p(dof_state, F32, "dof_state", n * 36),
        _p(root_states, F32, "root_states", n * actors * 13, True),
        _p(initial_root_states, F32, "initial_root_states", n * actors * 13, True), _p(goal, F32, "goal", n * 2, True),
        _p(progress, I64, "progress", n), _p(reset, I64, "reset", n), C.byref(cfg), int(env_base), n, _stream(progress)),
        "bezk_reset_idx_task")


def goal_uniforms(seed, step, out=None, device="cuda"):
    out = torch.empty(2, dtype=F32, device=device) if out is None else out
    _lib.check(_lib.load().bezk_goal_uniforms(seed, step, _p(out, F32, "out", 2), _stream(out)), "bezk_goal_uniforms")
    return out


def philox_uniforms(seed, step, out):
    n = out.shape[0]
    lib = _lib.load()
    _lib.check(lib.bezk_philox_uniforms(seed, step, _p(out, F32, "out", n * 36), n, _stream(out)), "bezk_philox_uniforms")
    return out


# ------------------------------------------------------------------------------------------- learner
def gae(rewards, values, dones, last_values, last_dones, gamma, tau, advs, returns):
    horizon = rewards.shape[0]
    n = rewards.numel() // max(horizon, 1)
    if dones.dtype == U8:
        kind, dt = 0, U8
    elif dones.dtype == F32:
        kind, dt = 1, F32
    else:
        raise BezkError(f"dones must be uint8 or float32, got {dones.dtype}")
    lib = _lib.load()
    _lib.check(lib.bezk_gae(_p(rewards, F32, "rewards", horizon * n), _p(values, F32, "values", horizon * n),
                            _p(dones, dt, "dones", horizon * n), _p(last_values, F32, "last_values", n),
                            _p(last_dones, dt, "last_dones", n), kind, float(gamma), float(tau),
                            _p(advs, F32, "advs", horizon * n), _p(returns, F32, "returns", horizon * n), horizon, n,
                            _stream(rewards)), "bezk_gae")
    return advs, returns


def rms_scratch_doubles(c):
    return int(_lib.load().bezk_rms_scratch_doubles(int(c)))


def rms_moments(x, pivot, acc, partials):
    c = x.shape[-1] if x.dim() > 1 else 1
    m = x.numel() // c
    lib = _lib.load()
    _lib.check(lib.bezk_rms_moments(_p(x, F32, "x"), _p(pivot, F64, "pivot", c, True), _p(acc, F64, "acc", 1 + 2 * c),
                                    _p(partials, F64, "partials"), m, c, _stream(x)), "bezk_rms_moments")
    if partials.numel() < rms_scratch_doubles(c):
        raise BezkError("partials scratch too small")
    return acc


def rms_merge(acc, pivot, running_mean, running_var, count):
    c = running_mean.numel()
    lib = _lib.load()
    _lib.check(lib.bezk_rms_merge(_p(acc, F64, "acc", 1 + 2 * c), _p(pivot, F64, "pivot", c, True),
                                  _p(running_mean, F64, "running_mean", c), _p(running_var, F64, "running_var", c),
                                  _p(count, F64, "count", 1), c, _stream(acc)), "bezk_rms_merge")


def rms_merge_sequence(acc, order, pivot, running_mean, running_var, count, seq):
    """``acc`` (n_batches, 1+2c) moments of the distinct batches (one pivot), ``order`` (n_updates,) int32 device tensor: replays
    the reference's update for batch ``order[u]``, u in order; ``seq`` (n_updates, 2, c) gets [mean, var] after each update."""
    c = running_mean.numel()
    nb, nu = acc.numel() // (1 + 2 * c), order.numel()
    lib = _lib.load()
    _lib.check(lib.bezk_rms_merge_sequence(_p(acc, F64, "acc", nb * (1 + 2 * c)), nb, _p(order, torch.int32, "order"), nu,
                                           _p(pivot, F64, "pivot", c, True), _p(running_mean, F64, "running_mean", c),
                                           _p(running_var, F64, "running_var", c), _p(count, F64, "count", 1),
                                           _p(seq, F64, "seq", nu * 2 * c), c, _stream(acc)), "bezk_rms_merge_sequence")
    return seq


def rms_normalize(x, running_mean, running_var, y, eps=1e-5, unnorm=False):
    c = running_mean.numel()
    m = x.numel() // c
    lib = _lib.load()
    _lib.check(lib.bezk_rms_normalize(_p(x, F32, "x", m * c), _p(running_mean, F64, "running_mean", c),
                                      _p(running_var, F64, "running_var", c), eps, int(bool(unnorm)),
                                      _p(y, F32, "y", m * c), m, c, _stream(x)), "bezk_rms_normalize")
    return y


def rms_train_forward(x, running_mean, running_var, count, y, partials, eps=1e-5):
    """The whole train-mode ``RunningMeanStd.forward`` in ONE call (one cooperative kernel at the reference's minibatch sizes):
    merge the batch moments of ``x`` into the running statistics, then ``y`` = normalise(x) with the updated statistics.
    ``x``: contiguous (m, c) / (m,) or a slab view ``storage[:, e0:e0+E]``; ``y``: contiguous, m * c elements."""
    c = running_mean.numel()
    ptr, rows, stride, m = _slab_view(x, F32, "x", c)
    if partials.numel() < rms_scratch_doubles(c):
        raise BezkError("partials scratch too small")
    lib = _lib.load()
    _lib.check(lib.bezk_rms_train_forward(ptr, rows, stride, _p(running_mean, F64, "running_mean", c), _p(running_var, F64, "running_var", c),
                                          _p(count, F64, "count", 1), float(eps), _p(y, F32, "y", m * c), _p(partials, F64, "partials"),
                                          m, c, _stream(x)), "bezk_rms_train_forward")
    return y


def rms_moments_ext(x, running_mean, running_var, count, acc_ext, partials):
    """Distributed half 1 of the train-mode forward: ``acc_ext`` (2 + 4c,) = pivoted batch moments + snapshot of the running
    statistics; all-reduce ``acc_ext[:1 + 2c]`` (SUM) before ``rms_merge_normalize``."""
    c = running_mean.numel()
    ptr, rows, stride, m = _slab_view(x, F32, "x", c)
    if partials.numel() < rms_scratch_doubles(c):
        raise BezkError("partials scratch too small")
    lib = _lib.load()
    _lib.check(lib.bezk_rms_moments_ext(ptr, rows, stride, _p(running_mean, F64, "running_mean", c), _p(running_var, F64, "running_var", c),
                                        _p(count, F64, "count", 1), _p(acc_ext, F64, "acc_ext", 2 + 4 * c), _p(partials, F64, "partials"),
                                        m, c, _stream(x)), "bezk_rms_moments_ext")
    return acc_ext


def rms_merge_normalize(x, acc_ext, running_mean, running_var, count, y, eps=1e-5):
    """Distributed half 2: merge + normalise in one launch."""
    c = running_mean.numel()
    ptr, rows, stride, m = _slab_view(x, F32, "x", c)
    lib = _lib.load()
    _lib.check(lib.bezk_rms_merge_normalize(ptr, rows, stride, _p(acc_ext, F64, "acc_ext", 2 + 4 * c), _p(running_mean, F64, "running_mean", c),
                                            _p(running_var, F64, "running_var", c), _p(count, F64, "count", 1), float(eps),
                                            _p(y, F32, "y", m * c), m, c, _stream(x)), "bezk_rms_merge_normalize")
    return y


def adv_normalize_fused(returns, values, adv_out, partials, normalize=True):
    """``adv_out = returns - values`` normalised to zero mean / unit unbiased std, one call (single GPU)."""
    m = returns.numel()
    if partials.numel() < rms_scratch_doubles(1):
        raise BezkError("partials scratch too small")
    lib = _lib.load()
    _lib.check(lib.bezk_adv_normalize_fused(_p(returns, F32, "returns", m), _p(values, F32, "values", m), _p(adv_out, F32, "adv_out", m),
                                            _p(partials, F64, "partials"), int(bool(normalize)), m, _stream(returns)),
               "bezk_adv_normalize_fused")
    return adv_out


def adv_moments(returns, values, acc, partials):
    m = returns.numel()
    lib = _lib.load()
    _lib.check(lib.bezk_adv_moments(_p(returns, F32, "returns", m), _p(values, F32, "values", m), _p(acc, F64, "acc", 3),
                                    _p(partials, F64, "partials"), m, _stream(returns)), "bezk_adv_moments")
    return acc


def adv_normalize(returns, values, acc, adv_out, normalize=True):
    m = returns.numel()
    lib = _lib.load()
    _lib.check(lib.bezk_adv_normalize(_p(returns, F32, "returns", m), _p(values, F32, "values", m),
                                      _p(acc, F64, "acc", 3, not normalize), _p(adv_out, F32, "adv_out", m),
                                      int(bool(normalize)), m, _stream(returns)), "bezk_adv_normalize")
    return adv_out


def make_ppo_cfg(e_clip=0.2, critic_coef=2.0, entropy_coef=0.0, bounds_loss_coef=0.001, soft_bound=1.1,
                 clip_value=True, bound_form="v1.1.3") -> BezkPpoCfg:
    c = BezkPpoCfg()
    c.e_clip, c.critic_coef, c.entropy_coef = e_clip, critic_coef, entropy_coef
    c.bounds_loss_coef, c.soft_bound = bounds_loss_coef, soft_bound
    c.clip_value = int(bool(clip_value))
    c.bound_form = {"v1.1.3": 0, "outside": 1}[bound_form]
    return c


def ppo_scratch_doubles():
    return int(_lib.load().bezk_ppo_scratch_doubles())


def ppo_loss(actions, mu, logstd, old_mu, old_sigma, values, old_values, returns, old_neglogp, advantages, cfg,
             stats, partials, grad_mu=None, grad_values=None, grad_logstd=None, neglogp_out=None):
    m = mu.shape[0]
    lib = _lib.load()
    _lib.check(lib.bezk_ppo_loss(
        _p(actions, F32, "actions", m * 18), _p(mu, F32, "mu", m * 18), _p(logstd, F32, "logstd", 18),
        _p(old_mu, F32, "old_mu", m * 18), _p(old_sigma, F32, "old_sigma", m * 18), _p(values, F32, "values", m),
        _p(old_values, F32, "old_values", m), _p(returns, F32, "returns", m), _p(old_neglogp, F32, "old_neglogp", m),
        _p(advantages, F32, "advantages", m), C.byref(cfg), _p(stats, F64, "stats", 8),
        _p(grad_mu, F32, "grad_mu", m * 18, True), _p(grad_values, F32, "grad_values", m, True),
        _p(grad_logstd, F32, "grad_logstd", 18, True), _p(neglogp_out, F32, "neglogp_out", m, True),
        _p(partials, F64, "partials"), m, _stream(mu)), "bezk_ppo_loss")
    return stats


# ------------------------------------------------------------------------------------------- rollout storage
def _slab_view(t, dtype, name, width):
    """Pointer + slab geometry of a rollout-side tensor.  Accepts a contiguous (m, width) / (m,) tensor, or a VIEW
    ``storage[:, e0:e0+E]`` of time-major rollout storage: shape (T, E, width) (or (T, E) / (T, E, 1) for width 1)
    whose inner dims are contiguous and whose time stride is a whole number of rows.
    Returns (ptr, slab_rows, slab_stride, m)."""
    if not isinstance(t, torch.Tensor) or t.dtype != dtype:
        raise BezkError(f"{name} must be a {dtype} tensor")
    if not t.is_cuda:
        raise BezkError(f"{name} is on {t.device}: bez_isaacgym_b200 ops run on CUDA only (no CPU fallback)")
    if t.is_contiguous():
        if t.numel() % width:
            raise BezkError(f"{name}: {t.numel()} elements is not a multiple of the row width {width}")
        m = t.numel() // width
        return C.c_void_p(t.data_ptr()), m, m, m
    v = t
    if width == 1 and v.dim() == 3 and v.shape[-1] == 1:
        v = v.squeeze(-1)
    want_dim = 2 if width == 1 else 3
    if v.dim() != want_dim or (width > 1 and (v.shape[-1] != width or v.stride(-1) != 1)):
        raise BezkError(f"{name}: expected a contiguous tensor or a (T, E{', ' + str(width) if width > 1 else ''}) slab view")
    T, E = v.shape[0], v.shape[1]
    if v.stride(1) != width or v.stride(0) % width or v.stride(0) < E * width:
        raise BezkError(f"{name}: not a slab view of time-major storage (strides {tuple(v.stride())})")
    return C.c_void_p(v.data_ptr()), E, v.stride(0) // width, T * E


def _same_slabs(geoms, names):
    g0 = geoms[0][1:]
    for g, nme in zip(geoms[1:], names[1:]):
        if g[1:] != g0:
            raise BezkError(f"{nme} has slab geometry {g[1:]}, {names[0]} has {g0}: rollout tensors must share one (T, N, E)")
    return g0


def rms_moments_slabs(x, pivot, acc, partials):
    """``rms_moments`` over ``x = obses[:, e0:e0+E]`` (a slab view of time-major storage) without flattening it."""
    c = x.shape[-1]
    ptr, rows, stride, m = _slab_view(x, F32, "x", c)
    if partials.numel() < rms_scratch_doubles(c):
        raise BezkError("partials scratch too small")
    lib = _lib.load()
    _lib.check(lib.bezk_rms_moments_slabs(ptr, rows, stride, _p(pivot, F64, "pivot", c, True), _p(acc, F64, "acc", 1 + 2 * c),
                                          _p(partials, F64, "partials"), m, c, _stream(x)), "bezk_rms_moments_slabs")
    return acc


def rms_normalize_slabs(x, running_mean, running_var, y, eps=1e-5, unnorm=False):
    """``y`` (m, c) contiguous = normalise(rows of the slab view ``x``), batch row = t * E + (env - e0)."""
    c = running_mean.numel()
    ptr, rows, stride, m = _slab_view(x, F32, "x", c)
    lib = _lib.load()
    _lib.check(lib.bezk_rms_normalize_slabs(ptr, rows, stride, _p(running_mean, F64, "running_mean", c),
                                            _p(running_var, F64, "running_var", c), eps, int(bool(unnorm)),
                                            _p(y, F32, "y", m * c), m, c, _stream(x)), "bezk_rms_normalize_slabs")
    return y


def _spaced_slabs(batches, c):
    """(ptr, slab_rows, slab_stride, m, batch_stride_rows) of equally spaced slab views / contiguous blocks of ONE tensor."""
    nb = len(batches)
    ptr, rows, stride, m = _slab_view(batches[0], F32, "batches[0]", c)
    step_bytes = (batches[1].data_ptr() - batches[0].data_ptr()) if nb > 1 else 0
    for b in range(1, nb):
        p2, r2, s2, m2 = _slab_view(batches[b], F32, f"batches[{b}]", c)
        if (r2, s2, m2) != (rows, stride, m) or p2.value - ptr.value != b * step_bytes or step_bytes <= 0 or step_bytes % (4 * c):
            raise BezkError("batches must be equally spaced views of one tensor with the same slab geometry")
    return ptr, rows, stride, m, step_bytes // (4 * c)


def rms_moments_slabs_batched(batches, pivot, acc, partials):
    """The moments of ``len(batches)`` equally spaced minibatches in one pair of launches; ``acc`` (len(batches), 1 + 2c)."""
    c = acc.shape[-1] // 2
    nb = len(batches)
    ptr, rows, stride, m, step = _spaced_slabs(batches, c)
    if partials.numel() < rms_scratch_doubles(c):
        raise BezkError("partials scratch too small")
    lib = _lib.load()
    _lib.check(lib.bezk_rms_moments_slabs_batched(ptr, rows, stride, step, _p(pivot, F64, "pivot", c, True),
                                                  _p(acc, F64, "acc", nb * (1 + 2 * c)), _p(partials, F64, "partials"), m, c, nb,
                                                  _stream(batches[0])), "bezk_rms_moments_slabs_batched")
    return acc


def rms_normalize_slabs_batched(batches, seq, u0, y, eps=1e-5):
    """``batches``: equally spaced slab views (or contiguous (m, c) blocks) of ONE tensor -- the minibatches of a mini-epoch;
    ``seq`` (n_updates, 2, c) from ``rms_merge_sequence``; batch b is normalised with the statistics of update ``u0 + b`` into
    ``y[b]`` (``y``: (len(batches), m, c) contiguous).  One launch."""
    nb, c = len(batches), seq.shape[-1]
    ptr, rows, stride, m, step = _spaced_slabs(batches, c)
    if u0 < 0 or u0 + nb > seq.shape[0]:
        raise BezkError("u0 + len(batches) exceeds the planned updates")
    mean = seq[u0, 0]
    lib = _lib.load()
    _lib.check(lib.bezk_rms_normalize_slabs_batched(ptr, rows, stride, step, C.c_void_p(mean.data_ptr()),
                                                    C.c_void_p(mean.data_ptr() + 8 * c), 2 * c, eps, _p(y, F32, "y", nb * m * c), m, c,
                                                    nb, _stream(batches[0])), "bezk_rms_normalize_slabs_batched")
    return y


def ppo_loss_slabs(actions, mu, logstd, old_mu, old_sigma, values, old_values, returns, old_neglogp, advantages, cfg,
                   stats, partials, grad_mu=None, grad_values=None, grad_logstd=None, neglogp_out=None):
    """``ppo_loss`` with the rollout-side tensors given as slab views (``storage[:, e0:e0+E]``); ``mu`` / ``values`` and
    the gradients are contiguous batch rows in the same time-major-within-batch order."""
    m = mu.shape[0]
    wide = [_slab_view(t, F32, nme, 18) for t, nme in ((actions, "actions"), (old_mu, "old_mu"), (old_sigma, "old_sigma"))]
    flat = [_slab_view(t, F32, nme, 1) for t, nme in ((old_values, "old_values"), (returns, "returns"),
                                                      (old_neglogp, "old_neglogp"), (advantages, "advantages"))]
    rows, stride, mm = _same_slabs(wide + flat, ["actions", "old_mu", "old_sigma", "old_values", "returns", "old_neglogp",
                                                 "advantages"])
    if mm != m:
        raise BezkError(f"rollout tensors hold {mm} rows, mu has {m}")
    lib = _lib.load()
    _lib.check(lib.bezk_ppo_loss_slabs(
        wide[0][0], _p(mu, F32, "mu", m * 18), _p(logstd, F32, "logstd", 18), wide[1][0], wide[2][0],
        _p(values, F32, "values", m), flat[0][0], flat[1][0], flat[2][0], flat[3][0], rows, stride, C.byref(cfg),
        _p(stats, F64, "stats", 8), _p(grad_mu, F32, "grad_mu", m * 18, True), _p(grad_values, F32, "grad_values", m, True),
        _p(grad_logstd, F32, "grad_logstd", 18, True), _p(neglogp_out, F32, "neglogp_out", m, True),
        _p(partials, F64, "partials"), m, _stream(mu)), "bezk_ppo_loss_slabs")
    return stats


def swap_and_flatten01(src, out=None, env0=0, envs=None):
    """rl_games' ``swap_and_flatten01`` on a contiguous time-major tensor (T, N, ...) of any dtype:
    returns (envs*T, ...) with row (e - env0)*T + t = src[t, e]."""
    if not src.is_cuda or not src.is_contiguous() or src.dim() < 2:
        raise BezkError("src must be a contiguous CUDA tensor of shape (T, N, ...)")
    T, N = src.shape[0], src.shape[1]
    envs = N - env0 if envs is None else envs
    row_bytes = (src.numel() // max(T * N, 1)) * src.element_size()
    if out is None:
        out = torch.empty((envs * T,) + tuple(src.shape[2:]), dtype=src.dtype, device=src.device)
    if not out.is_contiguous() or out.dtype != src.dtype or out.numel() * out.element_size() != envs * T * row_bytes:
        raise BezkError("out must be contiguous, of src's dtype, with envs*T rows")
    lib = _lib.load()
    _lib.check(lib.bezk_swap_and_flatten01(C.c_void_p(src.data_ptr()), C.c_void_p(out.data_ptr()), T, N, env0, envs, row_bytes,
                                           _stream(src)), "bezk_swap_and_flatten01")
    return out


def policy_head(mu, logstd, value_norm=None, value_mean=None, value_var=None, value_eps=1e-5, noise=None, seed=0, step=0,
                actions=None, neglogp=None, values=None, mus=None, sigmas=None, task_cfg=None, env_actions=None, targets=None,
                env_base=0):
    """Sampling / neglogp / value un-normalisation / experience-slot writes / clamp / K0 in one launch (see bezk.h).
    ``env_base``: global id of row 0 (the rank's shard offset), the Philox key of the exploration noise."""
    n = mu.shape[0]
    lib = _lib.load()
    _lib.check(lib.bezk_policy_head(
        _p(mu, F32, "mu", n * 18), _p(logstd, F32, "logstd", 18), _p(value_norm, F32, "value_norm", n, True),
        _p(value_mean, F64, "value_mean", 1, True), _p(value_var, F64, "value_var", 1, True), float(value_eps),
        _p(noise, F32, "noise", n * 18, True), int(seed), int(step), _p(actions, F32, "actions", n * 18, True),
        _p(neglogp, F32, "neglogp", n, True), _p(values, F32, "values", n, True), _p(mus, F32, "mus", n * 18, True),
        _p(sigmas, F32, "sigmas", n * 18, True), C.byref(task_cfg) if task_cfg is not None else None,
        _p(env_actions, F32, "env_actions", n * 18, True), _p(targets, F32, "targets", n * 18, True), int(env_base), n,
        _stream(mu)), "bezk_policy_head")


def normal_noise(seed, step, out, env_base=0):
    n = out.shape[0]
    lib = _lib.load()
    _lib.check(lib.bezk_normal_noise(int(seed), int(step), _p(out, F32, "out", n * 18), int(env_base), n, _stream(out)),
               "bezk_normal_noise")
    return out


# ------------------------------------------------------------------------------------------- domain-randomisation noise
def make_noise_cfg(distribution="gaussian", operation="additive", a=0.0, b=0.0, a_corr=0.0, b_corr=0.0) -> BezkNoiseCfg:
    """``y = op(x, (corr * a_corr + b_corr) + w * a + b)``; gaussian: (a, b) = (var, mu); uniform: (a, b) = (hi - lo, lo)."""
    c = BezkNoiseCfg()
    c.distribution = {"gaussian": 0, "uniform": 1}[distribution]
    c.operation = {"additive": 0, "scaling": 1}[operation]
    c.a, c.b, c.a_corr, c.b_corr = float(a), float(b), float(a_corr), float(b_corr)
    return c


def dr_noise(x, cfg: BezkNoiseCfg, corr=None, white=None, seed=0, step=0, out=None, out_clipped=None, clip=None):
    """``out_clipped`` / ``clip``: also write ``clamp(y, -clip, clip)`` in the same pass (``bezk_dr_noise_clip``)."""
    total = x.numel()
    y = x if out is None else out
    lib = _lib.load()
    if out_clipped is not None:
        _lib.check(lib.bezk_dr_noise_clip(_p(x, F32, "x"), _p(corr, F32, "corr", total, True), _p(white, F32, "white", total, True),
                                          int(seed), int(step), C.byref(cfg), _p(y, F32, "y", total),
                                          _p(out_clipped, F32, "out_clipped", total), float(clip), total, _stream(x)), "bezk_dr_noise_clip")
        return y
    _lib.check(lib.bezk_dr_noise(_p(x, F32, "x"), _p(corr, F32, "corr", total, True), _p(white, F32, "white", total, True),
                                 int(seed), int(step), C.byref(cfg), _p(y, F32, "y", total), total, _stream(x)), "bezk_dr_noise")
    return y


def dr_fill(seed, step, out, distribution="gaussian"):
    lib = _lib.load()
    _lib.check(lib.bezk_dr_fill(int(seed), int(step), {"gaussian": 0, "uniform": 1}[distribution], _p(out, F32, "out"),
                                out.numel(), _stream(out)), "bezk_dr_fill")
    return out


# ------------------------------------------------------------------------------------------- generic jit helpers
def quat_rotate(q, v, out=None, inverse=False):
    """isaacgym.torch_utils ``quat_rotate`` / ``quat_rotate_inverse`` (xyzw): q (n,4), v (n,3) -> (n,3)."""
    n = q.shape[0]
    out = torch.empty(n, 3, dtype=F32, device=q.device) if out is None else out
    _lib.check(_lib.load().bezk_quat_rotate(_p(q, F32, "q", n * 4), _p(v, F32, "v", n * 3), _p(out, F32, "out", n * 3), int(bool(inverse)),
                                            n, _stream(q)), "bezk_quat_rotate")
    return out


def scale_transform(x, lower, upper, out=None, mode="scale"):
    """``utils/torch_jit_utils.py`` ``scale_transform`` / ``unscale_transform`` / ``saturate`` on x (n, dims)."""
    dims = lower.numel()
    n = x.numel() // max(dims, 1)
    out = torch.empty_like(x) if out is None else out
    _lib.check(_lib.load().bezk_scale_transform(_p(x, F32, "x", n * dims), _p(lower, F32, "lower", dims), _p(upper, F32, "upper", dims),
                                                _p(out, F32, "out", n * dims), {"scale": 0, "unscale": 1, "saturate": 2}[mode], n, dims,
                                                _stream(x)), "bezk_scale_transform")
    return out
