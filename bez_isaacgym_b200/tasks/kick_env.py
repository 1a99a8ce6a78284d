"""``KickEnv`` -- drop-in for the reference's BezKick task (``bez_isaacgym/tasks/kick_env.py:44-850``) on B200.

Same constructor (``cfg, sim_device, graphics_device_id, headless``), public attributes and
``step`` / ``reset`` / ``reset_idx`` / ``pre_physics_step`` / ``post_physics_step`` / ``compute_observations`` /
``compute_reward`` methods; underneath, ``step`` is TWO launches of hand-written sm_100a kernels through the C ABI
(``libbezk.so``):

    K0  ``bezk_pre_physics``    action clip, head zeroing, PD targets        (before the simulator)
    K*  ``bezk_post_physics``   timeout, progress, masked reset of the envs flagged by the previous step,
                                54-wide observation, reward / termination / new reset mask   (after it)

``fusion="split"`` launches the north-star's two kernels instead of the fused one (observation kernel =
bookkeeping + reset + observations, then the reward / termination kernel).  There is no CPU path: with
``use_gpu_pipeline: False`` the simulator tensors stay in pinned host memory and are staged to the GPU each step.

Reference behaviours kept bug-for-bug (SURVEY 7 "hard parts"): xyzw quaternion fed to the real-first matrix
formula; unit gravity vector; ``prev_lin_vel`` aliasing the velocity view after the first observation (so
``lin_acc == R(q)(0,0,1)`` from the second step on; ``env.imuPrevVelAliasing: False`` keeps a real buffer);
in-place contact noise filter; resets applied at the start of the NEXT step; ``reset_buf`` starting at ones.
Documented deviations: reset noise comes from Philox4x32-10 keyed by (seed, step, env id) instead of torch's
global generator (invariant to sharding and to how many envs reset); ``default_dof_pos`` / joint limits are
kernel constants (the ``(N,18)`` tensor attributes are kept for API compatibility); ``obs_dict['obs']``
aliases ``obs_buf`` when ``clip_obs`` is infinite (the reference's clamp is then a plain copy).
"""
import ctypes as C
import math
import weakref

import numpy as np
import torch

from .. import _lib, bez_model as bm, ops
from ..synthetic_sim import SimBackend, SyntheticGym
from .base.vec_task import VecTask

_P = C.c_void_p


def _ptr(t):
    return _P(t.data_ptr()) if t is not None else None


def _l2_release(lib, tensors):
    if torch.cuda.is_current_stream_capturing():   # collected while another graph is being captured: not into that graph
        return
    for t in tensors:
        lib.bezk_l2_release(t.data_ptr(), t.numel() * t.element_size(), torch.cuda.current_stream(t.device).cuda_stream)


class KickEnv(VecTask):
    #: "kick" here; the sibling tasks (tasks/walk_env.py, tasks/orient_env.py) subclass this with "walk" / "orient": same
    #: skeleton, one actor per env, 52-wide observation, their own heading term / reward / goal randomisation (bezk.h)
    TASK = "kick"
    #: host pipelines (``sim.use_gpu_pipeline: False``), selected by ``env.hostPipeline``
    HOST_PIPELINES = ("zero_copy", "staged", "staged_ce", "staged_pack")

    def __init__(self, cfg, sim_device, graphics_device_id, headless, sim: SimBackend = None, fusion="fused"):
        self.cfg = cfg
        env_cfg = cfg["env"]
        self.randomize = cfg["task"]["randomize"]
        self.randomization_params = cfg["task"].get("randomization_params", {})
        if fusion not in ("fused", "split"):
            raise ValueError(fusion)
        self.fusion = fusion

        def state13(key):
            s = env_cfg[key]
            return list(s["pos"]) + list(s["rot"]) + list(s["vLinear"]) + list(s["vAngular"])

        self._state13 = state13
        self.bez_init_state = state13("bezInitState")
        self._read_task_cfg(env_cfg)
        goal = env_cfg["goalState"]["goal"]
        self._actors, _, self._obs_width = bm.task_dims(self.TASK)
        self.cleats = env_cfg["asset"]["cleats"]
        self.debug_rewards = env_cfg.get("debug", {}).get("rewards", False)
        self.named_default_joint_angles = env_cfg["readyJointAngles"]
        self.max_episode_length_s = env_cfg["learn"]["episodeLength_s"]
        self.Kp = env_cfg["control"]["stiffness"]
        self.Kd = env_cfg["control"]["damping"]
        self.orn_dim, self.imu_dim, self.feet_dim, self.dof_dim, self.rnn_dim, self.ball_dim = 2, 6, 8, 18, 1, 2
        self.imu_max_ang_vel = bm.IMU_MAX_ANG_VEL
        self.imu_max_lin_acc = bm.IMU_MAX_LIN_ACC
        env_cfg["numObservations"] = self._obs_width
        env_cfg["numActions"] = bm.NUM_ACTIONS
        self._sim_arg = sim
        self._seed = int(cfg.get("seed", 42))
        self._alias_prev = bool(env_cfg.get("imuPrevVelAliasing", True))
        #: global id of this instance's env 0 -- the shard offset when num_envs is partitioned over ranks (dist.shard_range).
        #: Keys the Philox reset noise (and, through A2CAgent, the exploration noise) so that results do not depend on sharding.
        self.env_base = int(env_cfg.get("envBase", 0))
        if self.env_base and fusion != "fused":
            raise ValueError("env.envBase needs fusion='fused'")

        super().__init__(config=cfg, sim_device=sim_device, graphics_device_id=graphics_device_id, headless=headless)

        self.dt = cfg["sim"]["dt"]
        self.max_episode_length = int(self.max_episode_length_s / self.dt + 0.5)
        dev, n = self.compute_device, self.num_envs
        f32 = dict(dtype=torch.float32, device=dev)

        # simulator tensors (borrowed) and their device images
        self.root_states, self.dof_state = self.sim.root_states, self.sim.dof_state
        self.rigid_body, self.net_contact = self.sim.rigid_body, self.sim.net_contact
        # host pipelines (every task; default "auto", resolved below): "zero_copy" hands the PINNED host tensors straight to the
        # kernels -- they gather the few bytes they need over PCIe and write resets back in place; "staged" copies all four
        # tensors to HBM first;
        # "staged_ce" moves everything with the copy engines in a chunked three-stream pipeline (dense tensors by
        # cudaMemcpyAsync, the sparse AoS rows by strided cudaMemcpy2DAsync pulls, results back by cudaMemcpyAsync);
        # "staged_pack" is staged_ce with the sparse rows gathered by HOST worker threads into pinned pack buffers
        # (bezk_host_pack_begin / _wait) and moved by dense copies -- the engine is row-rate-bound on strided pulls
        self.host_mode = env_cfg.get("hostPipeline", "auto") if self.host_staged else None
        if self.host_mode == "auto":
            # the fastest pipeline for this size on this host (profiles/r02_host_pack.md).  Small tasks (< 49 152 envs): the
            # zero-copy kernels (two launches, no staging: 0.12 ms per step at the reference's default 4 096 envs vs 0.21-0.57 ms
            # for a staged pipeline's copies, events and launches).  Large ones: the packed pipeline when the process has ~8 worker threads
            # to stay ahead of the link (98 vs 69 M env-steps/s at 262 144 envs on 16 cores / 1 GPU); with 4 cores per GPU
            # (8 ranks on 32 cores) the gather becomes the bottleneck and the copy-engine pulls win (176 vs 151 M).
            n_envs = int(env_cfg["numEnvs"])
            pack_ok = self._host_core_share() - 1 >= 8
            if fusion != "fused" or bool(env_cfg.get("writeContactFilter", False)):
                self.host_mode = "zero_copy"              # the staged pipelines run the fused step and cannot write the filter back
            elif n_envs < 49152:                          # 16 384 envs: zero_copy 0.33 ms, packed 0.32; 65 536: 1.23 vs 0.82
                self.host_mode = "zero_copy"
            elif pack_ok and self._host_gather_fast_enough():
                # (a core count says little about an overcommitted guest: the gather itself is timed before it is relied on)
                self.host_mode = "staged_pack"
            else:
                self.host_mode = "staged_ce" if n_envs >= 98304 else "zero_copy"
        #: the resolved pipeline name ("staged_pack" runs on the staged_ce machinery: host_mode reads "staged_ce" for both)
        self.host_pipeline = self.host_mode
        self._pack = self.host_mode == "staged_pack"
        if self._pack:
            self.host_mode = "staged_ce"                  # same pipeline; only the sparse staging differs
        if self.host_mode is not None and self.host_mode not in self.HOST_PIPELINES + ("auto",):
            raise ValueError(f"env.hostPipeline must be one of {self.HOST_PIPELINES}, got {self.host_mode}")
        if self.host_staged and self.host_mode in ("zero_copy", "staged_ce") and not all(
                t.is_pinned() for t in (self.root_states, self.dof_state, self.rigid_body, self.net_contact)):
            raise ValueError(f"hostPipeline='{self.host_mode}' needs the simulator tensors in pinned (page-locked) host memory")
        if self.host_mode == "staged_ce":
            self._d_root, self._d_dof = (torch.empty_like(t, device=dev) for t in (self.root_states, self.dof_state))
            if self._pack:                               # per-env records (bezk_host_pack_begin): IMU slice, foot rows, root subset
                self._d_rb = self._d_cf = None
                self._d_root.copy_(self.root_states)      # the columns the step reads are refreshed from the records every step
            else:
                self._d_rb = torch.zeros(n, 10, **f32)                                # IMU-link slices (bezk_stage_sparse_rows)
                self._d_cf = torch.zeros(n, 24 if self.cleats else 8, **f32)          # foot / cleat force rows
        elif self.host_mode == "staged":
            self._d_root, self._d_dof = (torch.empty_like(t, device=dev) for t in (self.root_states, self.dof_state))
            self._d_rb, self._d_cf = (torch.empty_like(t, device=dev) for t in (self.rigid_body, self.net_contact))
        else:
            self._d_root, self._d_dof, self._d_rb, self._d_cf = self.root_states, self.dof_state, self.rigid_body, self.net_contact
        for name, t, width in (("root_states", self.root_states, 13 * self._actors), ("dof_state", self.dof_state, 36),
                               ("rigid_body", self.rigid_body, 13 * self.sim.num_bodies),
                               ("net_contact", self.net_contact, 3 * self.sim.num_bodies)):
            if t.dtype != torch.float32 or not t.is_contiguous() or t.numel() != n * width:
                raise ValueError(f"simulator tensor {name} must be contiguous float32 with {n * width} elements")

        self.goal = torch.tensor([goal], **f32).repeat((n, 1))
        self.bez_init_xy = torch.tensor(self.bez_init_state[0:2], **f32)
        self.ball_init = self.goal_angle = None
        self._init_task_tensors(env_cfg, n, f32)          # initial_root_states (+ ball_init / goal_angle): per task
        self.initial_root_states[:, 7:13] = 0
        self.num_dof = bm.NUM_DOF
        self.num_dofs = bm.NUM_DOF
        self.dof_names = list(bm.DOF_NAMES)

        # strided views with the reference's names (kick_env.py:168-196)
        self.dof_pos_bez = self.dof_state.view(n, 18, -1)[..., 0]
        self.dof_vel_bez = self.dof_state.view(n, 18, -1)[..., 1]
        self.root_pos_bez = self.root_states.view(n, -1, 13)[..., 0, 0:3]
        self.root_orient_bez = self.rigid_body.view(n, -1, 13)[..., bm.IMU_BODY, 3:7]
        self.root_vel_bez = self.rigid_body.view(n, -1, 13)[..., bm.IMU_BODY, 7:10]
        self.root_ang_bez = self.rigid_body.view(n, -1, 13)[..., bm.IMU_BODY, 10:13]
        self._init_task_views(n)

        ready = [float(self.named_default_joint_angles[name]) for name in bm.DOF_NAMES]
        self.default_dof_pos = torch.tensor(ready, **f32).repeat((n, 1))
        self.dof_pos_limits_lower = torch.tensor(bm.DOF_LOWER, **f32)
        self.dof_pos_limits_upper = torch.tensor(bm.DOF_UPPER, **f32)
        self.gravity_vec = torch.tensor([[0.0, 0.0, -1.0]], **f32).repeat((n, 1))
        self.up_vec = torch.tensor([[0.0, 0.0, 1.0]], **f32).repeat((n, 1))

        self._kcfg = ops.make_task_cfg(
            num_bodies=self.sim.num_bodies, cleats=self.cleats, dt=self.dt, max_episode_length=self.max_episode_length,
            clip_actions=float(self.clip_actions), clip_obs=float(self.clip_obs), default_dof_pos=ready,
            bez_init_xy=tuple(self.bez_init_state[0:2]),
            write_contact_filter=bool(env_cfg.get("writeContactFilter", not self.host_staged)) and self.host_mode != "staged_ce",
            reset_root_states=not self.sim.owns_root_reset)

        # persistent task state
        self._prev_buf = torch.zeros(n, 3, **f32)       # the reference's int64 zeros, promoted (kick_env.py:183)
        self._prev_is_view = False
        # PD targets go to the simulator: pinned host memory (written by K0 over PCIe) when the simulator lives on the host
        self.targets = torch.zeros(n, 18, dtype=torch.float32).pin_memory() if self.host_mode in ("zero_copy", "staged_ce") \
            else torch.zeros(n, 18, **f32)
        self._d_targets = torch.zeros(n, 18, **f32) if self.host_mode == "staged_ce" else self.targets
        self._actions_in = torch.zeros(n, 18, **f32)      # staging buffer for actions arriving from another device
        self._actions_src = self._actions_in
        self._actions_cache = None
        self.obs_clipped_buf = torch.zeros(n, self._obs_width, **f32) if math.isfinite(float(self.clip_obs)) else None
        if self.host_mode == "zero_copy":
            # write-only outputs live in pinned host memory: the kernel's stores (TMA bulk store for the obs tile) cross
            # PCIe while its gathers come the other way (full duplex), and step() needs no D2H copies for them
            self.obs_buf = torch.zeros(n, self._obs_width, dtype=torch.float32).pin_memory()
            self.rew_buf = torch.zeros(n, dtype=torch.float32).pin_memory()
            self.timeout_buf = torch.zeros(n, dtype=torch.long).pin_memory()
            if self.obs_clipped_buf is not None:
                self.obs_clipped_buf = torch.zeros(n, self._obs_width, dtype=torch.float32).pin_memory()
        self._rng_step = 0
        self._ce_copy_out = False
        self._rollout = None                # (BezkRolloutCfg, values, shaped_rewards, dones_u8) set by set_rollout_targets
        self._episode = None                # (episode_returns, episode_lengths, episode_partials) set by set_rollout_targets
        self._obs_norm = None               # (obs_mean, obs_var, obs_eps, obs_norm) set by set_rollout_targets
        self._d_values = None               # staged_ce host pipeline: device image of host-resident critic values
        self._lib = _lib.load()
        # the step keeps these in L2 with evict_last (bezk.h, bezk_l2_release): demoted again when the env goes away
        carried = [self.obs_buf, self.obs_clipped_buf, self.reset_buf, self.progress_buf, self.timeout_buf, self.rew_buf,
                   self._prev_buf, self.goal, self.ball_init, self.goal_angle]
        self._l2_finalizer = weakref.finalize(self, _l2_release, self._lib, [t for t in carried if t is not None and t.is_cuda])
        self._l2_finalizer.atexit = False   # at interpreter exit the CUDA context goes away with the process
        if self.host_staged:
            pin = dict(pin_memory=True)
            self._h_obs = torch.empty(n, self._obs_width, **pin); self._h_rew = torch.empty(n, **pin)
            self._h_reset = torch.empty(n, dtype=torch.long, **pin); self._h_timeout = torch.empty(n, dtype=torch.long, **pin)
            self._h_actions = torch.empty(n, 18, **pin)
        if self.host_mode == "staged_ce":
            if self.fusion != "fused":
                raise ValueError("hostPipeline='staged_ce' runs the fused step (fusion='fused')")
            if self._kcfg.flags & _lib.F_WRITE_CONTACT_FILTER:
                raise ValueError("hostPipeline='staged_ce' cannot write the contact filter back (env.writeContactFilter must be False)")
            self._s_in, self._s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
            self._ce_split = bool(env_cfg.get("hostPipelineSplitSparse", True))
            # env.hostPipelineChunks: a count (equal chunks) or a list of relative sizes -- a small first chunk shortens the
            # pipeline's fill (its gather + H2D are exposed), a small last one its drain (its D2H is)
            # default: ~32 768+ envs per chunk, at most 4 (1 chunk at 16 384 envs, 2 at 65 536, 4 from 131 072 on: measured)
            chunks = env_cfg.get("hostPipelineChunks", min(4, max(1, n // 32768)))
            weights = [1.0] * max(1, int(chunks)) if isinstance(chunks, (int, float)) else [float(w) for w in chunks]
            if not weights or min(weights) <= 0:
                raise ValueError("env.hostPipelineChunks must be a positive count or a list of positive relative sizes")
            edges, acc = [0], 0.0
            for w in weights[:-1]:                                     # chunk starts stay multiples of 128 envs (TMA alignment)
                acc += w
                edges.append(min(n, max(edges[-1] + 128, int(round(n * acc / sum(weights) / 128)) * 128)))
            edges.append(n)
            self._ce_chunks = [(lo, hi) for lo, hi in zip(edges[:-1], edges[1:]) if hi > lo]
            #: env.hostPipelineTimeline: timing-enabled events + host stamps of the last step (tools/exp_e2e.py --timeline)
            self._timeline = bool(env_cfg.get("hostPipelineTimeline", False))
            mk = lambda: torch.cuda.Event(enable_timing=self._timeline)               # noqa: E731
            self._ev_in, self._ev_k = [mk() for _ in self._ce_chunks], [mk() for _ in self._ce_chunks]
            self._ev_out, self._ev_t0 = [mk() for _ in self._ce_chunks], mk()
            self._host_stamps = []
            self._ev_tgt = mk()
            self._ev_pack = mk()                                       # last H2D that read the pack buffers
            if self._pack:
                rs = self._lib.bezk_host_pack_record_floats(ops._TASK_ID[self.TASK], C.byref(self._kcfg))
                if rs <= 0:
                    _lib.check(-rs or 1, "bezk_host_pack_record_floats")
                # env.hostPackDof (default off): the workers also copy the chunk's dof_state rows, so that ONE cudaMemcpyAsync per
                # chunk moves [dof rows | records].  A second H2D call per chunk costs the link ~40 us, but streaming 144 B/env
                # through the host cores makes the gather the bottleneck: 81 M vs 92 M env-steps/s (profiles/r02_host_pack.md)
                self._pack_dof = bool(env_cfg.get("hostPackDof", False))
                self._rs = rs
                self._pw = rs + (36 if self._pack_dof else 0)            # floats per env in the pack buffers
                self._h_pack = torch.zeros(n * self._pw, dtype=torch.float32).pin_memory()
                self._d_pack = torch.zeros(n * self._pw, **f32)
                threads = int(env_cfg.get("hostPackThreads", 0))
                if threads <= 0:         # this rank's share of the host cores (one process per GPU), minus the issuing thread
                    threads = max(1, min(16, self._host_core_share() - 1))
                k = self._lib.bezk_host_pack_config(threads, int(env_cfg.get("hostPackSpinUs", -1)), int(env_cfg.get("hostPackPin", -1)))
                if k <= 0:
                    _lib.check(-k or 1, "bezk_host_pack_config")
                self.host_pack_threads = k
        self._bind()
        self._link = {"h2d_bytes": 0, "d2h_bytes": 0}
        self._link_per_step = self._host_link_bytes_per_step() if self.host_staged else (0, 0)
        if self.randomize:                                # kick_env.py:248-249: once at start-up, before the first step
            self.apply_randomizations(self.randomization_params)
        self.reset_idx(torch.arange(n, device=dev))       # kick_env.py:238

    # ------------------------------------------------------------------ per-task pieces (overridden by WalkEnv / OrientEnv)
    def _read_task_cfg(self, env_cfg):
        """BezKick has a second actor, the ball (kick_env.py:161-166)."""
        self.ball_init_state = self._state13("ballInitState")

    def _init_task_tensors(self, env_cfg, n, f32):
        """kick_env.py:159-166, 213: the constant ``ball_init`` rows of the observation and the two-actor reset rows."""
        self.ball_init = torch.tensor([self.ball_init_state[0:2]], **f32).repeat((n, 1))
        self.initial_root_states = torch.tensor([self.bez_init_state, self.ball_init_state], **f32).repeat((n, 1))

    def _init_task_views(self, n):
        """kick_env.py:179-181: the ball's views of the root-state tensor."""
        self.root_pos_ball = self.root_states.view(n, -1, 13)[..., 1, 0:3]
        self.root_orient_ball = self.root_states.view(n, -1, 13)[..., 1, 3:7]
        self.root_vel_ball = self.root_states.view(n, -1, 13)[..., 1, 7:10]

    def _reset_goal_tensor(self):
        """The tensor ``reset_idx`` redraws on reset: none for BezKick (its goal is fixed)."""
        return None

    @staticmethod
    def _host_core_share():
        """Host cores available to this process: the CPU affinity mask divided among the ranks of the node (torchrun's
        LOCAL_WORLD_SIZE; one process per GPU)."""
        import os
        try:
            cores = len(os.sched_getaffinity(0))
        except AttributeError:
            cores = os.cpu_count() or 2
        return max(1, cores // max(1, int(os.environ.get("LOCAL_WORLD_SIZE", "1"))))

    def _host_gather_fast_enough(self, limit_ns_per_env=7.0):
        """Calibration for ``hostPipeline: auto``: the packed pipeline only pays when the host threads gather an env faster than the
        link moves one (~7.6 ns per env-step at 262 144 envs); on the B200 hosts the gather runs at 3-4 ns per env on 15 threads,
        on an overcommitted guest (this repo's development container: 35 ns) the copy-engine pipeline is the better choice.
        Three timed gathers of up to 65 536 envs of the simulator's own tensors, best of three."""
        import time
        lib = _lib.load()
        task = ops._TASK_ID[self.TASK]
        kcfg = ops.make_task_cfg(num_bodies=self.sim.num_bodies, cleats=self.cleats)
        rs = lib.bezk_host_pack_record_floats(task, C.byref(kcfg))
        threads = max(1, min(16, self._host_core_share() - 1))
        if rs <= 0 or lib.bezk_host_pack_config(threads, -1, -1) <= 0:
            return False
        m = min(self.num_envs, 65536)
        rec = torch.empty(m * rs, dtype=torch.float32)
        best = float("inf")
        for _ in range(3):
            t0 = time.perf_counter()
            t = lib.bezk_host_pack_begin(task, _ptr(self.rigid_body), _ptr(self.net_contact), _ptr(self.root_states), None, None,
                                         C.byref(kcfg), _ptr(rec), 0, m)
            if t < 0 or lib.bezk_host_pack_wait(t):
                return False
            best = min(best, time.perf_counter() - t0)
        self.host_gather_ns_per_env = 1e9 * best / m
        return self.host_gather_ns_per_env <= limit_ns_per_env

    # ------------------------------------------------------------------ construction helpers
    def create_sim(self):
        """The reference builds the PhysX scene here (kick_env.py:240-408, out of scope); this attaches the
        simulator backend that owns the state tensors."""
        self.up_axis_idx = 2
        if self._sim_arg is not None:
            self.sim = self._sim_arg
        else:
            host = self.device == "cpu"
            self.sim = SyntheticGym(self.num_environments, device=f"cuda:{self.device_id}", cleats=self.cfg["env"]["asset"]["cleats"],
                                    seed=int(self.cfg.get("seed", 42)), host=host, task=self.TASK)
        if self.sim.root_states.is_cuda != (self.device != "cpu"):
            raise ValueError("simulator tensors must live on the pipeline device "
                             f"({'cuda' if self.device != 'cpu' else 'pinned host'})")

    def _bind(self):
        """Pre-convert every pointer argument once: buffers are persistent, so a step costs two ctypes calls."""
        n = self.num_envs
        kc = C.byref(self._kcfg)
        self._pre_args = [_ptr(self._actions_in), None, _ptr(self.targets), kc, n]
        self._post_fixed = dict(
            head=[_ptr(self._d_dof), _ptr(self._d_rb), _ptr(self._d_root), _ptr(self._d_cf)],
            mid=[_ptr(self.goal), _ptr(self.ball_init), _ptr(self.initial_root_states), None],
            # bezk_post_physics_task: goal, goal_angle, ball_init, initial_root_states, uniforms, goal_uniforms
            mid_task=[_ptr(self.goal), _ptr(self.goal_angle), _ptr(self.ball_init), _ptr(self.initial_root_states), None, None],
            tail=[_ptr(self.reset_buf), _ptr(self.progress_buf), _ptr(self.timeout_buf), None, kc,
                  _ptr(self.obs_buf), _ptr(self.obs_clipped_buf), _ptr(self.rew_buf)])

    def _stream(self):
        return _P(torch.cuda.current_stream(self.compute_device).cuda_stream)

    def _launch_staged(self, parts, lo=0, hi=None, whole_dof=True):
        """``bezk_post_physics_staged`` over envs [lo, hi) of the staged_ce host pipeline (device staging in, device results
        out, reset rows written straight back into the simulator's pinned host tensors)."""
        n = self.num_envs
        hi = n if hi is None else hi
        rw, ow = 13 * self._actors, self._obs_width
        off = lambda t, k: None if t is None else _P(t.data_ptr() + k * t.element_size())      # noqa: E731
        clip = self.obs_clipped_buf
        ro = self._rollout if parts == _lib.PART_ALL else None       # (cfg, values, shaped_rewards, dones_u8): reward epilogue
        if ro is None:
            tail = [None, None, None, None]
        else:                            # values: a device tensor, or None when they ride in the packed records
            dv = ro[1] if (ro[1] is not None and ro[1].is_cuda) else (None if self._pack else self._d_values)
            tail = [C.byref(ro[0]), off(dv, lo), off(ro[2], lo), off(ro[3], lo)]
        if self._pack:
            # chunk (lo, hi) of the pack buffer: [dof rows (hi - lo) x 36 |] records (hi - lo) x rs
            d_dof = off(self._d_pack, lo * self._pw) if (self._pack_dof and not whole_dof) else off(self._d_dof, lo * 36)
            d_rec = off(self._d_pack, lo * self._pw + ((hi - lo) * 36 if self._pack_dof else 0))
            rc = self._lib.bezk_post_physics_packed(
                ops._TASK_ID[self.TASK], d_dof, d_rec, off(self._d_root, lo * rw),
                None if self._prev_is_view else off(self._prev_buf, lo * 3),
                off(self.goal, lo * 2), off(self.goal_angle, lo), off(self.ball_init, lo * 2), off(self.initial_root_states, lo * rw),
                None, None, self._seed, self._rng_step, off(self.reset_buf, lo), off(self.progress_buf, lo), off(self.timeout_buf, lo),
                None, C.byref(self._kcfg), off(self.obs_buf, lo * ow), off(clip, lo * ow), off(self.rew_buf, lo), parts, hi - lo,
                self.env_base + lo, off(self.dof_state, lo * 36), off(self.root_states, lo * rw), *tail, self._stream())
            if rc:
                _lib.check(rc, "bezk_post_physics_packed")
            return
        rc = self._lib.bezk_post_physics_staged(
            ops._TASK_ID[self.TASK], off(self._d_dof, lo * 36), off(self._d_rb, lo * 10), off(self._d_root, lo * rw),
            off(self._d_cf, lo * self._d_cf.shape[1]), None if self._prev_is_view else off(self._prev_buf, lo * 3),
            off(self.goal, lo * 2), off(self.goal_angle, lo), off(self.ball_init, lo * 2), off(self.initial_root_states, lo * rw),
            None, None, self._seed, self._rng_step, off(self.reset_buf, lo), off(self.progress_buf, lo), off(self.timeout_buf, lo),
            None, C.byref(self._kcfg), off(self.obs_buf, lo * ow), off(clip, lo * ow), off(self.rew_buf, lo), parts, hi - lo,
            self.env_base + lo, off(self.dof_state, lo * 36), off(self.root_states, lo * rw), *tail, self._stream())
        if rc:
            _lib.check(rc, "bezk_post_physics_staged")

    def _post_staged_ce(self, copy_out):
        """One post-physics step of the copy-engine host pipeline, chunked so that chunk c's transfers overlap chunk c-1's kernel
        and chunk c-2's results going back: [s_in] dense cudaMemcpyAsync + strided cudaMemcpy2DAsync pulls of the sparse rows ->
        [current stream] fused kernel on device staging -> [s_out] results to the pinned host buffers."""
        cur = torch.cuda.current_stream(self.compute_device)
        rw, ow = 13 * self._actors, self._obs_width
        root_h, root_d = self.root_states.view(-1, rw), self._d_root.view(-1, rw)
        dof_h, dof_d = self.dof_state.view(-1, 36), self._d_dof.view(-1, 36)
        kc = C.byref(self._kcfg)
        self._s_in.wait_stream(cur)                       # staging buffers are free again (previous step's kernels are done)
        s_in_h = _P(self._s_in.cuda_stream)
        out = self._observations_out()
        tl = self._timeline
        if tl:
            import time
            self._host_stamps = [("start", time.perf_counter())]
            self._ev_t0.record(self._s_in)
        tickets = self._pack_begin(self._ce_chunks) if self._pack else None
        if tl:
            self._host_stamps.append(("pack_issued", time.perf_counter()))
        ro = self._rollout
        if ro is not None and ro[1] is not None and not ro[1].is_cuda and not self._pack:
            with torch.cuda.stream(self._s_in):          # copy-engine pipeline: the step's critic values, one dense copy
                self._d_values.copy_(ro[1].view(-1), non_blocking=True)
        for c, (lo, hi) in enumerate(self._ce_chunks):
            with torch.cuda.stream(self._s_in):
                if self._pack:           # records gathered by the host workers while the engine moved the previous chunk
                    if not self._pack_dof and c == 0:
                        dof_d[lo:hi].copy_(dof_h[lo:hi], non_blocking=True)
                    rc = self._lib.bezk_host_pack_wait(tickets[c])
                    if tl:
                        self._host_stamps.append((f"pack_done{c}", time.perf_counter()))
                    pw = self._pw
                    self._d_pack[lo * pw:hi * pw].copy_(self._h_pack[lo * pw:hi * pw], non_blocking=True)
                    if c == len(self._ce_chunks) - 1:
                        self._ev_pack.record(self._s_in)
                    self._ev_in[c].record(self._s_in)
                    if not self._pack_dof and c + 1 < len(self._ce_chunks):      # keep the engine fed while this chunk is launched
                        lo2, hi2 = self._ce_chunks[c + 1]
                        dof_d[lo2:hi2].copy_(dof_h[lo2:hi2], non_blocking=True)
                else:
                    dof_d[lo:hi].copy_(dof_h[lo:hi], non_blocking=True)
                    root_d[lo:hi].copy_(root_h[lo:hi], non_blocking=True)
                    if self._ce_split:   # IMU slices by the copy engine, foot rows by an SM gather kernel on the compute stream
                        rc = self._lib.bezk_stage_sparse_rows_split(_ptr(self.rigid_body), _ptr(self.net_contact), kc,
                                                                    _ptr(self._d_rb), _ptr(self._d_cf), lo, hi - lo, s_in_h,
                                                                    _P(cur.cuda_stream))
                    else:
                        rc = self._lib.bezk_stage_sparse_rows(_ptr(self.rigid_body), _ptr(self.net_contact), kc, _ptr(self._d_rb),
                                                              _ptr(self._d_cf), lo, hi - lo, s_in_h)
                if rc:
                    _lib.check(rc, "bezk_host_pack_wait" if self._pack else "bezk_stage_sparse_rows")
                if not self._pack:
                    self._ev_in[c].record(self._s_in)
            cur.wait_event(self._ev_in[c])
            self._launch_staged(_lib.PART_ALL, lo, hi, whole_dof=False)
            if copy_out:
                self._ev_k[c].record(cur)
                with torch.cuda.stream(self._s_out):
                    self._s_out.wait_event(self._ev_k[c])
                    self._h_obs[lo:hi].copy_(out[lo:hi], non_blocking=True)
                    self._h_rew[lo:hi].copy_(self.rew_buf[lo:hi], non_blocking=True)
                    self._h_reset[lo:hi].copy_(self.reset_buf[lo:hi], non_blocking=True)
                    self._h_timeout[lo:hi].copy_(self.timeout_buf[lo:hi], non_blocking=True)
                    if tl:
                        self._ev_out[c].record(self._s_out)
            if tl:
                self._host_stamps.append((f"issued{c}", time.perf_counter()))

    def host_timeline(self):
        """After a synchronised ``step`` with ``env.hostPipelineTimeline``: per chunk, when its inputs had landed, its kernel had
        finished and its results were back (ms after the step's first copy was queued, device clock), and the host stamps."""
        t0 = self._ev_t0
        dev = [{"chunk": c, "h2d_done": round(t0.elapsed_time(self._ev_in[c]), 4), "kernel_done": round(t0.elapsed_time(self._ev_k[c]), 4),
                "d2h_done": round(t0.elapsed_time(self._ev_out[c]), 4)} for c in range(len(self._ce_chunks))]
        h0 = self._host_stamps[0][1]
        return {"device_ms": dev, "host_ms": {k: round(1e3 * (v - h0), 4) for k, v in self._host_stamps[1:]}}

    def _pack_begin(self, chunks, with_dof=None):
        """Queue the host-side gather of ``chunks`` into their regions of the pinned pack buffer (served in order); returns the
        tickets."""
        self._ev_pack.synchronize()                       # the previous step's copies out of the pack buffer are done
        kc = C.byref(self._kcfg)
        with_dof = self._pack_dof if with_dof is None else with_dof
        ro = self._rollout
        hv = _ptr(ro[1]) if (ro is not None and ro[1] is not None and not ro[1].is_cuda) else None    # host values -> records
        tickets = []
        for lo, hi in chunks:
            dst = _P(self._h_pack.data_ptr() + 4 * (lo * self._pw + (0 if with_dof or not self._pack_dof else (hi - lo) * 36)))
            t = self._lib.bezk_host_pack_begin(ops._TASK_ID[self.TASK], _ptr(self.rigid_body), _ptr(self.net_contact),
                                               _ptr(self.root_states), _ptr(self.dof_state) if with_dof else None, hv, kc, dst,
                                               lo, hi - lo)
            if t < 0:
                _lib.check(int(-t), "bezk_host_pack_begin")
            tickets.append(t)
        return tickets

    def _launch_post(self, parts):
        if self.host_mode == "staged_ce":
            return self._launch_staged(parts)
        f = self._post_fixed
        prev = None if self._prev_is_view else _ptr(self._prev_buf)
        if parts == _lib.PART_ALL:
            # the whole step, with rl_games' per-step reward path in the epilogue when set_rollout_targets() armed it
            ro = self._rollout
            tail = ([C.byref(ro[0]), _ptr(ro[1]), _ptr(ro[2]), _ptr(ro[3])] if ro is not None else [None, None, None, None])
            t = f["tail"]
            if self._episode is not None:     # + rl_games' episode return / length bookkeeping (set_rollout_targets)
                # + the eval-mode observation normaliser when armed (all NULL: exactly bezk_post_physics_rollout_ep)
                mean, var, eps, out = self._obs_norm or (None, None, 0.0, None)
                rc = self._lib.bezk_post_physics_rollout_ep_norm(ops._TASK_ID[self.TASK], *f["head"], prev, *f["mid_task"], self._seed,
                                                                 self._rng_step, t[0], t[1], t[2], t[3], t[4], t[5], t[6], t[7], *tail,
                                                                 self.env_base, self.num_envs, *[_ptr(x) for x in self._episode],
                                                                 _ptr(mean), _ptr(var), eps, _ptr(out), self._stream())
                if rc:
                    _lib.check(rc, "bezk_post_physics_rollout_ep_norm")
                return
            rc = self._lib.bezk_post_physics_rollout(ops._TASK_ID[self.TASK], *f["head"], prev, *f["mid_task"], self._seed,
                                                     self._rng_step, t[0], t[1], t[2], t[3], t[4], t[5], t[6], t[7], *tail,
                                                     self.env_base, self.num_envs, self._stream())
            if rc:
                _lib.check(rc, "bezk_post_physics_rollout")
            return
        if self.TASK == "kick":
            rc = self._lib.bezk_post_physics(*f["head"], prev, *f["mid"], self._seed, self._rng_step, *f["tail"], parts,
                                             self.num_envs, self._stream())
        else:
            rc = self._lib.bezk_post_physics_task(ops._TASK_ID[self.TASK], *f["head"], prev, *f["mid_task"], self._seed,
                                                  self._rng_step, *f["tail"], parts, self.num_envs, self._stream())
        if rc:
            _lib.check(rc, "bezk_post_physics")

    # ------------------------------------------------------------------ host-link accounting (bench.py's e2e byte counts)
    def _host_link_bytes_per_step(self):
        """Bytes one ``step`` moves over the host link, from the tensors / address ranges involved (not a formula per env):
        staged = the sizes of the tensors copied; zero_copy = the dense tensors the kernels read / write in pinned memory
        whole, plus the sparse AoS rows counted as the DISTINCT 64-byte granules their address ranges touch."""
        n, nb = self.num_envs, self.sim.num_bodies
        nbytes = lambda t: t.numel() * t.element_size()      # noqa: E731
        outs = nbytes(self._observations_out()) + nbytes(self.rew_buf) + nbytes(self.timeout_buf) + nbytes(self.reset_buf) \
            + nbytes(self.targets)
        e = np.arange(n, dtype=np.int64)

        def granules(base, stride, off, width):               # distinct 64-byte granules of [a, a + width) per env
            a = base + e * stride + off
            return int(((a + width - 1) // 64 - a // 64 + 1).sum()) * 64
        fw = 48 if self.cleats else 12
        if self.host_mode == "staged_ce":                 # the arguments of the copies issued each step
            if self._pack:                                # dense copies: dof_state, the packed records, the actions
                return (0 if self._pack_dof else nbytes(self.dof_state)) + nbytes(self._h_pack) + n * 18 * 4, outs
            if self._ce_split:                          # foot rows: zero-copy reads of the gather kernel, as 64-byte granules
                feet = granules(self.net_contact.data_ptr(), nb * 12, self._kcfg.left_foot_body * 12, fw) + \
                    granules(self.net_contact.data_ptr(), nb * 12, self._kcfg.right_foot_body * 12, fw)
            else:
                feet = n * 2 * fw
            return nbytes(self.dof_state) + nbytes(self.root_states) + n * 18 * 4 + n * 40 + feet, outs
        if self.host_mode == "staged":
            h2d = sum(nbytes(t) for t in (self.root_states, self.dof_state, self.rigid_body, self.net_contact)) + n * 18 * 4
            d2h = outs + nbytes(self.dof_state)
            if self._kcfg.flags & _lib.F_WRITE_CONTACT_FILTER:
                d2h += nbytes(self.net_contact)
            if self._kcfg.flags & _lib.F_RESET_ROOT_STATES:
                d2h += nbytes(self.root_states)
            return h2d, d2h
        sparse = granules(self.rigid_body.data_ptr(), nb * 52, (bm.IMU_BODY * 13 + 3) * 4, 40)
        sparse += granules(self.net_contact.data_ptr(), nb * 12, self._kcfg.left_foot_body * 12, fw)
        sparse += granules(self.net_contact.data_ptr(), nb * 12, self._kcfg.right_foot_body * 12, fw)
        h2d = nbytes(self.dof_state) + nbytes(self.root_states) + n * 18 * 4 + sparse
        return h2d, outs

    def reset_link_counters(self):
        self._link = {"h2d_bytes": 0, "d2h_bytes": 0}

    def link_counters(self):
        how = {"staged": "sizes of the tensors copied by cudaMemcpyAsync each step",
               "staged_pack": "byte counts of the cudaMemcpyAsync calls issued each step (the pack buffer the host worker threads fill: dense "
                              "dof_state rows + per-env records of the sparse rows and the root-state subset; actions; results and PD "
                              "targets back) "
                              "(+ the rare reset rows the kernel writes back into the simulator's host tensors, not counted)",
               "staged_ce": "byte counts of the cudaMemcpyAsync / cudaMemcpy2DAsync (width x rows) calls issued each step; with the split "
                            "sparse staging (default) the foot rows are zero-copy reads of a gather kernel, counted as distinct 64-byte "
                            "granules (+ the rare reset rows the kernel writes back into the simulator's host tensors, not counted)",
               "zero_copy": "address ranges the kernels dereference in pinned host memory each step: dense tensors whole, sparse AoS rows as "
                            "distinct 64-byte granules (+ the rare reset rows written back, not counted)",
               None: "GPU pipeline: nothing crosses the host link"}["staged_pack" if self._pack else self.host_mode]
        return dict(self._link, how=how)

    # ------------------------------------------------------------------ reference-named attributes
    @property
    def actions(self):
        """``self.actions`` of the reference (clipped, head zeroed, kick_env.py:413-414), materialised on demand."""
        if self._actions_cache is None:
            a = torch.clamp(self._actions_src.to(self.compute_device), -self.clip_actions, self.clip_actions)
            a[..., 0:2] = 0.0
            self._actions_cache = a
        return self._actions_cache

    @property
    def randomize_buf(self):
        """``randomize_buf += 1`` per step (kick_env.py:430) is applied lazily: with domain randomisation out of
        scope nothing on the device reads it, so the 16 B/env-step of traffic is only paid when somebody looks."""
        if self._randomize_pending:
            self._randomize_base += self._randomize_pending
            self._randomize_pending = 0
        return self._randomize_base

    @randomize_buf.setter
    def randomize_buf(self, value):
        self._randomize_base = value
        self._randomize_pending = 0

    @property
    def prev_lin_vel(self):
        return self.root_vel_bez if self._prev_is_view else self._prev_buf

    @property
    def feet(self):
        return self.obs_buf[:, bm.OBS_FEET]

    # ------------------------------------------------------------------ the step
    def _stage_in(self):
        if self.host_mode == "staged":
            for d, h in ((self._d_root, self.root_states), (self._d_dof, self.dof_state), (self._d_rb, self.rigid_body),
                         (self._d_cf, self.net_contact)):
                d.copy_(h, non_blocking=True)
        elif self.host_mode == "staged_ce":                # unchunked, on the current stream: the stand-alone calls
            self._d_root.copy_(self.root_states, non_blocking=True)
            self._d_dof.copy_(self.dof_state, non_blocking=True)
            if self._pack:                                 # the records of "chunk" (0, n); dof_state went dense above
                n = self.num_envs
                rc = self._lib.bezk_host_pack_wait(self._pack_begin([(0, n)], with_dof=False)[0])
                o = n * 36 if self._pack_dof else 0
                self._d_pack[o:o + n * self._rs].copy_(self._h_pack[o:o + n * self._rs], non_blocking=True)
                self._ev_pack.record(torch.cuda.current_stream(self.compute_device))
            else:
                rc = self._lib.bezk_stage_sparse_rows(_ptr(self.rigid_body), _ptr(self.net_contact), C.byref(self._kcfg),
                                                      _ptr(self._d_rb), _ptr(self._d_cf), 0, self.num_envs, self._stream())
            if rc:
                _lib.check(rc, "bezk_stage_sparse_rows")

    def pre_physics_step(self, actions):
        """kick_env.py:410-419 (+ the clamp of vec_task.py:317): one K0 launch."""
        if actions.shape != (self.num_envs, 18) or actions.dtype != torch.float32:
            raise ValueError(f"actions must be float32 of shape ({self.num_envs}, 18)")
        if self.host_mode == "staged_ce":
            return self._pre_physics_staged_ce(actions)
        if actions.device != self.compute_device:
            if self.host_staged and actions.device.type == "cpu" and not actions.is_pinned():
                self._h_actions.copy_(actions)
                actions = self._h_actions
            if self.host_mode == "zero_copy" and actions.device.type == "cpu" and actions.is_contiguous():
                src = actions                   # K0 reads the pinned host buffer directly
            else:
                self._actions_in.copy_(actions, non_blocking=True)
                src = self._actions_in
        else:
            src = actions if actions.is_contiguous() else actions.contiguous()
        self._actions_cache = None
        self._actions_src = src
        a = self._pre_args
        rc = self._lib.bezk_pre_physics(_ptr(src), a[1], a[2], a[3], a[4], self._stream())
        if rc:
            _lib.check(rc, "bezk_pre_physics")
        self.sim.set_dof_position_targets(self.targets)

    def _pre_physics_staged_ce(self, actions):
        """actions H2D [s_in] -> K0 [current stream] -> PD targets D2H into the simulator's pinned ``targets`` [s_out], in the
        same chunks as the post-physics pipeline so that the two directions of the link overlap."""
        cur = torch.cuda.current_stream(self.compute_device)
        if actions.device.type == "cpu" and not actions.is_pinned():
            self._h_actions.copy_(actions)
            actions = self._h_actions
        self._actions_cache = None
        on_device = actions.device == self.compute_device
        src = (actions if actions.is_contiguous() else actions.contiguous()) if on_device else self._actions_in
        self._actions_src = src
        kc = C.byref(self._kcfg)
        if not on_device:                                 # every chunk's H2D is queued first: the engine streams them back to back
            self._s_in.wait_stream(cur)                   # while the launches / D2H copies below are being issued
            with torch.cuda.stream(self._s_in):
                for c, (lo, hi) in enumerate(self._ce_chunks):
                    self._actions_in[lo:hi].copy_(actions[lo:hi], non_blocking=True)
                    self._ev_in[c].record(self._s_in)
        for c, (lo, hi) in enumerate(self._ce_chunks):
            if not on_device:
                cur.wait_event(self._ev_in[c])
            rc = self._lib.bezk_pre_physics(_P(src.data_ptr() + lo * 72), None, _P(self._d_targets.data_ptr() + lo * 72), kc, hi - lo,
                                            self._stream())
            if rc:
                _lib.check(rc, "bezk_pre_physics")
            self._ev_k[c].record(cur)
            with torch.cuda.stream(self._s_out):
                self._s_out.wait_event(self._ev_k[c])
                self.targets[lo:hi].copy_(self._d_targets[lo:hi], non_blocking=True)
        self._ev_tgt.record(self._s_out)
        self.sim.set_dof_position_targets(self.targets)

    def post_physics_step(self):
        """vec_task.py:331-332 + kick_env.py:426-438 in one launch (two with ``fusion='split'``)."""
        self._rng_step += 1
        self._randomize_pending += 1                      # randomize_buf += 1 (kick_env.py:430), applied lazily
        if self.randomize and self._resets_pending():     # reset_idx -> apply_randomizations (kick_env.py:433-435, 781-782)
            self.apply_randomizations(self.randomization_params)
        if self.host_mode == "staged_ce" and self.fusion == "fused":
            self._post_staged_ce(copy_out=self._ce_copy_out)
            if self._alias_prev:
                self._prev_is_view = True
            return
        self._stage_in()
        if self.fusion == "fused":
            self._launch_post(_lib.PART_ALL)
        else:
            self._launch_post(_lib.PART_BOOKKEEP | _lib.PART_OBS)
            self._launch_post(_lib.PART_REWARD)
        if self._alias_prev:
            self._prev_is_view = True       # kick_env.py:930: compute_imu hands back the velocity VIEW
        if self.host_mode == "staged":
            self.dof_state.copy_(self._d_dof, non_blocking=True)      # resets are written into the simulator tensor
            if self._kcfg.flags & _lib.F_WRITE_CONTACT_FILTER:
                self.net_contact.copy_(self._d_cf, non_blocking=True)
            if self._kcfg.flags & _lib.F_RESET_ROOT_STATES:
                self.root_states.copy_(self._d_root, non_blocking=True)

    def compute_observations(self):
        """kick_env.py:749-777 as a stand-alone call (observation kernel only, no bookkeeping)."""
        self._stage_in()
        prev = None if self._prev_is_view else self._prev_buf
        if self.host_mode == "staged_ce":
            self._launch_staged(_lib.PART_OBS)
        elif self.TASK == "kick":
            ops.compute_observations(self._d_dof, self._d_rb, self._d_root, self._d_cf, self.goal, self.ball_init, self._kcfg,
                                     self.obs_buf, prev_lin_vel=prev, obs_clipped=self.obs_clipped_buf)
        else:
            ops.post_physics_task(self.TASK, self._d_dof, self._d_rb, self._d_root, self._d_cf, self.goal, None, None, None, None,
                                  self._kcfg, self.obs_buf, None, goal_angle=self.goal_angle, prev_lin_vel=prev,
                                  obs_clipped=self.obs_clipped_buf, parts=_lib.PART_OBS)
        if self._alias_prev:
            self._prev_is_view = True

    def compute_reward(self, actions=None):
        """kick_env.py:724-747 as a stand-alone call (reward / termination kernel only)."""
        if self.host_mode == "staged_ce":
            self._stage_in()
            self._launch_staged(_lib.PART_REWARD)
        elif self.TASK == "kick":
            ops.compute_reward(self._d_dof, self._d_rb, self._d_root, self.goal, self.ball_init, self.reset_buf,
                               self.progress_buf, self._kcfg, self.rew_buf, self.reset_buf)
        else:
            ops.post_physics_task(self.TASK, self._d_dof, self._d_rb, self._d_root, None, self.goal, None, self.reset_buf,
                                  self.progress_buf, None, self._kcfg, None, self.rew_buf, goal_angle=self.goal_angle,
                                  parts=_lib.PART_REWARD)

    def close(self):
        """Give back the L2 priority the step gave this env's carried buffers (also done when the env is collected)."""
        self._l2_finalizer()

    def reset_idx(self, env_ids):
        """kick_env.py:779-850 for an explicit id list (the per-step path uses the masked reset inside the fused
        kernel instead, which needs no ``nonzero()``)."""
        env_ids = env_ids.to(device=self.compute_device, dtype=torch.long).contiguous()
        if self.randomize:                                # kick_env.py:781-782
            self.apply_randomizations(self.randomization_params)
        self._stage_in()
        ops.reset_idx_task(self.TASK, env_ids, self._d_dof, self._d_root, self.initial_root_states,
                           self._reset_goal_tensor(), self.progress_buf, self.reset_buf, self._kcfg,
                           seed=self._seed, step=self._rng_step, env_base=self.env_base)
        if self.host_mode in ("staged", "staged_ce"):
            self.dof_state.copy_(self._d_dof)
            if self._kcfg.flags & _lib.F_RESET_ROOT_STATES:
                self.root_states.copy_(self._d_root)

    def _observations_out(self):
        return self.obs_buf if self.obs_clipped_buf is None else self.obs_clipped_buf

    def _resets_pending(self):
        """``len(reset_buf.nonzero()) > 0`` -- the reference's per-step host sync (kick_env.py:432-434), paid here ONLY when
        domain randomisation is on (its frequency gate is host logic); the default path never syncs."""
        return bool(self.reset_buf.any())

    # ------------------------------------------------------------------ rollout-storage hooks (SURVEY 8f rows 1-2)
    def set_obs_target(self, tensor):
        """Make the step kernel write its (N,54) observation rows straight into ``tensor`` -- e.g.
        ``experience.slot('obses', t)`` -- instead of a private buffer (rl_games copies ``obs`` into its experience
        buffer after every step; here the copy never happens).  ``obs_buf`` (``obs_clipped_buf`` when ``clip_obs`` is finite)
        becomes that tensor."""
        if self.host_staged:
            raise NotImplementedError("set_obs_target needs the GPU pipeline")
        if tensor.shape != (self.num_envs, self._obs_width) or tensor.dtype != torch.float32 or not tensor.is_contiguous() \
                or tensor.device != self.compute_device:
            raise ValueError(f"obs target must be a contiguous float32 ({self.num_envs}, {self._obs_width}) tensor on "
                             f"{self.compute_device}")
        self._kcfg.flags |= _lib.F_OBS_STREAMED      # a rollout slot is written once per rollout: not worth keeping in L2
        if self.obs_clipped_buf is not None:
            # finite clip_obs: what step() returns -- and what rl_games stores -- is the CLIPPED row (vec_task.py:343); the
            # raw obs_buf stays private
            self.obs_clipped_buf = tensor
            self._post_fixed["tail"][6] = _ptr(tensor)
        else:
            self.obs_buf = tensor
            self._post_fixed["tail"][5] = _ptr(tensor)

    def set_rollout_targets(self, values=None, shaped_rewards=None, dones_u8=None, gamma=0.99, scale_value=0.01, shift_value=0.0,
                            value_bootstrap=True, episode_returns=None, episode_lengths=None, episode_partials=None, obs_norm=None,
                            obs_mean=None, obs_var=None, obs_eps=1e-5):
        """Arm the reward epilogue of the fused step (SURVEY 8 a16; rl_games ``play_steps``): the NEXT steps also write
        ``shaped_rewards = (rew + shift) * scale + gamma * values * time_outs`` (e.g. ``mb_rewards[t]``) and the uint8 reset
        mask ``dones_u8`` (e.g. the experience buffer's ``dones`` slot ``t + 1``).  ``values``: the (N,)/(N,1) un-normalised
        critic values of the step (what ``policy_head`` wrote).
        ``episode_returns`` / ``episode_lengths`` ((N,) float32) and ``episode_partials`` ((3, ceil(N/32)) float64), all three or
        none, GPU pipeline only: the step also carries rl_games' ``current_rewards`` / ``current_lengths`` (unshaped reward; zeroed
        by a multiply when the env is done) and writes its done envs' count / return sum / length sum per group of 32 envs, the
        input of ``learner.EpisodeMeter``.
        ``obs_norm`` ((N, obs width) float32), ``obs_mean`` / ``obs_var`` ((obs width,) float64), all three or none, with the episode
        tensors armed, GPU pipeline only: the step also writes the row it returns through ``RunningMeanStd.forward`` in eval mode
        (``running_mean`` / ``running_var``, epsilon ``obs_eps``; read on the device every step) into ``obs_norm`` -- the input of
        ``learner.PpoPlayerContinuous``' policy.  Call with no arguments to disarm everything."""
        if self.fusion != "fused":
            raise NotImplementedError("the reward epilogue rides in the fused step (fusion='fused')")
        n, dev = self.num_envs, self.compute_device
        norm = (obs_mean, obs_var, obs_norm)
        if any(t is not None for t in norm):
            if self.host_staged:
                raise NotImplementedError("the fused observation normaliser needs the GPU pipeline")
            if self.dr_randomizations.get("observations", None):
                # the noise is applied after the step kernel: a normaliser inside it would see the noise-free rows
                raise NotImplementedError("observation domain randomisation is active: normalise the noisy rows separately")
            if any(t is None for t in norm):
                raise ValueError("obs_norm, obs_mean and obs_var are armed together")
            if episode_returns is None:
                raise ValueError("obs_norm needs the episode tensors (episode_returns, episode_lengths, episode_partials)")
            w = self._obs_width
            for t, dtype, numel, name in zip(norm, (torch.float64, torch.float64, torch.float32), (w, w, n * w),
                                             ("obs_mean", "obs_var", "obs_norm")):
                if t.dtype != dtype or t.numel() != numel or not t.is_contiguous() or t.device != dev:
                    raise ValueError(f"{name} must be a contiguous {dtype} tensor with {numel} elements on {dev}")
            norm = (obs_mean, obs_var, float(obs_eps), obs_norm)
        else:
            norm = None
        eps = (episode_returns, episode_lengths, episode_partials)
        if any(t is not None for t in eps):
            if self.host_staged:
                raise NotImplementedError("episode statistics need the GPU pipeline")
            if any(t is None for t in eps):
                raise ValueError("episode_returns, episode_lengths and episode_partials are armed together")
            for t, dtype, numel, name in zip(eps, (torch.float32, torch.float32, torch.float64), (n, n, 3 * ((n + 31) // 32)),
                                             ("episode_returns", "episode_lengths", "episode_partials")):
                if t.dtype != dtype or t.numel() != numel or not t.is_contiguous() or t.device != dev:
                    raise ValueError(f"{name} must be a contiguous {dtype} tensor with {numel} elements on {dev}")
            self._episode = eps
        else:
            self._episode = None
        self._obs_norm = norm
        if shaped_rewards is None and dones_u8 is None:
            self._rollout = None
            return

        def chk(t, dtype, name, host_ok=False):
            if t is None:
                return None
            on_host = host_ok and self.host_staged and t.device.type == "cpu"
            if on_host and not t.is_pinned():
                raise ValueError(f"{name} on the host must be pinned")
            if t.dtype != dtype or t.numel() != n or not t.is_contiguous() or (t.device != dev and not on_host):
                raise ValueError(f"{name} must be a contiguous {dtype} tensor with {n} elements on {dev}"
                                 + (" (or pinned host memory)" if host_ok and self.host_staged else ""))
            return t

        if shaped_rewards is not None and value_bootstrap and values is None:
            raise ValueError("value_bootstrap needs the step's critic values")
        # host pipelines: `values` may live in pinned HOST memory (the policy ran there) -- staged_pack carries them in the
        # records' pad float, staged_ce uploads them with one dense copy, zero_copy / staged let the kernel read them in place;
        # the outputs stay DEVICE tensors (the rollout storage GAE reads)
        values = chk(values, torch.float32, "values", host_ok=True)
        if values is not None and not values.is_cuda and self.host_mode == "staged_ce" and not self._pack and self._d_values is None:
            self._d_values = torch.zeros(n, dtype=torch.float32, device=dev)
        self._rollout = (ops.make_rollout_cfg(gamma, scale_value, shift_value, value_bootstrap), values,
                         chk(shaped_rewards, torch.float32, "shaped_rewards"), chk(dones_u8, torch.uint8, "dones_u8"))

    def step_precomputed_targets(self, env_actions=None):
        """``step`` for callers whose PD ``targets`` were already written by ``learner.policy_head(..., env=self)`` (the
        policy-head kernel runs K0 in its epilogue): simulate + post-physics only.  ``env_actions``: what ``self.actions``
        should report (the clamped actions the head produced)."""
        if self.host_staged:
            raise NotImplementedError("step_precomputed_targets needs the GPU pipeline")
        if self.dr_randomizations.get("actions", None):
            # vec_task.py:314-315 perturbs the actions BEFORE pre_physics_step; the targets handed over here were computed from
            # the noise-free actions, so this path would silently drop the action noise
            raise RuntimeError("action domain randomisation is active: use env.step(actions) (the noise precedes the PD targets)")
        if env_actions is not None:
            self._actions_cache = None
            self._actions_src = env_actions
        self.sim.set_dof_position_targets(self.targets)
        for _ in range(self.control_freq_inv):
            self.sim.simulate()
        self.post_physics_step()
        self._apply_obs_randomization()                   # vec_task.py:338-339, 343
        self.extras["time_outs"] = self.timeout_buf.to(self.rl_device)
        self.obs_dict["obs"] = self._observations_out().to(self.rl_device)
        return self.obs_dict, self.rew_buf.to(self.rl_device), self.reset_buf.to(self.rl_device), self.extras

    def step(self, actions):
        if not self.host_staged:
            return super().step(actions)
        # host pipeline: same sequence, results leave through pinned buffers with ONE stream sync
        self._link["h2d_bytes"] += self._link_per_step[0]
        self._link["d2h_bytes"] += self._link_per_step[1]
        self.pre_physics_step(actions)
        # a simulator on the host reads the PD targets now: they must have landed in its memory
        if self.host_mode == "staged_ce":
            self._ev_tgt.synchronize()
        else:
            torch.cuda.current_stream(self.compute_device).synchronize()
        for _ in range(self.control_freq_inv):
            self.sim.simulate()
        if self.host_mode == "staged_ce":
            self._ce_copy_out = True
            try:
                self.post_physics_step()
            finally:
                self._ce_copy_out = False
            self._s_out.synchronize()
            torch.cuda.current_stream(self.compute_device).wait_stream(self._s_out)
            rl = torch.device(self.rl_device)
            if rl.type == "cpu":
                self.extras["time_outs"] = self._h_timeout
                self.obs_dict["obs"] = self._h_obs
                return self.obs_dict, self._h_rew, self._h_reset, self.extras
            self.extras["time_outs"] = self.timeout_buf.to(rl)
            self.obs_dict["obs"] = self._observations_out().to(rl)
            return self.obs_dict, self.rew_buf.to(rl), self.reset_buf.to(rl), self.extras
        self.post_physics_step()
        self._h_reset.copy_(self.reset_buf, non_blocking=True)
        if self.host_mode == "zero_copy":
            h_obs, h_rew, h_timeout = self._observations_out(), self.rew_buf, self.timeout_buf   # already on the host
        else:
            h_obs, h_rew, h_timeout = self._h_obs, self._h_rew, self._h_timeout
            h_obs.copy_(self._observations_out(), non_blocking=True)
            h_rew.copy_(self.rew_buf, non_blocking=True)
            h_timeout.copy_(self.timeout_buf, non_blocking=True)
        torch.cuda.current_stream(self.compute_device).synchronize()
        rl = torch.device(self.rl_device)
        if rl.type == "cpu":
            self.extras["time_outs"] = h_timeout
            self.obs_dict["obs"] = h_obs
            return self.obs_dict, h_rew, self._h_reset, self.extras
        self.extras["time_outs"] = self.timeout_buf.to(rl)
        self.obs_dict["obs"] = self._observations_out().to(rl)
        return self.obs_dict, self.rew_buf.to(rl), self.reset_buf.to(rl), self.extras
