"""``A2CAgent`` -- the rl_games continuous-PPO epoch (rl_games/common/a2c_common.py ``ContinuousA2CBase.train_epoch`` /
``play_steps`` / ``prepare_dataset``, rl_games/algos_torch/a2c_continuous.py ``A2CAgent.calc_gradients``, v1.1.3, driven by
``cfg/train/bez_kickPPO.yaml:45-79``) with every piece of the BezKick hot path on the libbezk kernels:

    play_steps      T x [ obs RMS (eval) -> policy MLP (torch) -> ``policy_head`` kernel (sample, neglogp, value un-norm,
                    experience slots, PD targets) -> simulate -> fused post-physics kernel writing the next ``obses`` slot ->
                    reward shaping ]  ->  GAE kernel
    prepare_dataset value RMS x2 (train), advantage moments + normalise; minibatches = slab views (no flattening pass)
    calc_gradients  obs RMS (train) on the slab view -> MLP -> fused PPO loss fwd+bwd -> MLP backward -> gradient all-reduce
                    -> clip -> Adam; adaptive-KL learning rate (``schedulers.AdaptiveScheduler``, legacy per-minibatch schedule)

The policy MLP GEMMs and Adam stay in torch.  One process per GPU; with a process group the normaliser / advantage moments are
SUM-all-reduced (exact merge) and the gradients averaged on one flat bucket.  ``get_full_state_weights`` /
``set_full_state_weights`` use rl_games' checkpoint keys (``model``, ``running_mean_std``, ``reward_mean_std``, ``optimizer``,
``epoch``, ``frame``, ``last_mean_rewards``), with the network's parameters under the ``a2c_network.*`` names of the reference's
shipped checkpoint (``results/Bez_Kick/Normal/Bez_Kick_33.pth``), so that checkpoint loads.
"""
import os

import torch
from torch import nn

from .. import dist as bdist
from . import a2c_common, experience, losses
from .episode_meter import EpisodeMeter, GameTermMeter, OutcomeMeter, RewardTerms
from .policy_head import policy_head as _policy_head
from .running_mean_std import RunningMeanStd


class A2CNetwork(nn.Module):
    """cfg/train/bez_kickPPO.yaml:10-32: MLP 54-400-200-100 (ELU), ``mu`` head (no activation), ``value`` head, fixed ``sigma``
    parameter (const_initializer 0).  Parameter names follow rl_games' ``A2CBuilder.Network`` (``actor_mlp.{0,2,4}``)."""

    def __init__(self, obs_dim=54, act_dim=18, units=(400, 200, 100)):
        super().__init__()
        layers, d = [], obs_dim
        for u in units:
            layers += [nn.Linear(d, u), nn.ELU()]
            d = u
        self.actor_mlp = nn.Sequential(*layers)
        self.mu = nn.Linear(d, act_dim)
        self.value = nn.Linear(d, 1)
        self.sigma = nn.Parameter(torch.zeros(act_dim))

    def forward(self, obs):
        h = self.actor_mlp(obs)
        return self.mu(h), self.value(h)


class AdaptiveScheduler:
    """rl_games/common/schedulers.py AdaptiveScheduler."""

    def __init__(self, kl_threshold=0.008, min_lr=1e-6, max_lr=1e-2):
        self.kl_threshold, self.min_lr, self.max_lr = kl_threshold, min_lr, max_lr

    def update(self, current_lr, entropy_coef, epoch, frames, kl_dist):
        lr = current_lr
        if kl_dist > 2.0 * self.kl_threshold:
            lr = max(current_lr / 1.5, self.min_lr)
        if kl_dist < 0.5 * self.kl_threshold:
            lr = min(current_lr * 1.5, self.max_lr)
        return lr, entropy_coef


DEFAULT_CONFIG = dict(gamma=0.99, tau=0.95, learning_rate=3e-4, lr_schedule="adaptive", kl_threshold=0.008, grad_norm=1.0,
                      truncate_grads=True, e_clip=0.2, horizon_length=32, minibatch_size=32768, mini_epochs=5, critic_coef=2.0,
                      clip_value=True, entropy_coef=0.0, bounds_loss_coef=0.001, normalize_input=True, normalize_value=True,
                      normalize_advantage=True, value_bootstrap=True, reward_shaper=dict(scale_value=0.01), mixed_precision=True,
                      bound_form="v1.1.3", cuda_graph=False)
#: rl_games A2CBase's training-loop settings (RECALLED defaults of v1.1.3): meters of the last ``games_to_track`` episodes, best
#: checkpoint ``<name>.pth`` once ``epoch >= save_best_after``, a ``last_`` checkpoint every ``save_frequency`` epochs (0: never),
#: stop when the best mean return exceeds ``score_to_win`` or after ``max_epochs`` epochs
TRAIN_DEFAULTS = dict(games_to_track=100, save_best_after=100, save_frequency=0, score_to_win=1e9, max_epochs=int(1e6),
                      name="Bez_Kick")
#: this project's own options (not rl_games settings): ``track_outcomes`` -- count how each episode ended (the env's ``OUTCOMES``)
#: in the step kernel, into the ``game_outcomes`` meter and an ``outcomes`` entry of each ``train()`` history row
OUTCOME_DEFAULTS = dict(track_outcomes=False)
#: this project's own option: ``track_reward_terms`` -- sum each of the env's ``REWARD_TERMS`` in the step kernel and add a
#: ``reward_terms`` entry (term name -> mean per env-step of the epoch's rollout) to each ``train()`` history row
REWARD_TERM_DEFAULTS = dict(track_reward_terms=False)
#: this project's own option: ``track_game_reward_terms`` -- carry each episode's return per term of the env's ``REWARD_TERMS`` in
#: the step kernel, into the ``game_reward_terms`` meter and a ``game_reward_terms`` entry (term name -> mean return per game) of
#: each ``train()`` history row
GAME_TERM_DEFAULTS = dict(track_game_reward_terms=False)


class A2CAgent:
    def __init__(self, env, config=None, process_group=None, seed=0, global_advantage_stats=True):
        """``process_group``: ONE convention for every exchange of the learner -- ``None`` means "all ranks" (the WORLD group)
        whenever ``torch.distributed`` is initialised with more than one rank, and single-process otherwise.  Gradients, the
        KL average, the start-up parameter broadcast, both ``RunningMeanStd`` moment merges and (with
        ``global_advantage_stats``) the advantage moments all use the same group, so a rank-0 checkpoint carries the
        statistics of every shard.  Pass ``env.env_base`` = the rank's shard offset (``cfg['env']['envBase']``) so that the
        reset / exploration noise is keyed by global env ids."""
        cfg = dict(DEFAULT_CONFIG, **TRAIN_DEFAULTS, **OUTCOME_DEFAULTS, **REWARD_TERM_DEFAULTS, **GAME_TERM_DEFAULTS)
        cfg.update(config or {})
        process_group = bdist.resolve_group(process_group)
        self.config, self.env, self.group = cfg, env, process_group
        self.device = env.compute_device
        self.num_actors, self.horizon_length = env.num_envs, int(cfg["horizon_length"])
        self.batch_size = self.num_actors * self.horizon_length
        self.minibatch_size = int(cfg["minibatch_size"])
        if self.batch_size % self.minibatch_size:
            raise ValueError("batch_size must be a multiple of minibatch_size")          # rl_games asserts the same
        self.mini_epochs_num = int(cfg["mini_epochs"])
        self.gamma, self.tau = cfg["gamma"], cfg["tau"]
        self.last_lr = float(cfg["learning_rate"])
        self.scheduler = AdaptiveScheduler(cfg["kl_threshold"]) if cfg["lr_schedule"] == "adaptive" else None
        torch.manual_seed(seed)
        self.model = A2CNetwork(env.num_obs, env.num_acts).to(self.device)
        bdist.broadcast_parameters(self.model, 0, process_group)
        # the learning rate lives on the device (a tensor the capturable Adam reads): the adaptive-KL schedule can then run inside
        # a CUDA graph with no host round trip per minibatch (``cuda_graph: True``); eager mode fills the same tensor
        self._lr_t = torch.tensor(self.last_lr, dtype=torch.float32, device=self.device)
        self.optimizer = torch.optim.Adam(self.model.parameters(), self._lr_t, eps=1e-08, weight_decay=0.0, capturable=True)
        self._learn_graph = None
        self._learn_last = None
        self._epochs_eager = 0
        self.running_mean_std = RunningMeanStd(env.num_obs, process_group=process_group).to(self.device)
        self.value_mean_std = RunningMeanStd(1, process_group=process_group).to(self.device)
        self.adv_group = process_group if global_advantage_stats else None
        self.loss_cfg = losses.PPOLossConfig(cfg["e_clip"], cfg["critic_coef"], cfg["entropy_coef"], cfg["bounds_loss_coef"], 1.1,
                                             cfg["clip_value"], cfg["bound_form"])
        self.experience_buffer = experience.ExperienceBuffer(
            dict(observation_space=env.observation_space, action_space=env.action_space),
            dict(num_actors=self.num_actors, horizon_length=self.horizon_length), self.device)
        T, N, f32 = self.horizon_length, self.num_actors, dict(dtype=torch.float32, device=self.device)
        self.mb_rewards = torch.empty(T, N, 1, **f32)
        self.mb_returns, self.mb_advs = torch.empty(T, N, 1, **f32), torch.empty(T, N, 1, **f32)
        self.advantages = torch.empty(T, N, **f32)
        self.values_norm, self.returns_norm = torch.empty(T, N, 1, **f32), torch.empty(T, N, 1, **f32)
        self._bucket = torch.empty(sum(p.numel() for p in self.model.parameters()), **f32)
        # rl_games 1.1.3 autocasts inside calc_gradients only; get_action_values (the rollout forward) runs in fp32, so the
        # stored neglogpacs / mus / values are fp32-exact.  Here autocast is bf16 (no GradScaler needed) -- a documented
        # deviation from rl_games' fp16 + GradScaler -- and likewise confined to calc_gradients.
        self._amp = dict(device_type="cuda", dtype=torch.bfloat16, enabled=bool(cfg["mixed_precision"]))
        self.frame = self.epoch_num = 0
        self._head_step = 0
        self._seed = seed
        self.last_mean_rewards = -100500.0
        # rl_games play_steps' episode statistics, carried by the step kernel: current_rewards / current_lengths per env, the
        # per-step done-env partials (count, return sum, length sum per 32 envs) and the game_rewards / game_lengths meters
        self.current_rewards = torch.zeros(N, **f32)
        self.current_lengths = torch.zeros(N, **f32)
        self._ep_partials = torch.zeros(T, 3, (N + 31) // 32, dtype=torch.float64, device=self.device)
        self.game_rewards, self.game_lengths = EpisodeMeter.pair(int(cfg["games_to_track"]), self.device)
        # track_outcomes: the per-step outcome partials (done envs per outcome class per 32 envs) and their meter
        self.track_outcomes = bool(cfg["track_outcomes"])
        if self.track_outcomes:
            self._oc_partials = torch.zeros(T, len(env.OUTCOMES), (N + 31) // 32, dtype=torch.int32, device=self.device)
            self.game_outcomes = OutcomeMeter(env.OUTCOMES, int(cfg["games_to_track"]), self.device)
        # track_reward_terms: the per-step reward term partials (term sums per 32 envs) and their per-rollout means
        self.track_reward_terms = bool(cfg["track_reward_terms"])
        if self.track_reward_terms:
            self._rt_partials = torch.zeros(T, len(env.REWARD_TERMS), (N + 31) // 32, dtype=torch.float64, device=self.device)
            self.reward_terms = RewardTerms(env.REWARD_TERMS, self.device)
        # track_game_reward_terms: each env's per-term episode return (carried across epochs like current_rewards), the per-step
        # sums of the done envs' per-term returns (per 32 envs) and their meter
        self.track_game_reward_terms = bool(cfg["track_game_reward_terms"])
        if self.track_game_reward_terms:
            k = len(env.REWARD_TERMS)
            self.current_term_rewards = torch.zeros(k, N, **f32)
            self._gt_partials = torch.zeros(T, k, (N + 31) // 32, dtype=torch.float64, device=self.device)
            self.game_reward_terms = GameTermMeter(env.REWARD_TERMS, int(cfg["games_to_track"]), self.device)
        self.obs = env.reset()["obs"].clone()
        self.dones = torch.zeros(N, dtype=torch.uint8, device=self.device)
        self.dataset = None

    # ------------------------------------------------------------------ rollout
    def set_eval(self):
        self.model.eval(); self.running_mean_std.eval(); self.value_mean_std.eval()

    def set_train(self):
        self.model.train(); self.running_mean_std.train(); self.value_mean_std.train()

    def _forward(self, obs_norm, autocast=False):
        if autocast:
            with torch.autocast(**self._amp):
                mu, value = self.model(obs_norm)
            return mu.float(), value.float()
        return self.model(obs_norm)

    def _norm_obs(self, obs):
        return self.running_mean_std(obs) if self.config["normalize_input"] else obs

    def play_steps(self):
        """a2c_common.py ``play_steps`` + ``discount_values``: returns the batch dict (time-major tensors, nothing flattened)."""
        env, buf, T = self.env, self.experience_buffer, self.horizon_length
        shaper = self.config["reward_shaper"]
        self.set_eval()
        buf.slot("obses", 0).copy_(self.obs)
        buf.slot("dones", 0).copy_(self.dones)
        with torch.no_grad():
            for t in range(T):
                mu, value = self._forward(self._norm_obs(buf.slot("obses", t)))
                # with action domain randomisation on, the noise precedes the PD targets (vec_task.py:314-317): the head then
                # leaves K0 to env.step
                head_targets = not env.dr_randomizations.get("actions", None)
                res = _policy_head(mu, self.model.sigma, value, self.value_mean_std if self.config["normalize_value"] else None,
                                     experience=buf, t=t, seed=self._seed, step=self._head_step, env=env if head_targets else None,
                                     env_base=env.env_base)
                self._head_step += 1
                env.set_obs_target(buf.slot("obses", t + 1) if t + 1 < T else self.obs)   # next slot written in place
                # reward shaping + value bootstrap + the uint8 dones of the NEXT slot ride in the step kernel's epilogue
                env.set_rollout_targets(values=res["values"], shaped_rewards=self.mb_rewards[t],
                                        dones_u8=buf.slot("dones", t + 1) if t + 1 < T else self.dones, gamma=self.gamma,
                                        scale_value=shaper.get("scale_value", 1.0), shift_value=shaper.get("shift_value", 0.0),
                                        value_bootstrap=self.config["value_bootstrap"], episode_returns=self.current_rewards,
                                        episode_lengths=self.current_lengths, episode_partials=self._ep_partials[t],
                                        episode_outcomes=self._oc_partials[t] if self.track_outcomes else None,
                                        reward_terms=self._rt_partials[t] if self.track_reward_terms else None,
                                        game_term_returns=self.current_term_rewards if self.track_game_reward_terms else None,
                                        game_term_partials=self._gt_partials[t] if self.track_game_reward_terms else None)
                if head_targets:
                    env.step_precomputed_targets(res["env_actions"])
                else:
                    env.step(res["env_actions"])
            env.set_rollout_targets()
            self.game_rewards.update(self._ep_partials, self.num_actors)      # both meters, the T steps in order
            if self.track_outcomes:
                self.game_outcomes.update(self._oc_partials, self.num_actors)
            if self.track_reward_terms:
                self.reward_terms.update(self._rt_partials, self.num_actors)
            if self.track_game_reward_terms:
                self.game_reward_terms.update(self._ep_partials, self._gt_partials, self.num_actors)
            _, last_v = self._forward(self._norm_obs(self.obs))
            last_values = self.value_mean_std(last_v, unnorm=True) if self.config["normalize_value"] else last_v
            a2c_common.discount_values(self.dones, last_values, buf.tensor_dict["dones"], buf.tensor_dict["values"], self.mb_rewards,
                                       self.gamma, self.tau, out_advs=self.mb_advs, out_returns=self.mb_returns)
        self.frame += self.batch_size
        return dict(returns=self.mb_returns, played_frames=self.batch_size)

    # ------------------------------------------------------------------ dataset
    def prepare_dataset(self, batch_dict):
        """a2c_common.py ``prepare_dataset``: advantages = returns - values (then normalised), values / returns through the
        value normaliser in TRAIN mode (two updates per epoch: the shipped checkpoint has count = 1 + 2*frame)."""
        values = self.experience_buffer.tensor_dict["values"]
        a2c_common.normalize_advantages(batch_dict["returns"], values, normalize=self.config["normalize_advantage"],
                                        process_group=self.adv_group, out=self.advantages.view(-1))
        if self.config["normalize_value"]:
            self.value_mean_std.train()
            self.value_mean_std(values, out=self.values_norm)
            self.value_mean_std(batch_dict["returns"], out=self.returns_norm)
            old_values, returns = self.values_norm, self.returns_norm
        else:
            old_values, returns = values, batch_dict["returns"]
        self.dataset = experience.SlabDataset(self.experience_buffer, self.minibatch_size,
                                              extra=dict(returns=returns, advantages=self.advantages, old_values=old_values))

    # ------------------------------------------------------------------ learner
    def _plan_obs_normaliser(self):
        """The epoch's mini_epochs x minibatches train-mode updates of the obs normaliser, planned: one moments pass per distinct
        minibatch (+ one all-reduce), one merge kernel (``RunningMeanStd.plan``); ``calc_gradients`` then normalises update ``u``."""
        if self.config["normalize_input"]:
            nmb = len(self.dataset)
            self._obs_views = [self.dataset[i]["obses"] for i in range(nmb)]
            self.running_mean_std.plan(self._obs_views, list(range(nmb)) * self.mini_epochs_num)

    def calc_gradients(self, input_dict, update=None):
        """a2c_continuous.py ``calc_gradients`` on one minibatch (slab views).  ``update``: index of this call in the planned
        sequence of obs-normaliser updates (None: the per-minibatch train forward)."""
        if not self.config["normalize_input"]:
            obs = input_dict["obses"]
        elif update is None:
            obs = self.running_mean_std(input_dict["obses"])
        else:
            nmb = len(self.dataset)
            if update % nmb == 0:        # ONE normalise launch per mini-epoch: every minibatch with the statistics of ITS update
                self._obs_norm = self.running_mean_std.planned_group(update, self._obs_views, out=getattr(self, "_obs_norm", None))
            obs = self._obs_norm[update % nmb]
        obs = obs.reshape(-1, obs.shape[-1]).contiguous()        # (T*E, obs): a single-minibatch epoch hands over (T, N, obs)
        mu, value = self._forward(obs, autocast=True)
        loss, info = losses.ppo_loss(mu, value, self.model.sigma, input_dict["actions"], input_dict["mus"], input_dict["sigmas"],
                                     input_dict["old_values"], input_dict["returns"], input_dict["neglogpacs"],
                                     input_dict["advantages"], self.loss_cfg)
        self.optimizer.zero_grad(set_to_none=False)
        loss.backward()
        bdist.allreduce_grads_(list(self.model.parameters()), self.group, True, self._bucket)
        if self.config["truncate_grads"]:
            nn.utils.clip_grad_norm_(self.model.parameters(), self.config["grad_norm"])
        self.optimizer.step()
        return info

    def update_lr(self, lr):
        self.last_lr = float(lr)
        self._lr_t.fill_(self.last_lr)

    def _mean_kl(self, kl):
        """rl_games averages the KL over ranks before the adaptive schedule (HorovodWrapper.average_value)."""
        kl = kl.clone()
        if bdist.is_distributed(self.group):
            torch.distributed.all_reduce(kl, group=self.group)
            kl /= torch.distributed.get_world_size(self.group)
        return kl

    def _learn_eager(self):
        last = None
        self._plan_obs_normaliser()
        for me in range(self.mini_epochs_num):
            for i in range(len(self.dataset)):
                last = self.calc_gradients(self.dataset[i], me * len(self.dataset) + i)
                if self.scheduler is not None:
                    kl = self._mean_kl(last["kl"])
                    lr, _ = self.scheduler.update(self.last_lr, self.config["entropy_coef"], self.epoch_num, 0, float(kl))
                    self.update_lr(lr)
        return last

    def _learn_device_schedule(self):
        """The same loop with the adaptive-KL schedule evaluated ON THE DEVICE (schedulers.AdaptiveScheduler.update as two
        ``torch.where``): no host synchronisation, so the whole learner phase can be captured into one CUDA graph."""
        last = None
        sch = self.scheduler
        self._plan_obs_normaliser()
        for me in range(self.mini_epochs_num):
            for i in range(len(self.dataset)):
                last = self.calc_gradients(self.dataset[i], me * len(self.dataset) + i)
                if sch is not None:
                    kl = self._mean_kl(last["kl"]).float()
                    lr = self._lr_t
                    down = torch.clamp(lr / 1.5, min=sch.min_lr)
                    up = torch.clamp(lr * 1.5, max=sch.max_lr)
                    self._lr_t.copy_(torch.where(kl > 2.0 * sch.kl_threshold, down, torch.where(kl < 0.5 * sch.kl_threshold, up, lr)))
        return last

    def _learn_graphed(self):
        """mini_epochs x minibatches of ``calc_gradients`` (obs RunningMeanStd, MLP forward / backward, fused PPO loss, gradient
        all-reduce, clip, Adam, adaptive LR) replayed as ONE CUDA graph.  Every input is a persistent buffer (the time-major
        rollout tensors, ``advantages``, ``values_norm`` / ``returns_norm``), so the graph captured on the second epoch stays valid."""
        if self._learn_graph is None:
            if self._epochs_eager < 1:                      # first epoch eagerly: allocator / workspaces / Adam state warm-up
                self._epochs_eager += 1
                last = self._learn_device_schedule()
                self.last_lr = float(self._lr_t)
                return last
            g = torch.cuda.CUDAGraph()
            torch.cuda.synchronize(self.device)
            with torch.cuda.graph(g, capture_error_mode="thread_local"):
                self._learn_last = self._learn_device_schedule()
            self._learn_graph = g
        self._learn_graph.replay()
        self.last_lr = float(self._lr_t)                    # ONE host read per epoch (reporting only)
        return self._learn_last

    def train_epoch(self):
        """One epoch: play_steps -> prepare_dataset -> mini_epochs x minibatches of calc_gradients (+ adaptive LR on the KL,
        averaged over ranks).  Returns dict(a_loss, c_loss, kl, lr) as device scalars / floats."""
        batch = self.play_steps()
        self.set_train()
        self.prepare_dataset(batch)
        last = self._learn_graphed() if self.config["cuda_graph"] else self._learn_eager()
        self.epoch_num += 1
        return dict(a_loss=last["a_loss"], c_loss=last["c_loss"], kl=last["kl"], lr=self.last_lr)

    def train(self, directory):
        """rl_games ``A2CBase.train`` (RECALLED): ``train_epoch`` until a stop rule fires.  After each epoch with finished games
        (``game_rewards.current_size > 0``), rank 0 saves ``<directory>/<name>.pth`` when the mean return beats
        ``last_mean_rewards`` and ``epoch >= save_best_after`` (then stops if it exceeds ``score_to_win``), and
        ``last_<name>_ep_<epoch>.pth`` every ``save_frequency`` epochs; the loop stops after ``max_epochs`` epochs.  The meters
        are per rank, as in rl_games.  Deviation: rank 0 broadcasts its stop decision every epoch, so every rank leaves on the
        same epoch (in rl_games the other ranks would wait in the next epoch's collectives).  Returns ``(last_mean_rewards,
        epoch)`` and a per-epoch history (mean return / length or None before the first finished game, losses, lr; with
        ``track_outcomes`` also ``outcomes``: outcome name -> share of the tracked games, None before the first finished game; with
        ``track_reward_terms`` also ``reward_terms``: term name -> mean per env-step of the epoch's rollout, on this rank's envs;
        with ``track_game_reward_terms`` also ``game_reward_terms``: term name -> mean return per tracked game, None before the first
        finished game -- the terms sum to ``mean_reward`` up to fp32 rounding)."""
        cfg = self.config
        rank0 = not bdist.is_distributed(self.group) or torch.distributed.get_rank() == 0
        if rank0:
            os.makedirs(directory, exist_ok=True)
        history = []
        while True:
            info = self.train_epoch()
            epoch = self.epoch_num
            row = dict(epoch=epoch, mean_reward=None, mean_length=None, a_loss=float(info["a_loss"]), c_loss=float(info["c_loss"]),
                       kl=float(info["kl"]), lr=float(info["lr"]))
            if self.track_outcomes:
                row["outcomes"] = None
            if self.track_reward_terms:
                row["reward_terms"] = self.reward_terms.as_dict()
            if self.track_game_reward_terms:
                row["game_reward_terms"] = None
            should_exit = False
            if rank0:
                if self.game_rewards.current_size > 0:
                    mean_rewards = float(self.game_rewards.get_mean()[0])
                    row["mean_reward"], row["mean_length"] = mean_rewards, float(self.game_lengths.get_mean()[0])
                    if self.track_outcomes:
                        row["outcomes"] = self.game_outcomes.as_dict()
                    if self.track_game_reward_terms:
                        row["game_reward_terms"] = self.game_reward_terms.as_dict()
                    if cfg["save_frequency"] > 0 and epoch % cfg["save_frequency"] == 0 and mean_rewards <= self.last_mean_rewards:
                        self.save(os.path.join(directory, f"last_{cfg['name']}_ep_{epoch}"))
                    if mean_rewards > self.last_mean_rewards and epoch >= cfg["save_best_after"]:
                        self.last_mean_rewards = mean_rewards
                        self.save(os.path.join(directory, cfg["name"]))
                        if self.last_mean_rewards > cfg["score_to_win"]:
                            should_exit = True
                if epoch >= cfg["max_epochs"]:
                    should_exit = True
            history.append(row)
            if bdist.is_distributed(self.group):
                flag = torch.tensor([1.0 if should_exit else 0.0], device=self.device)
                torch.distributed.broadcast(flag, src=0, group=self.group)
                should_exit = bool(flag.item())
            if should_exit:
                return (self.last_mean_rewards, epoch), history

    def save(self, path):
        """rl_games ``torch_ext.save_checkpoint``: ``torch.save(get_full_state_weights(), path + '.pth')``."""
        torch.save(self.get_full_state_weights(), path + ".pth")

    # ------------------------------------------------------------------ checkpoints (rl_games keys)
    def get_full_state_weights(self):
        model = {"a2c_network." + k: v for k, v in self.model.state_dict().items()}
        return dict(model=model, running_mean_std=self.running_mean_std.state_dict(), reward_mean_std=self.value_mean_std.state_dict(),
                    optimizer=self.optimizer.state_dict(), epoch=self.epoch_num, frame=self.frame,
                    last_mean_rewards=self.last_mean_rewards)

    def set_full_state_weights(self, weights):
        self.model.load_state_dict({k[len("a2c_network."):]: v for k, v in weights["model"].items()})
        self.running_mean_std.load_state_dict(weights["running_mean_std"])
        self.value_mean_std.load_state_dict(weights["reward_mean_std"])
        if "optimizer" in weights:
            self.optimizer.load_state_dict(weights["optimizer"])
            for g in self.optimizer.param_groups:           # keep the learning rate on the device tensor the graph reads
                self.last_lr = float(g["lr"])
                g["lr"] = self._lr_t
            self._lr_t.fill_(self.last_lr)
            self._learn_graph = None
        self.epoch_num, self.frame = int(weights.get("epoch", 0)), int(weights.get("frame", 0))
        self.last_mean_rewards = weights.get("last_mean_rewards", self.last_mean_rewards)
