"""``PpoPlayerContinuous`` -- rl_games' continuous-PPO player (rl_games/algos_torch/players.py ``PpoPlayerContinuous`` and
rl_games/common/player.py ``BasePlayer.run``, v1.1.x, RECALLED; the reference's fork is ``utils/player.py`` / ``utils/players.py``,
run by ``train.py`` with ``test=True``): score a checkpoint on the fused step.

One player step is three launches and no host synchronisation:

    policy MLP (torch) on ``obs_norm``  ->  PD targets (``bezk_pre_physics`` on mu, or the ``policy_head`` kernel when sampling)
    ->  simulate  ->  fused step with the episode accumulators and the eval-mode observation normaliser in its epilogue
        (``bezk_post_physics_rollout_ep_norm``: writes the next ``obs_norm``)

rl_games' per-step tally (``done.nonzero()``, ``cr[done].sum().item()``, ``steps[done].sum().item()``) is one fold launch
(``bezk_player_tally_update``) and one host read every ``sync_every`` steps; the fold stops adding at the step that reaches
``games_num * n_game_life`` games, so the result does not depend on ``sync_every``.  With ``track_outcomes`` the step also counts
how each episode ended (the env's ``OUTCOMES``), and a second fold with the same cutoff (``bezk_player_outcome_update``) joins the
same host read.  With ``track_reward_terms`` the step also carries each episode's return per reward term (the env's
``REWARD_TERMS``), and a third fold with the same cutoff (``bezk_player_game_terms_update``) joins that read too.  With observation
domain randomisation the
noise lands after the step kernel, so the player then normalises the noisy rows with ``RunningMeanStd`` (eval mode) instead.
"""
import math

import torch

from .. import _lib, ops
from ..utils.config import PLAYER_DEFAULTS
from .agent import A2CNetwork
from .running_mean_std import RunningMeanStd

#: rl_games ``BasePlayer.max_steps`` (RECALLED): steps of one ``env_reset()`` before ``run()`` restarts from a reset
MAX_STEPS = 108000 // 4


class PpoPlayerContinuous:
    def __init__(self, env, config=None, seed=0, sync_every=32, track_outcomes=False, track_reward_terms=False):
        """``config``: ``PLAYER_DEFAULTS`` keys (``utils.config.player_config``; the older spelling ``determenistic`` is accepted)
        and ``normalize_input`` (default True, as ``learner.A2CAgent``).  ``seed``: Philox key of the sampled actions.
        ``sync_every``: env steps per tally fold and host read.  ``track_outcomes``: also count the games per outcome class
        (``run()`` then returns ``outcomes`` / ``outcome_rates`` and prints an ``outcomes:`` line).  ``track_reward_terms``: also
        sum the games' returns per reward term (``run()`` then returns ``reward_terms`` and prints a ``reward terms:`` line)."""
        config = dict(config or {})
        if "determenistic" in config:
            config.setdefault("deterministic", config.pop("determenistic"))
        cfg = dict(PLAYER_DEFAULTS, normalize_input=True, max_steps=MAX_STEPS)
        cfg.update(config)
        if int(sync_every) < 1:
            raise ValueError("sync_every must be >= 1")
        if getattr(env, "host_staged", False):
            raise NotImplementedError("PpoPlayerContinuous needs the GPU pipeline (the episode accumulators live on the device)")
        self.config, self.env = cfg, env
        self.device = env.compute_device
        self.games_num, self.n_game_life = int(cfg["games_num"]), int(cfg["n_game_life"])
        self.is_determenistic, self.print_stats = bool(cfg["deterministic"]), bool(cfg["print_stats"])
        self.normalize_input, self.max_steps = bool(cfg["normalize_input"]), int(cfg["max_steps"])
        self.sync_every, self.seed = int(sync_every), int(seed)
        self._head_step = 0
        self.model = A2CNetwork(env.num_obs, env.num_acts).to(self.device).eval()
        self.running_mean_std = RunningMeanStd(env.num_obs).to(self.device).eval()
        n, w = env.num_envs, (env.num_envs + 31) // 32
        f32, f64 = dict(dtype=torch.float32, device=self.device), dict(dtype=torch.float64, device=self.device)
        # rl_games' cr / steps, the per-step partials of one chunk, the fused normaliser's output, the tally and its per-step rows
        self.current_rewards, self.current_lengths = torch.zeros(n, **f32), torch.zeros(n, **f32)
        self._partials = torch.zeros(self.sync_every, 3, w, **f64)
        self.obs_norm = torch.zeros(n, env.num_obs, **f32)
        self._tally = torch.zeros(4, **f64)
        self._per_step = torch.zeros(self.sync_every, 3, **f64)
        self._env_actions = torch.zeros(n, env.num_acts, **f32)
        self._targets = torch.zeros(n, env.num_acts, **f32)        # K0 output when env.step recomputes the targets
        # track_outcomes: the outcome partials of one chunk and [games_counted, count per class]
        self.track_outcomes = bool(track_outcomes)
        if self.track_outcomes:
            self._oc_partials = torch.zeros(self.sync_every, len(env.OUTCOMES), w, dtype=torch.int32, device=self.device)
            self._oc_counts = torch.zeros(1 + len(env.OUTCOMES), **f64)
        # track_reward_terms: each env's per-term episode return, the game term partials of one chunk and [games_counted, sum per term]
        self.track_reward_terms = bool(track_reward_terms)
        if self.track_reward_terms:
            k = len(env.REWARD_TERMS)
            self.current_term_rewards = torch.zeros(k, n, **f32)
            self._gt_partials = torch.zeros(self.sync_every, k, w, **f64)
            self._gt_sums = torch.zeros(1 + k, **f64)

    # ------------------------------------------------------------------ checkpoints
    def restore(self, fn):
        """rl_games ``PpoPlayerContinuous.restore``: ``model`` (``a2c_network.*`` keys) and, with ``normalize_input``,
        ``running_mean_std``, both loaded strictly.  Takes ``A2CAgent.save`` files and rl_games checkpoints alike.  Like rl_games'
        ``torch_ext.load_checkpoint`` this unpickles the file: load only checkpoints you trust."""
        ckpt = torch.load(fn, map_location=self.device, weights_only=False)
        prefix = "a2c_network."
        self.model.load_state_dict({(k[len(prefix):] if k.startswith(prefix) else k): v for k, v in ckpt["model"].items()}, strict=True)
        if self.normalize_input:
            # copied into the existing buffers: the fused step reads them by address
            self.running_mean_std.load_state_dict(ckpt["running_mean_std"], strict=True)

    # ------------------------------------------------------------------ actions
    def _fused(self):
        return self.normalize_input and not self.env.dr_randomizations.get("observations", None)

    def _net_input(self, obs, fused):
        if fused:
            return self.obs_norm
        return self.running_mean_std(obs) if self.normalize_input else obs

    def _act(self, net_in, is_determenistic):
        """mu -> env actions ``rescale_actions(-1, 1, clamp(a, -1, 1))`` and, unless action noise is on (then ``env.step``
        recomputes them after the noise), the env's PD targets, in one launch."""
        env = self.env
        targets = self._targets if env.dr_randomizations.get("actions", None) else env.targets
        mu, _ = self.model(net_in)
        mu = mu.contiguous()
        if is_determenistic:
            # K0 with clip_actions = min(1, clip) is K0(rescale_actions(-1, 1, clamp(mu, -1, 1))) bit for bit: the * 1 + 0 of
            # rescale_actions only changes the sign of a zero, which the default joint angle added by K0 removes
            cfg = _lib.BezkTaskCfg.from_buffer_copy(env._kcfg)
            cfg.clip_actions = min(1.0, float(cfg.clip_actions))
            ops.pre_physics(mu, targets, cfg, actions_out=self._env_actions)
        else:
            ops.policy_head(mu, self.model.sigma.detach().contiguous(), seed=self.seed, step=self._head_step, task_cfg=env._kcfg,
                            env_actions=self._env_actions, targets=targets, env_base=env.env_base)
            self._head_step += 1
        return self._env_actions

    def get_action(self, obs, is_determenistic=False):
        """rl_games ``get_action``: the env actions for raw observations ``obs`` (normalised with ``running_mean_std`` in eval mode
        when ``normalize_input``); the env's PD targets are written by the same launch, as ``env.step_precomputed_targets``
        expects."""
        with torch.no_grad():
            return self._act(self.running_mean_std(obs) if self.normalize_input else obs, is_determenistic)

    # ------------------------------------------------------------------ the loop
    def _arm(self, t, fused):
        rms = self.running_mean_std
        extra = dict(obs_norm=self.obs_norm, obs_mean=rms.running_mean, obs_var=rms.running_var, obs_eps=rms.epsilon) if fused else {}
        if self.track_outcomes:
            extra["episode_outcomes"] = self._oc_partials[t]
        if self.track_reward_terms:
            extra.update(game_term_returns=self.current_term_rewards, game_term_partials=self._gt_partials[t])
        self.env.set_rollout_targets(episode_returns=self.current_rewards, episode_lengths=self.current_lengths,
                                     episode_partials=self._partials[t], **extra)

    def _env_step(self, actions):
        env = self.env
        if env.dr_randomizations.get("actions", None):
            return env.step(actions)[0]["obs"]
        return env.step_precomputed_targets(actions)[0]["obs"]

    def env_reset(self, fused=None):
        """``env.reset()`` with the targets armed, so that the reset step's ``obs_norm`` feeds the first action; then rl_games'
        fresh ``cr`` / ``steps`` (the reset step is not counted, and its partials are never folded)."""
        fused = self._fused() if fused is None else fused
        self._arm(0, fused)
        obs = self.env.reset()["obs"]
        self.current_rewards.zero_()
        self.current_lengths.zero_()
        if self.track_reward_terms:
            self.current_term_rewards.zero_()
        return obs

    def run(self):
        """rl_games ``BasePlayer.run``: play until ``games_num * n_game_life`` games have finished (the last step may overshoot),
        restarting from ``env_reset()`` every ``max_steps`` steps.  Prints rl_games' ``reward: ... steps: ...`` line for every
        step with finished games (``print_stats``) and the final ``av reward: ... av steps: ...``.  Returns dict(games_played,
        sum_rewards, sum_steps, av_reward, av_steps); with ``track_outcomes`` also ``outcomes`` (outcome name -> games) and
        ``outcome_rates`` (outcome name -> share of the games played), printed as one ``outcomes:`` line after ``av reward``; with
        ``track_reward_terms`` also ``reward_terms`` (term name -> the term's return per game, scaled like ``av_reward``, so the terms
        sum to it up to rounding), printed as one ``reward terms:`` line after those."""
        env, n = self.env, self.env.num_envs
        n_games = self.games_num * self.n_game_life
        tally = self._tally.zero_()
        if self.track_outcomes:
            self._oc_counts.zero_()
        if self.track_reward_terms:
            self._gt_sums.zero_()
        games_played = sum_rewards = sum_steps = 0.0
        oc_host = gt_host = None
        try:
            with torch.no_grad():
                for _ in range(n_games):
                    if games_played >= n_games:
                        break
                    fused = self._fused()
                    obs = self.env_reset(fused)
                    done_steps = 0
                    while done_steps < self.max_steps and games_played < n_games:
                        k = min(self.sync_every, self.max_steps - done_steps)
                        for t in range(k):
                            actions = self._act(self._net_input(obs, fused), self.is_determenistic)
                            self._arm(t, fused)
                            obs = self._env_step(actions)
                        done_steps += k
                        ops.player_tally_update(self._partials[:k], n, n_games, tally, self._per_step[:k], steps=k)
                        parts = [tally, self._per_step[:k].reshape(-1)]
                        if self.track_outcomes:
                            ops.player_outcome_update(self._oc_partials[:k], n, env.TASK, n_games, self._oc_counts, steps=k)
                            parts.append(self._oc_counts)
                        if self.track_reward_terms:
                            ops.player_game_terms_update(self._partials[:k], self._gt_partials[:k], n, env.TASK, n_games, self._gt_sums,
                                                         steps=k)
                            parts.append(self._gt_sums)
                        host = torch.cat(parts).cpu()      # the one host read of the chunk
                        games_played, sum_rewards, sum_steps = float(host[0]), float(host[1]), float(host[2])
                        if self.track_reward_terms:
                            gt_host = host[-self._gt_sums.numel():]
                            host = host[:-self._gt_sums.numel()]
                        if self.track_outcomes:
                            oc_host = host[4 + 3 * k:]
                            host = host[:4 + 3 * k]
                        if self.print_stats:
                            for cnt, r, s in host[4:].view(k, 3).tolist():
                                if cnt > 0:
                                    print("reward:", r / cnt, "steps:", s / cnt)
        finally:
            env.set_rollout_targets()
        av_reward = sum_rewards / games_played * self.n_game_life if games_played else math.nan
        av_steps = sum_steps / games_played * self.n_game_life if games_played else math.nan
        print(sum_rewards)
        print("av reward:", av_reward, "av steps:", av_steps)
        res = dict(games_played=games_played, sum_rewards=sum_rewards, sum_steps=sum_steps, av_reward=av_reward, av_steps=av_steps)
        if self.track_outcomes:
            counts = [0.0] * len(env.OUTCOMES) if oc_host is None else [float(x) for x in oc_host[1:]]
            res["outcomes"] = dict(zip(env.OUTCOMES, counts))
            res["outcome_rates"] = {name: (c / games_played if games_played else math.nan) for name, c in res["outcomes"].items()}
            print("outcomes:", " ".join(f"{name} {int(c)} ({100.0 * res['outcome_rates'][name]:.1f} %)"
                                        for name, c in res["outcomes"].items()))
        if self.track_reward_terms:
            sums = [0.0] * len(env.REWARD_TERMS) if gt_host is None else [float(x) for x in gt_host[1:]]
            res["reward_terms"] = {name: (s / games_played * self.n_game_life if games_played else math.nan)
                                   for name, s in zip(env.REWARD_TERMS, sums)}
            print("reward terms:", " ".join(f"{name} {v}" for name, v in res["reward_terms"].items()))
        return res
