"""GPU: the player path -- the fused step's eval-mode observation normaliser (``bezk_post_physics_rollout_ep_norm``) against
``bezk_rms_normalize``, the game tally fold (``bezk_player_tally_update``) against ``tests/rl_games_player_oracle.py``, and
``learner.PpoPlayerContinuous`` (actions, restore, ``run``)."""
import json
import os

import numpy as np
import pytest
import torch

from bez_isaacgym_b200 import bez_model as bm
from tests import rl_games_player_oracle as po

pytestmark = pytest.mark.gpu
FACTS = os.path.join(os.path.dirname(__file__), "golden", "checkpoint_facts.json")


def _mover(seed):
    g = torch.Generator(device="cuda").manual_seed(seed)

    def move(sim):
        for t, s in ((sim.root_states, 0.02), (sim.rigid_body, 0.05), (sim.dof_state, 0.05), (sim.net_contact, 0.5)):
            t.add_(torch.randn(t.shape, generator=g, device=t.device) * s)
    return move


def _env(task, n, cleats=False, seed=3, hook=None, clip=None, randomize=None):
    from bez_isaacgym_b200 import tasks
    from bez_isaacgym_b200.synthetic_sim import SyntheticGym
    cls = {"kick": tasks.KickEnv, "walk": tasks.WalkEnv, "orient": tasks.OrientEnv}[task]
    move = _mover(seed)

    def on_sim(sim):
        move(sim)
        if hook is not None:
            hook(sim)
    sim = SyntheticGym(n, device="cuda:0", cleats=cleats, seed=seed, on_simulate=on_sim, task=task)
    cfg = bm.default_task_cfg(n, cleats=cleats, task=task)
    cfg["seed"] = seed
    if clip is not None:
        cfg["env"]["clipObservations"] = clip
    if randomize is not None:
        cfg["task"] = {"randomize": True, "randomization_params": randomize}
    env = cls(cfg, "cuda:0", 0, True, sim=sim)
    m = env.max_episode_length
    env.progress_buf.copy_(torch.randint(int(m) - 70, int(m), (n,), generator=torch.Generator().manual_seed(seed)).cuda())
    return env


def _same(a, b):
    """Bitwise equality, NaN payloads included."""
    return a.shape == b.shape and torch.equal(a.contiguous().view(torch.uint8), b.contiguous().view(torch.uint8))


def _stats(width, kind, seed=0):
    if kind == "checkpoint":
        with open(FACTS) as f:
            facts = json.load(f)
        return (torch.tensor(facts["obs_running_mean"], dtype=torch.float64, device="cuda"),
                torch.tensor(facts["obs_running_var"], dtype=torch.float64, device="cuda"))
    g = torch.Generator().manual_seed(seed)
    mean = torch.randn(width, generator=g, dtype=torch.float64) * 2
    var = torch.rand(width, generator=g, dtype=torch.float64) * 3
    var[::7] = 0.0                                                # zero-variance columns: sqrt(eps)
    return mean.cuda(), var.cuda()


def _poison(n):
    """on_simulate hook: a few envs get NaN / +-inf dof positions and velocities (they appear in the observation row as they are)."""
    def hook(sim):
        k = min(n, 5)
        d = sim.dof_state.view(n, 18, 2)
        vals = torch.tensor([float("nan"), float("inf"), -float("inf"), float("nan"), 1e30], device="cuda")[:k]
        d[:k, 3, 0] = vals
        d[:k, 7, 1] = vals.flip(0)
    return hook


def _arm(env, ret, length, part, norm=None, stats=None, rollout=None):
    kw = dict(episode_returns=ret, episode_lengths=length, episode_partials=part)
    if norm is not None:
        kw.update(obs_norm=norm, obs_mean=stats[0], obs_var=stats[1], obs_eps=1e-5)
    env.set_rollout_targets(**(rollout or {}), **kw)


# ------------------------------------------------------------------ obs_norm exactness
def _check_norm_steps(env, stat_sets, steps=3, seed=5):
    from bez_isaacgym_b200 import ops
    n, w = env.num_envs, env.num_obs
    ret, length = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    part = torch.zeros(3, (n + 31) // 32, dtype=torch.float64, device="cuda")
    norm = torch.full((n, w), float("nan"), device="cuda")
    g = torch.Generator(device="cuda").manual_seed(seed)
    seen = dict(nan=False, inf_in=False, clamped=False)
    for t in range(steps):
        stats = stat_sets[t % len(stat_sets)]
        _arm(env, ret, length, part, norm, stats)
        env.step(torch.rand(n, 18, device="cuda", generator=g) * 2 - 1)
        x = env._observations_out()
        want = ops.rms_normalize(x.contiguous(), stats[0], stats[1], torch.empty_like(x), eps=1e-5)
        assert _same(norm, want), f"step {t}: obs_norm differs from bezk_rms_normalize"
        seen["nan"] |= bool(torch.isnan(norm).any())
        seen["inf_in"] |= bool(torch.isinf(x).any())
        seen["clamped"] |= bool((norm.abs() == 5.0).any())
    env.set_rollout_targets()
    return seen


@pytest.mark.parametrize("task", ["kick", "walk", "orient"])
@pytest.mark.parametrize("cleats", [False, True])
@pytest.mark.parametrize("n,clip", [(1, None), (31, 5.0), (4099, None), (4099, 0.7)])
def test_obs_norm_is_bit_exact(task, cleats, n, clip):
    env = _env(task, n, cleats, hook=_poison(n), clip=clip)
    sets = [_stats(env.num_obs, "random", 1), _stats(env.num_obs, "random", 2)]
    if task == "kick":
        sets.insert(0, _stats(54, "checkpoint"))
    seen = _check_norm_steps(env, sets)
    assert seen["nan"] and seen["clamped"], "NaN rows and the +-5 clamp are exercised"
    if clip is None and n > 1:
        assert seen["inf_in"], "rows with +-inf are exercised"


def test_obs_norm_is_bit_exact_on_the_l2_kernel():
    n = 262144
    for clip in (None, 5.0):
        env = _env("kick", n, hook=_poison(n), clip=clip)
        _check_norm_steps(env, [_stats(54, "checkpoint"), _stats(54, "random", 4)], steps=2)


# ------------------------------------------------------------------ other outputs unchanged
@pytest.mark.parametrize("task,n,clip", [("kick", 4099, None), ("kick", 4096, 5.0), ("walk", 4096, 5.0), ("orient", 4099, None)])
def test_other_outputs_are_the_same_bytes(task, n, clip):
    logs = []
    for armed in (False, True):
        env = _env(task, n, clip=clip)
        ret, length = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
        part = torch.zeros(24, 3, (n + 31) // 32, dtype=torch.float64, device="cuda")
        norm = torch.zeros(n, env.num_obs, device="cuda")
        stats = _stats(env.num_obs, "random", 3)
        g = torch.Generator(device="cuda").manual_seed(9)
        log = []
        for t in range(24):
            ro = dict(values=torch.randn(n, device="cuda", generator=g), shaped_rewards=torch.empty(n, device="cuda"),
                      dones_u8=torch.empty(n, dtype=torch.uint8, device="cuda"))
            _arm(env, ret, length, part[t], norm if armed else None, stats, ro)
            env.step(torch.rand(n, 18, device="cuda", generator=g) * 2 - 1)
            log.append([env.obs_buf.clone(), env._observations_out().clone(), env.rew_buf.clone(), env.reset_buf.clone(),
                        env.progress_buf.clone(), env.timeout_buf.clone(), env.dof_state.clone(), env.root_states.clone(),
                        ro["shaped_rewards"], ro["dones_u8"]])
        env.set_rollout_targets()
        log.append([ret, length, part])
        logs.append(log)
    for a, b in zip(*logs):
        for x, y in zip(a, b):
            assert _same(x, y)


# ------------------------------------------------------------------ L2 choice unchanged
@pytest.mark.parametrize("n", [65536, 262144])
def test_l2_choice_is_the_ep_kernels(n):
    from torch.profiler import ProfilerActivity, profile
    env = _env("kick", n)
    ret, length = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    part = torch.zeros(3, n // 32, dtype=torch.float64, device="cuda")
    norm = torch.zeros(n, 54, device="cuda")
    stats = _stats(54, "random", 5)
    names = {}
    for armed in (False, True):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            for _ in range(2):
                _arm(env, ret, length, part, norm if armed else None, stats)
                env.step(torch.zeros(n, 18, device="cuda"))
            torch.cuda.synchronize()
        names[armed] = {e.name for e in prof.events() if "task_tile" in e.name}
    env.set_rollout_targets()
    ep_l2 = any("task_tile_ep_l2_kernel" in s for s in names[False])
    assert any("task_tile_ep_" in s for s in names[False]) and not any("obsnorm" in s for s in names[False])
    want = "task_tile_obsnorm_l2_kernel" if ep_l2 else "task_tile_obsnorm_kernel"
    assert any(want in s for s in names[True]) and not any("task_tile_ep_" in s for s in names[True]), names
    if not ep_l2:
        assert not any("obsnorm_l2" in s for s in names[True])
    if "B200" in torch.cuda.get_device_name(0):
        assert ep_l2 == (n == 262144), "B200: the L2 kernel at 262 144 envs only"


# ------------------------------------------------------------------ tally
def _fold_on_device(p, games_num, chunk, n):
    from bez_isaacgym_b200 import ops
    steps = p.shape[0]
    tally = torch.zeros(4, dtype=torch.float64, device="cuda")
    per = torch.full((steps, 3), float("nan"), dtype=torch.float64, device="cuda")
    for t0 in range(0, steps, chunk):
        k = min(chunk, steps - t0)
        ops.player_tally_update(p[t0:t0 + k], n, games_num, tally, per[t0:t0 + k], steps=k)
    return tally.cpu().numpy(), per.cpu().numpy()


@pytest.mark.parametrize("n", [100, 4096, 262144])
def test_tally_is_bit_exact_against_the_sequential_restatement(n):
    w = (n + 31) // 32
    g = torch.Generator(device="cuda").manual_seed(n)
    steps = 45
    cnt = torch.randint(0, 4, (steps, w), device="cuda", generator=g).double()
    cnt[5] = 0.0                                                          # an empty step
    p = torch.stack([cnt, cnt * torch.randn(steps, w, device="cuda", generator=g, dtype=torch.float64) * 7.3,
                     cnt * torch.randint(1, 900, (steps, w), device="cuda", generator=g).double()], 1).contiguous()
    games_num = int(cnt[:30].sum()) - 1                                   # the cutoff falls inside step 29
    want, want_per = po.fold_partials(p.cpu().numpy(), games_num)
    for chunk in (1, 7, 45):
        tally, per = _fold_on_device(p, games_num, chunk, n)
        assert tally.tobytes() == want.tobytes() and per.tobytes() == want_per.tobytes(), chunk
    assert want[3] == 30 and want[0] >= games_num


def test_tally_of_real_partials_with_nan_returns():
    n = 4096
    state = {"k": 0}

    def poison(sim):
        if state["k"] == 0:
            sim.root_states.view(n, -1)[:64, 2] = float("nan")
        state["k"] += 1
    env = _env("kick", n, hook=poison)
    ret, length = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    part = torch.zeros(40, 3, n // 32, dtype=torch.float64, device="cuda")
    for t in range(40):
        _arm(env, ret, length, part[t])
        env.step(torch.zeros(n, 18, device="cuda"))
    env.set_rollout_targets()
    want, want_per = po.fold_partials(part.cpu().numpy(), 10 ** 9)
    tally, per = _fold_on_device(part, 10 ** 9, 8, n)
    assert tally.tobytes() == want.tobytes() and per.tobytes() == want_per.tobytes()
    assert np.isnan(tally[1]) and tally[0] > 0


# ------------------------------------------------------------------ the player
def _player(env, sync_every=32, seed=0, **config):
    from bez_isaacgym_b200.learner import PpoPlayerContinuous
    torch.manual_seed(11)                                                 # same network weights for every player of a test
    p = PpoPlayerContinuous(env, dict(dict(print_stats=False), **config), seed=seed, sync_every=sync_every)
    mean, var = _stats(env.num_obs, "random", 6)
    p.running_mean_std.running_mean.copy_(mean)
    p.running_mean_std.running_var.copy_(var.clamp_min(0.05))
    return p


class _FixedMu:
    """Stands in for the policy network: always the given mu (and log-std)."""

    def __init__(self, mu, sigma=None):
        self.mu, self.sigma = mu, (torch.zeros(18, device="cuda") if sigma is None else sigma)

    def __call__(self, x):
        return self.mu, None


def _record(env):
    """Log (rew, reset) of every step the player takes (the reset step goes through env.step and is not logged)."""
    log = []
    inner = env.step_precomputed_targets

    def step(env_actions=None):
        out = inner(env_actions)
        log.append((env.rew_buf.clone(), env.reset_buf.clone()))
        return out
    env.step_precomputed_targets = step
    return log


def test_run_matches_rl_games_and_prints_its_lines(capsys):
    n = 4096
    env = _env("kick", n)
    log = _record(env)
    p = _player(env, games_num=2000, print_stats=True)
    res = p.run()
    ref = po.RlGamesTally(n, 2000)
    for rew, reset in log:
        if not ref.step(rew.cpu(), reset.cpu()):
            break
    want = ref.result()
    assert res["games_played"] == want["games_played"] and res["sum_steps"] == want["sum_steps"]
    assert res["sum_rewards"] == pytest.approx(want["sum_rewards"], rel=1e-5)
    assert res["av_reward"] == pytest.approx(want["av_reward"], rel=1e-5) and res["av_steps"] == want["av_steps"]
    out = capsys.readouterr().out
    assert out.count("reward:") - 1 == len(ref.lines) and "av reward:" in out and "av steps:" in out


def test_run_does_not_depend_on_sync_every():
    results = []
    for sync in (1, 7, 32):
        env = _env("kick", 4096)
        results.append(_player(env, sync_every=sync, games_num=3000).run())
    assert results[0] == results[1] == results[2]
    assert results[0]["games_played"] >= 3000


def test_fused_run_equals_the_separate_normaliser():
    results = []
    for fused in (True, False):
        env = _env("kick", 4096, clip=5.0)
        p = _player(env, games_num=1500)
        if not fused:
            p._fused = lambda: False
        results.append(p.run())
    assert results[0] == results[1]


def test_a_chunk_needs_no_host_sync():
    from bez_isaacgym_b200 import ops
    env = _env("kick", 4096)
    p = _player(env, sync_every=8)
    obs = p.env_reset(True)
    torch.cuda.synchronize()
    torch.cuda.set_sync_debug_mode("error")
    try:
        for t in range(8):
            actions = p._act(p._net_input(obs, True), True)
            p._arm(t, True)
            obs = p._env_step(actions)
        ops.player_tally_update(p._partials, 4096, 10 ** 6, p._tally, p._per_step)
    finally:
        torch.cuda.set_sync_debug_mode(0)
        env.set_rollout_targets()
    assert float(p._tally[3]) == 8.0


def test_deterministic_targets_are_k0_of_the_rescaled_clamp():
    from bez_isaacgym_b200 import ops
    n = 4096
    env = _env("kick", n)
    p = _player(env)
    g = torch.Generator(device="cuda").manual_seed(1)
    mu = torch.randn(n, 18, device="cuda", generator=g) * 2
    mu[0, :6] = torch.tensor([float("nan"), float("inf"), -float("inf"), 0.0, -0.0, 1.0])
    mu[1, 2:10] = torch.tensor([-0.0, 0.0, -1.0, 1.0, -0.0, float("nan"), 0.999999, -1.000001])
    p.model = _FixedMu(mu)
    ea = p._act(p.obs_norm, True).clone()
    got = env.targets.clone()
    rescaled = torch.clamp(mu, -1.0, 1.0) * 1.0 + 0.0                  # rl_games rescale_actions(-1, 1, clamp(mu, -1, 1))
    want = ops.pre_physics(rescaled.contiguous(), torch.empty_like(got), env._kcfg)
    assert _same(got, want)
    head_zeroed = rescaled.clone()
    head_zeroed[:, 0:2] = 0.0
    assert bool(((ea == head_zeroed) | (ea.isnan() & head_zeroed.isnan())).all())


def test_stochastic_actions_are_the_policy_heads():
    from bez_isaacgym_b200 import ops
    n = 4096
    env = _env("kick", n)
    p = _player(env, seed=7, deterministic=False)
    mu = torch.randn(n, 18, device="cuda") * 0.5
    sigma = torch.randn(18, device="cuda") * 0.3
    p.model = _FixedMu(mu, sigma)
    for step in range(2):
        ea = p._act(p.obs_norm, False).clone()
        tg = env.targets.clone()
        want_ea, want_tg = torch.empty_like(ea), torch.empty_like(tg)
        ops.policy_head(mu, sigma, seed=7, step=step,
                        actions=torch.empty_like(mu), neglogp=torch.empty(n, device="cuda"), task_cfg=env._kcfg, env_actions=want_ea,
                        targets=want_tg, env_base=env.env_base)
        assert _same(ea, want_ea) and _same(tg, want_tg)


def test_restore_round_trip_and_rl_games_layout(tmp_path):
    from bez_isaacgym_b200.learner import A2CAgent
    env = _env("kick", 1024)
    agent = A2CAgent(env, dict(horizon_length=8, minibatch_size=2048))
    agent.running_mean_std.running_mean.normal_()
    agent.running_mean_std.running_var.uniform_(0.5, 2.0)
    agent.save(str(tmp_path / "ck"))
    p = _player(env)
    p.restore(str(tmp_path / "ck.pth"))
    for (k, a), (k2, b) in zip(agent.model.state_dict().items(), p.model.state_dict().items()):
        assert k == k2 and torch.equal(a, b)
    assert torch.equal(p.running_mean_std.running_var, agent.running_mean_std.running_var)
    # an rl_games checkpoint: the shipped file's key names and shapes
    with open(FACTS) as f:
        facts = json.load(f)
    model = {k: torch.randn(*s) for k, s in facts["model_shapes"].items()}
    rms = dict(running_mean=torch.tensor(facts["obs_running_mean"], dtype=torch.float64),
               running_var=torch.tensor(facts["obs_running_var"], dtype=torch.float64),
               count=torch.tensor(facts["obs_count"], dtype=torch.float64))
    ck = dict(model=model, running_mean_std=rms, reward_mean_std=dict(rms), epoch=facts["epoch"], frame=facts["frame"])
    torch.save(ck, str(tmp_path / "rl.pth"))
    mean_ptr = p.running_mean_std.running_mean.data_ptr()
    p.restore(str(tmp_path / "rl.pth"))
    assert p.running_mean_std.running_mean.data_ptr() == mean_ptr, "the statistics stay where the fused step reads them"
    assert torch.equal(p.model.mu.weight.cpu(), model["a2c_network.mu.weight"])
    assert torch.equal(p.running_mean_std.running_var.cpu(), rms["running_var"])
    model["a2c_network.extra"] = torch.zeros(1)
    torch.save(ck, str(tmp_path / "bad.pth"))
    with pytest.raises(RuntimeError):
        p.restore(str(tmp_path / "bad.pth"))


@pytest.mark.parametrize("task", ["walk", "orient"])
def test_sibling_task_players(task):
    from bez_isaacgym_b200 import ops
    env = _env(task, 4096)
    log = _record(env)
    p = _player(env, games_num=1000)
    res = p.run()
    ref = po.RlGamesTally(4096, 1000)
    for rew, reset in log:
        if not ref.step(rew.cpu(), reset.cpu()):
            break
    assert res["games_played"] == ref.games_played and res["sum_steps"] == ref.sum_steps
    assert res["sum_rewards"] == pytest.approx(ref.sum_rewards, rel=1e-5)
    x = env._observations_out()
    rms = p.running_mean_std
    want = ops.rms_normalize(x.contiguous(), rms.running_mean, rms.running_var, torch.empty_like(x))
    assert env.num_obs == 52 and _same(p.obs_norm, want)


def test_obs_noise_falls_back_to_the_separate_normaliser():
    params = {"frequency": 1, "observations": {"range": [0, .002], "operation": "additive", "distribution": "gaussian"}}
    env = _env("kick", 4096, randomize=params)
    assert env.dr_randomizations.get("observations")
    p = _player(env, games_num=500)
    assert not p._fused()
    with pytest.raises(NotImplementedError):
        p._arm(0, True)
    res = p.run()
    assert res["games_played"] >= 500
    assert not bool(p.obs_norm.any()), "the fused output was never written"


def test_two_epoch_checkpoint_plays(tmp_path, capsys):
    from bez_isaacgym_b200.learner import A2CAgent
    env = _env("kick", 4096)
    agent = A2CAgent(env, dict(max_epochs=2, save_best_after=0, name="Bez_Kick"))
    agent.train(str(tmp_path))
    ck = tmp_path / "Bez_Kick.pth"
    assert ck.exists()
    env.close()
    env2 = _env("kick", 4096, seed=8)
    from bez_isaacgym_b200.learner import PpoPlayerContinuous
    p = PpoPlayerContinuous(env2, dict(games_num=100))
    p.restore(str(ck))
    res = p.run()
    assert res["games_played"] >= 100
    assert "av reward:" in capsys.readouterr().out
