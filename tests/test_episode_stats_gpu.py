"""GPU: rl_games' episode statistics from the fused step (``bezk_post_physics_rollout_ep``) and the device meters
(``bezk_episode_meter_update``, ``learner.EpisodeMeter``) against the torch restatement in ``tests/rl_games_episode_oracle.py``,
and ``A2CAgent.train``'s best-checkpoint / stop rules."""
import os
import socket

import numpy as np
import pytest
import torch

from bez_isaacgym_b200 import bez_model as bm
from tests import rl_games_episode_oracle as eo

pytestmark = pytest.mark.gpu


def _mover(seed):
    """on_simulate: a seeded random walk of the whole state, so rewards vary and termination rules fire."""
    g = torch.Generator(device="cuda").manual_seed(seed)

    def move(sim):
        for t, s in ((sim.root_states, 0.02), (sim.rigid_body, 0.05), (sim.dof_state, 0.05), (sim.net_contact, 0.5)):
            t.add_(torch.randn(t.shape, generator=g, device=t.device) * s)
    return move


def _env(task, n, cleats=False, seed=3, hook=None):
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
    env = cls(cfg, "cuda:0", 0, True, sim=sim)
    m = env.max_episode_length
    env.progress_buf.copy_(torch.randint(int(m) - 70, int(m), (n,), generator=torch.Generator().manual_seed(seed)).cuda())
    return env


def _run(env, steps, armed=True, actions_seed=5, rollout=False):
    """Steps the env with the episode targets armed; returns (per-step rew, reset, partials) and the final accumulators."""
    n = env.num_envs
    w = (n + 31) // 32
    ret, length = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    part = torch.full((steps, 3, w), float("nan"), dtype=torch.float64, device="cuda")       # every slot must be written
    g = torch.Generator(device="cuda").manual_seed(actions_seed)
    log = []
    extra = {}
    for t in range(steps):
        if rollout:
            extra = dict(values=torch.randn(n, device="cuda", generator=g), shaped_rewards=torch.empty(n, device="cuda"),
                         dones_u8=torch.empty(n, dtype=torch.uint8, device="cuda"))
        ep = dict(episode_returns=ret, episode_lengths=length, episode_partials=part[t]) if armed else {}
        env.set_rollout_targets(**extra, **ep)
        env.step(torch.rand(n, 18, device="cuda", generator=g) * 2 - 1)
        rec = dict(rew=env.rew_buf.clone(), reset=env.reset_buf.clone())
        if rollout:
            rec.update(obs=env.obs_buf.clone(), progress=env.progress_buf.clone(), timeout=env.timeout_buf.clone(),
                       dof=env.dof_state.clone(), root=env.root_states.clone(), shaped=extra["shaped_rewards"], dones=extra["dones_u8"])
        log.append(rec)
    env.set_rollout_targets()
    torch.cuda.synchronize()
    return log, part, ret, length


def _check_accumulators(log, part, ret, length):
    n = ret.numel()
    w = (n + 31) // 32
    r_ref, l_ref = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    fired = 0
    for t, rec in enumerate(log):
        r, l = r_ref + rec["rew"], l_ref + 1.0
        done = rec["reset"] != 0
        fired += int(done.sum())
        pad = w * 32 - n
        dz = torch.nn.functional.pad(done.double(), (0, pad)).view(w, 32)
        rz = torch.nn.functional.pad(torch.where(done, r, torch.zeros_like(r)).double(), (0, pad)).view(w, 32)
        lz = torch.nn.functional.pad(torch.where(done, l, torch.zeros_like(l)).double(), (0, pad)).view(w, 32)
        assert torch.equal(part[t, 0], dz.sum(1)), f"step {t}: done counts"
        assert torch.allclose(part[t, 1], rz.sum(1), rtol=1e-12, atol=0, equal_nan=True), f"step {t}: return sums"
        assert torch.equal(part[t, 2], lz.sum(1)), f"step {t}: length sums"
        not_done = 1.0 - done.float()
        r_ref, l_ref = r * not_done, l * not_done
    assert _same(ret, r_ref) and _same(length, l_ref), "accumulators"
    return fired


def _same(a, b):
    """Bitwise equality of float tensors, NaN == NaN."""
    return bool(((a == b) | (torch.isnan(a) & torch.isnan(b))).all())


@pytest.mark.parametrize("task,n,cleats", [("kick", 4096, False), ("kick", 4096, True), ("walk", 4096, False), ("orient", 4096, False),
                                           ("kick", 4099, False)])
def test_accumulators_and_partials_are_bit_exact(task, n, cleats):
    env = _env(task, n, cleats)
    log, part, ret, length = _run(env, 64)
    fired = _check_accumulators(log, part, ret, length)
    assert fired > 0
    timeouts_seen = any(bool((rec["reset"] != 0).any()) for rec in log)
    assert timeouts_seen


def test_large_kick_runs_the_l2_ep_kernel_when_the_policy_picks_it():
    from torch.profiler import ProfilerActivity, profile
    n = 262144
    env = _env("kick", n)
    l2 = torch.cuda.get_device_properties(0).L2_cache_size
    # the carried set of set_l2_policy, with the two accumulators: obs rows (+ the clipped copy), reset / progress / time-out, rew,
    # prev_lin_vel, goal, ball_init, episode return and length
    per_env = 54 * 4 * (1 + (env.obs_clipped_buf is not None)) + 3 * 8 + 4 + (0 if env._prev_is_view else 12) + 8 + 8 + 8
    expect_l2 = n * per_env <= l2 * 75 // 100 and n * (per_env + (36 + 26) * 4 + 3 * 64) > l2
    if "B200" in torch.cuda.get_device_name(0):
        assert expect_l2, "262 144 envs take the L2-hinted step on B200"
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        log, part, ret, length = _run(env, 2)
    names = [e.name for e in prof.events() if "task_tile" in e.name]
    want = "task_tile_ep_l2_kernel" if expect_l2 else "task_tile_ep_kernel"
    assert any(want in s for s in names), names
    assert not any("task_tile_kernel" in s or "task_tile_l2_kernel" in s for s in names), names
    env2 = _env("kick", n)
    log, part, ret, length = _run(env2, 64)
    assert _check_accumulators(log, part, ret, length) > 0


def test_nan_return_stays_nan_through_the_multiply():
    n, k = 4096, 256
    state = {"k": 0}

    def poison(sim):
        if state["k"] == 0:
            sim.root_states.view(n, -1)[:k, 2] = float("nan")         # envs 0..255: bez height NaN -> NaN rewards until reset
        state["k"] += 1
    env = _env("kick", n, hook=poison)
    log, part, ret, length = _run(env, 24)
    nan0 = torch.isnan(log[0]["rew"][:k])
    done_any = torch.stack([rec["reset"][:k] != 0 for rec in log]).any(0)
    first_done = torch.stack([rec["reset"][:k] != 0 for rec in log]).float().argmax(0)
    sel = (nan0 & done_any).nonzero().view(-1)
    assert sel.numel() > 0, "some NaN-reward env must finish inside the window"
    assert bool(torch.isnan(ret[sel]).all()), "NaN * (1 - done) stays NaN after the env is done"
    for e in sel[:8].tolist():
        assert torch.isnan(part[int(first_done[e]), 1, e // 32]), "the group's return sum is NaN in the step the env finished"
    _check_accumulators(log, part, ret, length)


def test_other_outputs_are_byte_identical_with_episode_targets_armed():
    n = 4096
    outs = []
    for armed in (False, True):
        env = _env("kick", n, seed=9)
        outs.append(_run(env, 24, armed=armed, rollout=True)[0])
    for t, (a, b) in enumerate(zip(*outs)):
        for k in a:
            x, y = a[k], b[k]
            same = (x == y) | (torch.isnan(x) & torch.isnan(y)) if x.is_floating_point() else (x == y)
            assert bool(same.all()), f"step {t}: {k}"


def _cpu_meter_from_partials(part, max_size):
    """The fold's recurrence on the CPU, fed the per-step (count, sum) read from the partials."""
    p = part.cpu().numpy()
    mr, ml = eo.AverageMeter(1, max_size), eo.AverageMeter(1, max_size)
    for t in range(p.shape[0]):
        cnt = float(p[t, 0].sum())
        if cnt == 0:
            continue
        mr.update_from_mean(torch.tensor([np.float32(p[t, 1].sum() / cnt)]), int(cnt))
        ml.update_from_mean(torch.tensor([np.float32(p[t, 2].sum() / cnt)]), int(cnt))
    return mr, ml


@pytest.mark.parametrize("n,max_size", [(4096, 100), (4099, 100), (4096, 7)])
def test_meters_match_the_restatements(n, max_size):
    from bez_isaacgym_b200 import ops
    env = _env("kick", n)
    log, part, ret, length = _run(env, 48)
    runs = []
    for _ in range(2):
        mean2 = torch.zeros(2, device="cuda")
        size2 = torch.zeros(2, dtype=torch.long, device="cuda")
        ops.episode_meter_update(part, n, max_size, mean2, size2)
        runs.append((mean2.cpu(), size2.cpu()))
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1]), "two folds, same bits"
    mean2, size2 = runs[0]
    mr, ml = _cpu_meter_from_partials(part, max_size)
    assert int(size2[0]) == int(size2[1]) == mr.current_size > 0
    assert torch.equal(mean2[0:1], mr.mean) and torch.equal(mean2[1:2], ml.mean), (mean2, mr.mean, ml.mean)
    # the pure rl_games restatement: torch mean over the done envs' values, every step
    gr, gl = eo.AverageMeter(1, max_size), eo.AverageMeter(1, max_size)
    cr, cl = torch.zeros(n, 1), torch.zeros(n)
    for rec in log:
        cr, cl = eo.episode_bookkeeping(cr, cl, rec["rew"].cpu(), rec["reset"].cpu(), gr, gl)
    assert gr.current_size == mr.current_size
    assert torch.allclose(mean2[0:1], gr.mean.view(1), rtol=1e-5) and torch.allclose(mean2[1:2], gl.mean.view(1), rtol=1e-5)
    # a fold split into two launches gives the same meters as one
    m2, s2 = torch.zeros(2, device="cuda"), torch.zeros(2, dtype=torch.long, device="cuda")
    ops.episode_meter_update(part[:20].contiguous(), n, max_size, m2, s2)
    ops.episode_meter_update(part[20:].contiguous(), n, max_size, m2, s2)
    assert torch.equal(m2.cpu(), mean2) and torch.equal(s2.cpu(), size2)


def test_episode_meter_interface():
    from bez_isaacgym_b200.learner import EpisodeMeter
    rew, lens = EpisodeMeter.pair(3, "cuda")
    part = torch.zeros(2, 3, 1, dtype=torch.float64, device="cuda")
    part[0, :, 0] = torch.tensor([2.0, 5.0, 30.0])
    part[1, :, 0] = torch.tensor([0.0, 0.0, 0.0])
    rew.update(part, 32)
    assert rew.current_size == lens.current_size == 2
    assert rew.get_mean().shape == (1,) and rew.get_mean()[0] == 2.5 and lens.get_mean()[0] == 15.0
    rew.clear()
    assert rew.current_size == 0 and lens.get_mean()[0] == 0.0


def _agent(n, T, **cfg):
    from bez_isaacgym_b200 import learner as L
    from bez_isaacgym_b200.synthetic_sim import SyntheticGym
    from bez_isaacgym_b200.tasks import KickEnv
    env = KickEnv(bm.default_task_cfg(n), "cuda:0", 0, True, sim=SyntheticGym(n, device="cuda:0", seed=2, on_simulate=_mover(4)))
    conf = dict(horizon_length=T, minibatch_size=n * T, mixed_precision=False)
    conf.update(cfg)
    agent = L.A2CAgent(env, conf, seed=1)
    env.progress_buf.copy_(torch.randint(870, 900, (n,), generator=torch.Generator().manual_seed(0)).cuda())
    return agent


def test_agent_meters_follow_the_experience_buffer():
    n, T = 2048, 16
    agent = _agent(n, T, reward_shaper=dict(scale_value=1.0, shift_value=0.0), value_bootstrap=False)
    gr, gl = eo.AverageMeter(1, 100), eo.AverageMeter(1, 100)
    cr, cl = torch.zeros(n, 1), torch.zeros(n)
    for _ in range(2):
        agent.train_epoch()
        rewards, dones = agent.mb_rewards.cpu(), agent.experience_buffer.tensor_dict["dones"].cpu()
        for t in range(T):
            d = dones[t + 1] if t + 1 < T else agent.dones.cpu()
            cr, cl = eo.episode_bookkeeping(cr, cl, rewards[t].view(-1), d, gr, gl)
    assert gr.current_size > 0 and agent.game_rewards.current_size == gr.current_size
    assert torch.equal(agent.current_rewards.cpu(), cr.view(-1)) and torch.equal(agent.current_lengths.cpu(), cl)
    assert np.allclose(agent.game_rewards.get_mean(), gr.get_mean(), rtol=1e-5)
    assert np.allclose(agent.game_lengths.get_mean(), gl.get_mean(), rtol=1e-5)


def test_train_saves_the_best_checkpoint_and_stops(tmp_path):
    n, T = 2048, 8
    agent = _agent(n, T, save_best_after=2, max_epochs=1, name="Kick")
    (last, epoch), hist = agent.train(str(tmp_path / "a"))
    assert epoch == 1 and len(hist) == 1 and last == -100500.0
    assert not (tmp_path / "a" / "Kick.pth").exists(), "epoch < save_best_after: no best checkpoint"

    agent = _agent(n, T, save_best_after=2, max_epochs=4, name="Kick")
    (last, epoch), hist = agent.train(str(tmp_path / "b"))
    assert epoch == 4 and [h["epoch"] for h in hist] == [1, 2, 3, 4]
    best = -100500.0
    for h in hist:
        if h["epoch"] >= 2 and h["mean_reward"] is not None and h["mean_reward"] > best:
            best = h["mean_reward"]
    assert last == best > -100500.0
    ck = torch.load(str(tmp_path / "b" / "Kick.pth"), weights_only=False)
    assert ck["last_mean_rewards"] == best and ck["epoch"] >= 2
    fresh = _agent(n, T)
    fresh.set_full_state_weights(ck)
    assert fresh.last_mean_rewards == best and fresh.epoch_num == ck["epoch"]
    for k, v in ck["model"].items():
        assert torch.equal(fresh.model.state_dict()[k[len("a2c_network."):]].cpu(), v.cpu())

    agent = _agent(n, T, save_best_after=2, max_epochs=50, score_to_win=-1e9, name="Kick")
    (last, epoch), hist = agent.train(str(tmp_path / "c"))
    assert epoch == 2 and (tmp_path / "c" / "Kick.pth").exists(), "score_to_win stops at the first best save"


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _worker(rank, world, port, tmp):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    try:
        from bez_isaacgym_b200 import learner as L
        from bez_isaacgym_b200.synthetic_sim import SyntheticGym
        from bez_isaacgym_b200.tasks import KickEnv
        n, T = 1024, 8
        dev = f"cuda:{rank}"
        cfg = bm.default_task_cfg(n, rl_device=dev)
        env = KickEnv(cfg, dev, rank, True, sim=SyntheticGym(n, device=dev, seed=2 + rank))
        agent = L.A2CAgent(env, dict(horizon_length=T, minibatch_size=n * T, mixed_precision=False, save_best_after=1,
                                     max_epochs=3, score_to_win=-1e9 if rank == 0 else 1e9), seed=1)
        env.progress_buf.copy_(torch.randint(880, 900, (n,), generator=torch.Generator().manual_seed(rank)).to(dev))
        (_, epoch), _ = agent.train(os.path.join(tmp, f"rank{rank}"))
        with open(os.path.join(tmp, f"epoch{rank}"), "w") as f:
            f.write(str(epoch))
    finally:
        dist.destroy_process_group()


@pytest.mark.timeout(300)
def test_both_ranks_stop_on_the_same_epoch(tmp_path):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    mp.spawn(_worker, args=(2, _free_port(), str(tmp_path)), nprocs=2, join=True)
    epochs = [int((tmp_path / f"epoch{r}").read_text()) for r in range(2)]
    assert epochs[0] == epochs[1]
    assert not (tmp_path / "rank1").exists(), "only rank 0 saves"
