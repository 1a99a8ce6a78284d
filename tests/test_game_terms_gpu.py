"""GPU: the fused step's game term returns (``bezk_post_physics_rollout_ep_game_terms``) -- the carried per-term accumulators and
the per-warp sums of the done envs' per-term returns against the terms restated in fp32 torch (``tests/test_reward_terms_gpu.py``)
and summed in the step's shuffle-tree order, the three identities (termination is exact, the terms sum to the return, the counts
agree), byte identity of every other output, the L2 choice, both folds against ``tests/game_terms_oracle.py``, ``A2CAgent`` with
``track_game_reward_terms`` and the player with ``track_reward_terms``."""
import numpy as np
import pytest
import torch

from bez_isaacgym_b200 import bez_model as bm
from tests import game_terms_oracle as go
from tests.test_outcomes_gpu import _env, _mover
from tests.test_reward_terms_gpu import _restate

pytestmark = pytest.mark.gpu
EPS32 = float(np.finfo(np.float32).eps)


def _same_bits(got, want):
    """Bit for bit, except that a NaN only has to be a NaN (the device's and numpy's NaN payloads differ)."""
    got, want = np.asarray(got), np.asarray(want)
    nan = np.isnan(want)
    return got.shape == want.shape and np.array_equal(np.isnan(got), nan) and got[~nan].tobytes() == want[~nan].tobytes()


def _run(env, steps, game=True, outcomes=False, terms=False, norm=False, check=None, actions_seed=5):
    """``steps`` steps with the episode accumulators (and the chosen packs) armed; every partial buffer NaN / -1 poisoned, so each
    must come back fully written.  check(t, acc_before, acc_after, game_partials, ep_partials) runs after each step."""
    n = env.num_envs
    w, k = (n + 31) // 32, len(env.REWARD_TERMS)
    ret, length = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    acc = torch.zeros(k, n, device="cuda")
    part = torch.full((steps, 3, w), float("nan"), dtype=torch.float64, device="cuda")
    oc = torch.full((steps, len(env.OUTCOMES), w), -1, dtype=torch.int32, device="cuda")
    tm = torch.full((steps, k, w), float("nan"), dtype=torch.float64, device="cuda")
    gp = torch.full((steps, k, w), float("nan"), dtype=torch.float64, device="cuda")
    g = torch.Generator(device="cuda").manual_seed(actions_seed)
    gm = torch.Generator().manual_seed(6)
    mean = (torch.randn(env.num_obs, generator=gm, dtype=torch.float64) * 2).cuda()
    var = (torch.rand(env.num_obs, generator=gm, dtype=torch.float64) * 3 + 0.05).cuda()
    log = []
    for t in range(steps):
        extra = dict(values=torch.randn(n, device="cuda", generator=g), shaped_rewards=torch.empty(n, device="cuda"),
                     dones_u8=torch.empty(n, dtype=torch.uint8, device="cuda"))
        if norm:
            extra.update(obs_norm=torch.empty(n, env.num_obs, device="cuda"), obs_mean=mean, obs_var=var)
        if game:
            extra.update(game_term_returns=acc, game_term_partials=gp[t])
        env.set_rollout_targets(**extra, episode_returns=ret, episode_lengths=length, episode_partials=part[t],
                                episode_outcomes=oc[t] if outcomes else None, reward_terms=tm[t] if terms else None)
        before = acc.clone()
        env.step(torch.rand(n, 18, device="cuda", generator=g) * 2 - 1)
        rec = dict(rew=env.rew_buf.clone(), reset=env.reset_buf.clone(), progress=env.progress_buf.clone(), obs=env.obs_buf.clone(),
                   timeout=env.timeout_buf.clone(), ret=ret.clone(), len=length.clone(), shaped=extra["shaped_rewards"],
                   dones=extra["dones_u8"])
        if norm:
            rec["obs_norm"] = extra["obs_norm"]
        log.append(rec)
        if check is not None:
            check(t, before, acc, gp[t], part[t])
    env.set_rollout_targets()
    torch.cuda.synchronize()
    return log, part, oc, tm, gp, acc


def _check_step(env, before, after, got, ep, stats):
    """One step's accumulators and (K, W) partials against fp32 ``acc + term`` of the restated terms, the masked write-back and the
    fp64 tree sums over the done envs; the three identities."""
    n = env.num_envs
    w = (n + 31) // 32
    terms, fired, band, exact = _restate(env)
    done = env.reset_buf.cpu() != 0
    before, after, got, ep = before.cpu(), after.cpu(), got.cpu(), ep.cpu()
    rew = env.rew_buf.cpu()
    assert not torch.isnan(got).any() or torch.isnan(before).any(), "every slot written"
    assert torch.equal(before[-1], torch.zeros(n)), "a live env's termination accumulator is exactly 0"
    r = before + terms                                                   # fp32, the kernel's recurrence
    ok = ~band
    keep = ~torch.nn.functional.pad(band.int(), (0, w * 32 - n)).view(w, 32).any(1)
    # the device's r_k of a done env is its episode's return in term k: recover it from the partials only through the sums; the
    # write-back of every env (band envs excluded) is checked directly
    want_after = r * (1.0 - done.float())
    for k in range(terms.shape[0]):
        if exact[k]:
            assert torch.equal(after[k, ok].view(torch.int32), want_after[k, ok].view(torch.int32)), (env.REWARD_TERMS[k], k)
        else:
            assert torch.allclose(after[k, ok], want_after[k, ok], rtol=1e-5, atol=1e-5), env.REWARD_TERMS[k]
    want = torch.from_numpy(go.done_warp_sums(r.numpy(), done.numpy(), n))
    for k in range(terms.shape[0]):
        if exact[k]:
            assert torch.equal(got[k, keep].view(torch.int64), want[k, keep].view(torch.int64)), (env.REWARD_TERMS[k], k)
        else:
            assert torch.allclose(got[k, keep], want[k, keep], rtol=1e-5, atol=1e-5), env.REWARD_TERMS[k]
    # 1. termination is exact: a finished game's termination return is the reward of its last step
    assert torch.equal(torch.from_numpy(go.done_warp_sums(rew[None].numpy(), done.numpy(), n))[0], got[-1])
    # 2. the terms sum to the return ep_partials holds, up to the fp32 rounding of the two running sums: at most (steps + K) roundings
    # of each env's running sum of |term|
    absr = stats["abs"] + terms.abs().sum(0)
    mag = torch.from_numpy(go.done_warp_sums(absr[None].numpy(), done.numpy(), n))[0]
    assert bool(((got.sum(0) - ep[1]).abs() <= 2 * (stats["steps"] + 8) * EPS32 * mag + 1e-6)[keep].all()), "terms sum to the return"
    stats["abs"] = absr * (1.0 - done.float())
    # 3. every done env is a game of ep_partials
    assert float(ep[0].sum()) == float(done.sum())
    stats["warps"] += w
    stats["excluded"] += int((~keep).sum())
    stats["done"] += int(done.sum())


# (outcomes, terms, norm): the six packs the game term returns ride with; 262 144 envs run the L2 variants
PACKS = [(False, False, False), (True, False, False), (False, True, False), (True, True, False), (False, False, True), (True, False, True)]
CASES = ([("kick", 4096, False, p) for p in PACKS] +
         [("kick", 4096, True, PACKS[0]), ("kick", 4096, True, PACKS[3]), ("walk", 4096, False, PACKS[0]), ("walk", 4096, True, PACKS[3]),
          ("walk", 4096, True, PACKS[5]), ("orient", 4096, False, PACKS[2]), ("orient", 4096, True, PACKS[0]),
          ("orient", 4096, True, PACKS[4]), ("kick", 4099, False, PACKS[5]), ("kick", 4099, True, PACKS[2]),
          ("walk", 4099, False, PACKS[1]), ("orient", 4099, True, PACKS[3]), ("kick", 262144, False, PACKS[0]),
          ("kick", 262144, False, PACKS[5]), ("walk", 262144, True, PACKS[2]), ("orient", 262144, False, PACKS[3]),
          ("kick", 1, False, PACKS[0]), ("walk", 31, True, PACKS[3]), ("orient", 31, False, PACKS[4])])


@pytest.mark.parametrize("task,n,cleats,pack", CASES)
def test_accumulators_and_per_warp_sums_match_the_restatement(task, n, cleats, pack):
    outcomes, terms, norm = pack
    env = _env(task, n, cleats)
    steps = 8 if n > 100000 else (64 if n < 64 else 24)
    stats = dict(warps=0, excluded=0, done=0, steps=steps, abs=torch.zeros(n))
    _, part, oc, tm, gp, _ = _run(env, steps, outcomes=outcomes, terms=terms, norm=norm,
                                  check=lambda t, b, a, g, ep: _check_step(env, b, a, g, ep, stats))
    assert not torch.isnan(gp).any() and not torch.isnan(part).any()
    assert stats["excluded"] <= 0.02 * stats["warps"] + 1, stats
    if n >= 4096:
        assert stats["done"] > 0, stats
    if outcomes:
        assert torch.equal(oc.sum(1).double(), part[:, 0])
    if terms:
        assert not torch.isnan(tm).any()


def test_nothing_else_moves_and_game_terms_repeat():
    for outcomes, terms, norm in PACKS:
        a = _run(_env("kick", 4099), 40, game=False, outcomes=outcomes, terms=terms, norm=norm)
        b = _run(_env("kick", 4099), 40, game=True, outcomes=outcomes, terms=terms, norm=norm)
        c = _run(_env("kick", 4099), 40, game=True, outcomes=outcomes, terms=terms, norm=norm)
        for ra, rb in zip(a[0], b[0]):
            for key in ra:
                assert torch.equal(ra[key].contiguous().view(torch.uint8), rb[key].contiguous().view(torch.uint8)), key
        assert torch.equal(a[1].view(torch.uint8), b[1].view(torch.uint8)), "episode partials"
        assert torch.equal(a[2], b[2]), "outcome partials"
        assert torch.equal(a[3].view(torch.uint8), b[3].view(torch.uint8)), "term partials"
        assert torch.equal(b[4].view(torch.int64), c[4].view(torch.int64)), "game term partials repeat"
        assert torch.equal(b[5].view(torch.int32), c[5].view(torch.int32)), "accumulators repeat"
    for task in ("walk", "orient"):
        a = _run(_env(task, 4096, cleats=True), 16, game=False, outcomes=True, terms=True)
        b = _run(_env(task, 4096, cleats=True), 16, game=True, outcomes=True, terms=True)
        assert all(torch.equal(ra[k].contiguous().view(torch.uint8), rb[k].contiguous().view(torch.uint8))
                   for ra, rb in zip(a[0], b[0]) for k in ra)
        assert torch.equal(a[1].view(torch.uint8), b[1].view(torch.uint8)) and torch.equal(a[2], b[2])
        assert torch.equal(a[3].view(torch.uint8), b[3].view(torch.uint8))


def test_large_kick_with_game_terms_takes_the_l2_step():
    from torch.profiler import ProfilerActivity, profile
    n = 262144
    env = _env("kick", n)
    l2 = torch.cuda.get_device_properties(0).L2_cache_size
    # obs, reset / progress / timeout, rew, prev_lin_vel, goal, ball_init, episode return and length, and the K accumulators
    per_env = 54 * 4 * (1 + (env.obs_clipped_buf is not None)) + 3 * 8 + 4 + (0 if env._prev_is_view else 12) + 8 + 8 + 8 + 4 * 6
    expect_l2 = n * per_env <= l2 * 75 // 100 and n * (per_env + (36 + 26) * 4 + 3 * 64) > l2
    if "B200" in torch.cuda.get_device_name(0):
        assert expect_l2, per_env
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        _run(env, 2)
    names = [e.name for e in prof.events() if "task_tile" in e.name]
    want = "task_tile_game_l2_kernel" if expect_l2 else "task_tile_game_kernel"
    assert any(want in s for s in names), names
    assert not any("task_tile_ep_" in s for s in names), names


def test_folds_on_the_device_match_the_oracle():
    from bez_isaacgym_b200 import ops
    g = torch.Generator().manual_seed(2)
    for task, k, n in (("kick", 6, 5000), ("walk", 5, 262144), ("orient", 5, 33), ("kick", 6, 1)):
        w = (n + 31) // 32
        steps = 40
        cnt = (torch.rand(steps, w, generator=g) < 0.3) * torch.randint(1, 33, (steps, w), generator=g)
        cnt[5, 0] = 3                                                       # the NaN below belongs to a step with finished games
        ep = torch.zeros(steps, 3, w, dtype=torch.float64)
        ep[:, 0] = cnt.double()
        ep[:, 1] = torch.randn(steps, w, generator=g, dtype=torch.float64)
        tp = torch.randn(steps, k, w, generator=g, dtype=torch.float64) * 9 * (cnt > 0).unsqueeze(1)
        tp[5, 1, 0] = float("nan")
        epd, tpd = ep.cuda(), tp.cuda()
        mean = torch.full((k,), 0.25, device="cuda")
        size = torch.full((1,), 3, dtype=torch.long, device="cuda")
        ops.game_terms_meter_update(epd, tpd, n, task, 50, mean, size)
        wm, ws = go.meter(ep.numpy(), tp.numpy(), 50, np.full(k, 0.25, np.float32), 3)
        assert _same_bits(mean.cpu().numpy(), wm) and int(size) == ws, task
        assert np.isnan(wm[1]) and not np.isnan(np.delete(wm, 1)).any()
        games_num = max(1, int(cnt.sum()) // 2)
        sums = torch.zeros(1 + k, dtype=torch.float64, device="cuda")
        per = torch.full((steps, k), float("nan"), dtype=torch.float64, device="cuda")
        ops.player_game_terms_update(epd, tpd, n, task, games_num, sums, per)
        want, wper = go.player_fold(ep.numpy(), tp.numpy(), games_num)
        assert _same_bits(sums.cpu().numpy(), want) and _same_bits(per.cpu().numpy(), wper), task
        chunked = torch.zeros(1 + k, dtype=torch.float64, device="cuda")
        for a, b in ((0, 1), (1, 17), (17, 40)):
            ops.player_game_terms_update(epd[a:b], tpd[a:b], n, task, games_num, chunked)
        assert _same_bits(chunked.cpu().numpy(), want), "independent of chunking"
    # real partials: the meter's size follows the game meters', the player's games_counted the tally's games_played
    from bez_isaacgym_b200.learner import EpisodeMeter, GameTermMeter
    env = _env("kick", 8192)
    _, part, _, _, gp, _ = _run(env, 48)
    rewards, _ = EpisodeMeter.pair(100, "cuda")
    meter = GameTermMeter(env.REWARD_TERMS, 100, "cuda")
    rewards.update(part, 8192)
    meter.update(part, gp, 8192)
    wm, ws = go.meter(part.cpu().numpy(), gp.cpu().numpy(), 100)
    assert meter.current_size == rewards.current_size == ws > 0
    assert meter.get_mean().tobytes() == wm.tobytes()
    mag = float(np.abs(meter.get_mean()).sum())
    assert abs(float(meter.get_mean().astype(np.float64).sum()) - float(rewards.get_mean()[0])) <= 1e-4 * (1 + mag)
    tally = torch.zeros(4, dtype=torch.float64, device="cuda")
    sums = torch.zeros(7, dtype=torch.float64, device="cuda")
    ops.player_tally_update(part, 8192, 10 ** 9, tally)
    ops.player_game_terms_update(part, gp, 8192, "kick", 10 ** 9, sums)
    assert float(sums[0]) == float(tally[0]) > 0
    mag = float(torch.from_numpy(go.step_sums(part.cpu().numpy(), gp.cpu().abs().numpy())[:, 1:]).sum())
    assert abs(float(sums[1:].sum()) - float(tally[1])) <= 1e-4 * (1 + mag)


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


def test_agent_game_reward_terms_change_nothing_else(tmp_path):
    n, T = 2048, 16
    off = _agent(n, T)
    on = _agent(n, T, track_game_reward_terms=True)
    all3 = _agent(n, T, track_game_reward_terms=True, track_outcomes=True, track_reward_terms=True)
    assert not hasattr(off, "game_reward_terms") and not hasattr(off, "current_term_rewards")
    for _ in range(3):
        a, b, c = off.train_epoch(), on.train_epoch(), all3.train_epoch()
        for key in ("a_loss", "c_loss", "kl"):
            assert torch.equal(torch.as_tensor(a[key]), torch.as_tensor(b[key])), key
            assert torch.equal(torch.as_tensor(a[key]), torch.as_tensor(c[key])), key
        assert torch.equal(on._gt_partials, all3._gt_partials) and torch.equal(on.current_term_rewards, all3.current_term_rewards)
    for x in (on, all3):
        for pa, pb in zip(off.model.parameters(), x.model.parameters()):
            assert torch.equal(pa, pb)
        assert np.array_equal(off.game_rewards.get_mean(), x.game_rewards.get_mean())
        assert np.array_equal(off.game_lengths.get_mean(), x.game_lengths.get_mean())
        assert torch.equal(off.current_rewards, x.current_rewards)
        assert x.game_reward_terms.current_size == x.game_rewards.current_size > 0
    # the accumulators carry across epochs: with every env's episode running on, they sum to current_rewards
    s = on.current_term_rewards.double().sum(0)
    assert bool(((s - on.current_rewards.double()).abs() <= 1e-4 * (1 + on.current_term_rewards.double().abs().sum(0))).all())
    assert bool((on.current_term_rewards[-1] == 0).all()), "live envs carry no termination return"
    (_, _), hist = _agent(n, 8, track_game_reward_terms=True, track_outcomes=True, track_reward_terms=True, max_epochs=3,
                          name="K").train(str(tmp_path))
    assert len(hist) == 3 and all("game_reward_terms" in h and "outcomes" in h and "reward_terms" in h for h in hist)
    rows = [h for h in hist if h["mean_reward"] is not None]
    assert rows, "games finished"
    for h in rows:
        assert list(h["game_reward_terms"]) == list(off.env.REWARD_TERMS)
        tot = sum(h["game_reward_terms"].values())
        assert abs(tot - h["mean_reward"]) <= 1e-4 * (1 + sum(abs(v) for v in h["game_reward_terms"].values())), (tot, h["mean_reward"])
    assert all(h["game_reward_terms"] is None for h in hist if h["mean_reward"] is None)
    (_, _), hist = _agent(n, 8, max_epochs=1, name="K").train(str(tmp_path / "off"))
    assert "game_reward_terms" not in hist[0]


def _player(env, sync_every=32, **config):
    from bez_isaacgym_b200.learner import PpoPlayerContinuous
    torch.manual_seed(11)
    return PpoPlayerContinuous(env, dict(dict(print_stats=False), **config), sync_every=sync_every, track_outcomes=True,
                               track_reward_terms=True)


def test_player_reward_terms_sum_to_av_reward_for_any_sync_every(capsys):
    results = [_player(_env("kick", 4096), sync_every=sync, games_num=3000).run() for sync in (1, 7, 32)]
    assert results[0] == results[1] == results[2]
    r = results[0]
    assert list(r["reward_terms"]) == ["ball_velocity", "approach", "height", "body_velocity", "posture", "termination"]
    mag = sum(abs(v) for v in r["reward_terms"].values())
    assert abs(sum(r["reward_terms"].values()) - r["av_reward"]) <= 2e-4 * (1 + mag)
    out = capsys.readouterr().out
    assert out.count("reward terms: ball_velocity") == 3
    assert out.index("av reward:") < out.index("outcomes:") < out.index("reward terms:")
    from bez_isaacgym_b200.learner import PpoPlayerContinuous
    torch.manual_seed(11)
    plain = PpoPlayerContinuous(_env("kick", 4096), dict(print_stats=False, games_num=3000)).run()
    assert plain == {k: r[k] for k in plain}, "the other results do not move"
    assert "reward terms:" not in capsys.readouterr().out
    for task in ("walk", "orient"):
        w = _player(_env(task, 4096), games_num=500, n_game_life=2).run()
        mag = sum(abs(v) for v in w["reward_terms"].values())
        assert abs(sum(w["reward_terms"].values()) - w["av_reward"]) <= 2e-4 * (1 + mag) and len(w["reward_terms"]) == 5


def test_player_fused_and_separate_normaliser_agree():
    results = []
    for fused in (True, False):
        p = _player(_env("kick", 4096), games_num=1500)
        if not fused:
            p._fused = lambda: False
        results.append(p.run())
    assert results[0] == results[1]
    # observation noise: the player normalises the noisy rows itself, the step still carries the game term returns
    from tests.test_player_gpu import _env as _noisy_env
    params = {"frequency": 1, "observations": {"range": [0, .002], "operation": "additive", "distribution": "gaussian"}}
    env = _noisy_env("kick", 4096, randomize=params)
    assert env.dr_randomizations.get("observations")
    p = _player(env, games_num=500)
    assert not p._fused()
    res = p.run()
    mag = sum(abs(v) for v in res["reward_terms"].values())
    assert res["games_played"] >= 500 and abs(sum(res["reward_terms"].values()) - res["av_reward"]) <= 2e-4 * (1 + mag)
    assert sum(res["outcomes"].values()) == res["games_played"]


@pytest.mark.parametrize("task", ["kick", "walk", "orient"])
@pytest.mark.parametrize("norm", [False, True])
def test_ops_wrapper_routes_every_argument(task, norm):
    """``ops.post_physics_rollout_ep_game_terms`` on a synthetic state against ``ops.post_physics_rollout_ep`` / ``_ep_norm`` on a
    copy of it: every output the same bytes; from zeroed accumulators a done env's per-term returns are this step's terms, so the
    termination row of the partials is the tree sum of the done envs' rewards and the live envs keep their terms."""
    from bez_isaacgym_b200 import ops, synthetic_gym as sg
    n = 4099
    w = (n + 31) // 32
    k = {"kick": 6, "walk": 5, "orient": 5}[task]
    actors, nb, width = bm.task_dims(task)
    cfg = ops.make_task_cfg(num_bodies=nb)
    runs = []
    for with_game in (False, True):
        st = sg.make_state(n, seed=21, task=task).to("cuda")
        progress, reset = sg.make_bookkeeping(n, seed=22, device="cuda", p_reset=0.1)
        progress[:64] = 899
        t = dict(st=st, progress=progress, reset=reset, timeout=torch.empty(n, dtype=torch.long, device="cuda"),
                 obs=torch.empty(n, width, device="cuda"), rew=torch.empty(n, device="cuda"), prev=torch.zeros(n, 3, device="cuda"),
                 goal=torch.tensor([[1.5, 0.0]] if task == "kick" else [[2.0, 0.5]], device="cuda").repeat(n, 1),
                 shaped=torch.empty(n, device="cuda"), dones=torch.empty(n, dtype=torch.uint8, device="cuda"),
                 ret=torch.rand(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1)),
                 len=torch.full((n,), 7.0, device="cuda"), part=torch.full((3, w), float("nan"), dtype=torch.float64, device="cuda"),
                 obs_norm=torch.empty(n, width, device="cuda"), acc=torch.zeros(k, n, device="cuda"),
                 gp=torch.full((k, w), float("nan"), dtype=torch.float64, device="cuda"))
        mean = torch.linspace(-1, 1, width, dtype=torch.float64, device="cuda")
        var = torch.linspace(0.1, 2, width, dtype=torch.float64, device="cuda")
        args = (task, st.dof_state, st.rigid_body, st.root_states, st.net_contact, t["goal"], sg.make_initial_root_states(n, "cuda", task=task),
                reset, progress, t["timeout"], cfg, t["obs"], t["rew"])
        kw = dict(rollout_cfg=ops.make_rollout_cfg(), values=torch.ones(n, device="cuda"), shaped_rewards=t["shaped"], dones_u8=t["dones"],
                  goal_angle=torch.full((n,), 1.5708, device="cuda") if task == "orient" else None,
                  ball_init=torch.tensor([[0.175, 0.0]], device="cuda").repeat(n, 1) if task == "kick" else None,
                  prev_lin_vel=t["prev"], seed=5, step=3)
        normkw = dict(obs_mean=mean, obs_var=var, obs_norm=t["obs_norm"]) if norm else {}
        if with_game:
            ops.post_physics_rollout_ep_game_terms(*args, t["ret"], t["len"], t["part"], t["acc"], t["gp"], **normkw, **kw)
        elif norm:
            ops.post_physics_rollout_ep_norm(*args, t["ret"], t["len"], t["part"], mean, var, t["obs_norm"], **kw)
        else:
            ops.post_physics_rollout_ep(*args, t["ret"], t["len"], t["part"], **kw)
        torch.cuda.synchronize()
        runs.append(t)
    a, b = runs
    for key in ("progress", "reset", "timeout", "obs", "rew", "prev", "goal", "shaped", "dones", "ret", "len", "part") + (("obs_norm",) if norm else ()):
        assert torch.equal(a[key].contiguous().view(torch.uint8), b[key].contiguous().view(torch.uint8)), key
    for key in ("dof_state", "root_states"):
        assert torch.equal(getattr(a["st"], key), getattr(b["st"], key)), key
    done = (b["reset"] != 0).cpu()
    assert int(done.sum()) > 0 and not torch.isnan(b["gp"]).any()
    rew = b["rew"].cpu()
    assert torch.equal(b["gp"][-1].cpu(), torch.from_numpy(go.done_warp_sums(rew[None].numpy(), done.numpy(), n))[0])
    acc = b["acc"].cpu()
    assert bool((acc[:, done] == 0).all()) and bool((acc[-1] == 0).all())
    live = acc[:, ~done].double().sum(0)
    assert bool(((live - rew[~done].double()).abs() <= 8 * EPS32 * (1 + acc[:, ~done].double().abs().sum(0))).all())
    assert float(b["part"][0].sum()) == float(done.sum())
