"""GPU: the fused step's per-warp episode outcome counts (``bezk_post_physics_rollout_ep_outcome``) against the termination rules
recomputed with the oracle's torch ops, restatement-free invariants against the step's own outputs, byte identity of everything
else, the two folds (``bezk_outcome_meter_update``, ``bezk_player_outcome_update``) against ``tests/rl_games_outcome_oracle.py``,
and ``A2CAgent`` / ``PpoPlayerContinuous`` with ``track_outcomes``."""
import numpy as np
import pytest
import torch

from bez_isaacgym_b200 import bez_model as bm
from oracle import task_oracle as to
from tests import _util as U
from tests import rl_games_outcome_oracle as oo

pytestmark = pytest.mark.gpu


def _mover(seed):
    g = torch.Generator(device="cuda").manual_seed(seed)

    def move(sim):
        for t, s in ((sim.root_states, 0.02), (sim.rigid_body, 0.05), (sim.dof_state, 0.05), (sim.net_contact, 0.5)):
            t.add_(torch.randn(t.shape, generator=g, device=t.device) * s)
    return move


def _env(task, n, cleats=False, seed=3, hook=None, move=True):
    from bez_isaacgym_b200 import tasks
    from bez_isaacgym_b200.synthetic_sim import SyntheticGym
    cls = {"kick": tasks.KickEnv, "walk": tasks.WalkEnv, "orient": tasks.OrientEnv}[task]
    mv = _mover(seed)

    def on_sim(sim):
        if move:
            mv(sim)
        if hook is not None:
            hook(sim)
    sim = SyntheticGym(n, device="cuda:0", cleats=cleats, seed=seed, on_simulate=on_sim, task=task)
    cfg = bm.default_task_cfg(n, cleats=cleats, task=task)
    cfg["seed"] = seed
    env = cls(cfg, "cuda:0", 0, True, sim=sim)
    m = env.max_episode_length
    env.progress_buf.copy_(torch.randint(int(m) - 70, int(m), (n,), generator=torch.Generator().manual_seed(seed)).cuda())
    return env


def _ulp_band(x, thr, k=4):
    return (x - thr).abs() <= k * U.ulp(thr)


def _reference(env):
    """Per env: the last firing rule (class index, -1 if none) recomputed from the post-step state, and the tie-band mask."""
    n = env.num_envs
    m = env.max_episode_length
    progress = env.progress_buf.cpu()
    over = progress >= m
    imu = env.rigid_body.view(n, -1, 13)[:, bm.IMU_BODY].cpu()
    quat, lin, ang = imu[:, 3:7], imu[:, 7:10], imu[:, 10:13]
    if env.TASK == "kick":
        root = env.root_states.view(n, 2, 13).cpu()
        bez, ball = root[:, 0, 0:3], root[:, 1, 0:3]
        goal, ball_init = env.goal.cpu(), env.ball_init.cpu()
        n_goal = torch.linalg.norm(goal - ball[:, 0:2], dim=1)
        u = (goal - ball[:, 0:2]) / n_goal.reshape(-1, 1)
        ui = (goal - ball_init) / torch.linalg.norm(goal - ball_init, dim=1).reshape(-1, 1)
        angle = (torch.atan2(ui[:, 1], ui[:, 0]) - torch.atan2(u[:, 1], u[:, 0])).abs()
        strayed = torch.linalg.norm(bez[:, 0:2] - env.bez_init_xy.cpu(), dim=1) > 0.5
        rules = [bez[:, 2] < 0.275, strayed, angle > 1.5708, n_goal < 0.05, over]
        # reward_tie_band reads the root rows only; the other views need shapes, not values
        nb = env.sim.num_bodies
        st = type("S", (), dict(root_states=env.root_states.cpu(), dof_state=torch.zeros(n * 36), rigid_body=torch.zeros(n * nb * 13),
                                net_contact=torch.zeros(n * nb * 3), num_envs=n))
        band = U.reward_tie_band(st, goal, ball_init, tuple(env.bez_init_xy.tolist())) | _ulp_band(bez[:, 2], 0.275)
    else:
        root = env.root_states.view(n, 13).cpu()
        bez = root[:, 0:3]
        dof = env.dof_state.view(n, 18, 2)[..., 0].cpu()
        up_proj, _, vel_lin, vel_ang, pos = to._walk_terms(dof, env.default_dof_pos.cpu(), lin, ang, quat, n)
        if env.TASK == "walk":
            goal = env.goal.cpu()
            d = goal - bez[:, 0:2]
            close_v = torch.linalg.norm(d, dim=1)
            u = d / close_v.reshape(-1, 1)
            ui = goal / torch.linalg.norm(goal, dim=1).reshape(-1, 1)
            out_v = (torch.atan2(ui[:, 1], ui[:, 0]) - torch.atan2(u[:, 1], u[:, 0])).abs()
            out, out_thr = out_v > 1.5708, 1.5708
        else:
            _, _, yaw = to.get_euler_xyz(quat)
            close_v = (env.goal_angle.cpu() - to.normalize_angle(yaw).unsqueeze(-1)).reshape(-1)
            out_v = torch.linalg.norm(bez[:, 0:2] - env.bez_init_xy.cpu(), dim=1)
            out, out_thr = out_v > 0.3, 0.3
        state = (close_v < 0.05).float() + (pos < 0.15).float() + (vel_ang < 0.1).float() + (vel_lin < 0.1).float()
        rules = [up_proj < 0.7, state == 4.0, out, over]
        band = (_ulp_band(up_proj, 0.7) | _ulp_band(pos, 0.15) | _ulp_band(vel_ang, 0.1) | _ulp_band(vel_lin, 0.1)
                | _ulp_band(close_v, 0.05) | _ulp_band(out_v, out_thr))
    cls = torch.full((n,), -1, dtype=torch.long)
    for k, r in enumerate(rules):
        cls = torch.where(r, torch.full_like(cls, k), cls)
    return cls, band


def _per_warp(cls, k, w):
    n = cls.numel()
    z = torch.nn.functional.pad(cls, (0, w * 32 - n), value=-1).view(w, 32)
    return torch.stack([(z == c).sum(1) for c in range(k)]).int()


def _run(env, steps, outcomes=True, norm=False, rollout=True, actions_seed=5, check=None):
    n = env.num_envs
    w, k = (n + 31) // 32, len(env.OUTCOMES)
    ret, length = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    part = torch.full((steps, 3, w), float("nan"), dtype=torch.float64, device="cuda")
    oc = torch.full((steps, k, w), -1, dtype=torch.int32, device="cuda")            # every slot must be written
    g = torch.Generator(device="cuda").manual_seed(actions_seed)
    gm = torch.Generator().manual_seed(6)
    mean = (torch.randn(env.num_obs, generator=gm, dtype=torch.float64) * 2).cuda()
    var = (torch.rand(env.num_obs, generator=gm, dtype=torch.float64) * 3 + 0.05).cuda()
    log = []
    for t in range(steps):
        extra = {}
        if rollout:
            extra = dict(values=torch.randn(n, device="cuda", generator=g), shaped_rewards=torch.empty(n, device="cuda"),
                         dones_u8=torch.empty(n, dtype=torch.uint8, device="cuda"))
        if norm:
            extra.update(obs_norm=torch.empty(n, env.num_obs, device="cuda"), obs_mean=mean, obs_var=var)
        env.set_rollout_targets(**extra, episode_returns=ret, episode_lengths=length, episode_partials=part[t],
                                episode_outcomes=oc[t] if outcomes else None)
        env.step(torch.rand(n, 18, device="cuda", generator=g) * 2 - 1)
        rec = dict(rew=env.rew_buf.clone(), reset=env.reset_buf.clone(), progress=env.progress_buf.clone(), obs=env.obs_buf.clone(),
                   timeout=env.timeout_buf.clone(), ret=ret.clone(), len=length.clone())
        if rollout:
            rec.update(shaped=extra["shaped_rewards"], dones=extra["dones_u8"])
        if norm:
            rec["obs_norm"] = extra["obs_norm"]
        if check is not None:
            check(t, oc[t])
        log.append(rec)
    env.set_rollout_targets()
    torch.cuda.synchronize()
    return log, part, oc


# norm: the step with the observation normaliser too (task_tile_obsnorm_outcome_kernel); 262 144 envs run the L2 variants
@pytest.mark.parametrize("task,n,cleats,norm", [("kick", 4096, False, False), ("kick", 4096, True, False), ("walk", 4096, False, False),
                                                ("orient", 4096, False, False), ("kick", 4099, False, False),
                                                ("walk", 4099, False, False), ("kick", 262144, False, False),
                                                ("kick", 4096, True, True), ("walk", 4099, False, True), ("orient", 4096, True, True),
                                                ("kick", 262144, False, True)])
def test_per_warp_counts_are_exact(task, n, cleats, norm):
    env = _env(task, n, cleats)
    w, k = (n + 31) // 32, len(env.OUTCOMES)
    stats = dict(warps=0, excluded=0, done=0)
    seen = torch.zeros(k, dtype=torch.long)

    def check(t, oc):
        cls, band = _reference(env)
        want = _per_warp(cls, k, w)
        got = oc.cpu()
        bad_warp = torch.nn.functional.pad(band.int(), (0, w * 32 - n)).view(w, 32).any(1)
        keep = ~bad_warp
        assert torch.equal(got[:, keep], want[:, keep]), f"step {t}"
        assert int((got < 0).sum()) == 0
        stats["warps"] += w
        stats["excluded"] += int(bad_warp.sum())
        stats["done"] += int(got.sum())
        seen.add_(got.sum(1).long())
    log, part, oc = _run(env, 64, norm=norm, check=check)
    assert stats["done"] > 0 and stats["excluded"] <= 0.01 * stats["warps"], stats
    # restatement-free: per slot, the class counts sum to the episode partials' done count
    assert torch.equal(oc.sum(1).double(), part[:, 0])
    # per warp, the counts agree with the rewards and progress the step stored
    m = env.max_episode_length
    for t, rec in enumerate(log):
        done, rew, prog = rec["reset"] != 0, rec["rew"], rec["progress"]
        pad = w * 32 - n

        def per_warp(mask):
            return torch.nn.functional.pad(mask.int(), (0, pad)).view(w, 32).sum(1)
        timeout = done & (prog >= m)
        rest = done & ~timeout
        if task == "kick":                    # fell / strayed / wide pay -1, scored 100 - 100 p / max >= 0
            assert torch.equal(oc[t, 4], per_warp(timeout))
            assert torch.equal(oc[t, 0] + oc[t, 1] + oc[t, 2], per_warp(rest & (rew == -1.0)))
            assert torch.equal(oc[t, 3], per_warp(rest & (rew != -1.0)))
        else:                                 # fell pays -100, out -100 (walk) / -5 (orient), reached 1000 - 1000 p / max >= 0
            assert torch.equal(oc[t, 3], per_warp(timeout))
            assert torch.equal(oc[t, 1], per_warp(rest & (rew >= 0.0)))
            if task == "walk":
                assert torch.equal(oc[t, 0] + oc[t, 2], per_warp(rest & (rew == -100.0)))
            else:
                assert torch.equal(oc[t, 0], per_warp(rest & (rew == -100.0)))
                assert torch.equal(oc[t, 2], per_warp(rest & (rew == -5.0)))
    assert int(seen[-1]) > 0, "timeouts fire"


def _hand_built_kick(n):
    """Eight groups (env % 8): none, fell, strayed, wide, scored, timeout, scored + timeout (timeout wins), fell + strayed + wide
    (wide wins)."""
    grp = torch.arange(n, device="cuda") % 8
    state = {}

    def hook(sim):
        if "env" not in state:
            return
        env = state["env"]
        root = sim.root_states.view(n, 2, 13)
        init = env.bez_init_xy.view(1, 2)
        goal, bi = env.goal, env.ball_init
        u = (goal - bi) / torch.linalg.norm(goal - bi, dim=1, keepdim=True)
        root[:, 0, 0:2] = init
        root[:, 0, 2] = 0.325
        root[:, 1, 0:2] = bi + 0.1 * u
        sel = lambda *g: torch.isin(grp, torch.tensor(g, device="cuda")).view(-1, 1)     # noqa: E731
        root[:, 0, 2] = torch.where(sel(1, 7).view(-1), torch.full_like(root[:, 0, 2], 0.2), root[:, 0, 2])
        root[:, 0, 0:2] = torch.where(sel(2, 7), init + torch.tensor([[0.6, 0.0]], device="cuda"), root[:, 0, 0:2])
        root[:, 1, 0:2] = torch.where(sel(3, 7), goal + 0.5 * u, root[:, 1, 0:2])
        root[:, 1, 0:2] = torch.where(sel(4, 6), goal - 0.01 * u, root[:, 1, 0:2])
    env = _env("kick", n, hook=hook, move=False)
    state["env"] = env
    m = env.max_episode_length
    env.reset_buf.zero_()
    env.progress_buf.copy_(torch.where((grp == 5) | (grp == 6), torch.full_like(env.progress_buf, m - 1), torch.full_like(env.progress_buf, 10)))
    return env, [0, 4, 4, 8, 4, 8]            # per warp: none (not counted), fell, strayed, wide, scored, timeout


def _hand_built_walk(n):
    """Six groups (env % 6): none, fell, reached, out, timeout, fell + out (out wins)."""
    grp = torch.arange(n, device="cuda") % 6
    state = {}

    def hook(sim):
        if "env" not in state:
            return
        env = state["env"]
        root = sim.root_states.view(n, 13)
        rb = sim.rigid_body.view(n, -1, 13)
        goal = env.goal
        ug = goal / torch.linalg.norm(goal, dim=1, keepdim=True)
        sel = lambda *g: torch.isin(grp, torch.tensor(g, device="cuda")).view(-1, 1)     # noqa: E731
        root[:, 0:2] = 0.0
        root[:, 2] = 0.4
        rb[:, bm.IMU_BODY, 3:7] = torch.tensor([0.0, 0.0, 0.0, 1.0], device="cuda")
        rb[:, bm.IMU_BODY, 7:13] = 0.0
        sim.dof_state.view(n, 18, 2)[..., 0] = env.default_dof_pos
        sim.dof_state.view(n, 18, 2)[..., 1] = 0.0
        rb[:, bm.IMU_BODY, 3:7] = torch.where(sel(1, 5), torch.tensor([[1.0, 0.0, 0.0, 0.0]], device="cuda"), rb[:, bm.IMU_BODY, 3:7])
        root[:, 0:2] = torch.where(sel(2), goal - 0.01 * ug, root[:, 0:2])
        root[:, 0:2] = torch.where(sel(3, 5), goal + 0.5 * ug, root[:, 0:2])
    env = _env("walk", n, hook=hook, move=False)
    state["env"] = env
    env.goal.copy_(torch.tensor([[1.0, 1.5]], device="cuda").expand(n, 2))
    m = env.max_episode_length
    env.reset_buf.zero_()
    env.progress_buf.copy_(torch.where(grp == 4, torch.full_like(env.progress_buf, m - 1), torch.full_like(env.progress_buf, 10)))
    return env, grp


def test_hand_built_states_fire_each_rule_and_the_later_rule_wins():
    n = 4096
    env, want = _hand_built_kick(n)
    _, part, oc = _run(env, 1)
    w = n // 32
    for c, cnt in enumerate(want[1:]):
        assert torch.equal(oc[0, c].cpu(), torch.full((w,), cnt, dtype=torch.int32)), (env.OUTCOMES[c], oc[0, c, :4])
    assert torch.equal(part[0, 0].cpu(), torch.full((w,), 28.0, dtype=torch.float64))

    n = 4032                                                  # 6 | 4032 and 32 | 4032
    env, grp = _hand_built_walk(n)
    _, part, oc = _run(env, 1)
    cls = torch.tensor([-1, 0, 1, 2, 3, 2])[grp.cpu()]
    assert torch.equal(oc[0].cpu(), _per_warp(cls, 4, n // 32))


def test_nothing_else_moves_and_counts_repeat():
    for norm in (False, True):
        a = _run(_env("kick", 4099), 48, outcomes=False, norm=norm)
        b = _run(_env("kick", 4099), 48, outcomes=True, norm=norm)
        c = _run(_env("kick", 4099), 48, outcomes=True, norm=norm)
        for ra, rb in zip(a[0], b[0]):
            for key in ra:
                x, y = ra[key], rb[key]
                assert torch.equal(x.contiguous().view(torch.uint8), y.contiguous().view(torch.uint8)), key
        assert torch.equal(a[1].view(torch.uint8), b[1].view(torch.uint8)), "episode partials"
        assert torch.equal(b[2], c[2]), "outcome partials repeat"
    a = _run(_env("orient", 4096, cleats=True), 32, outcomes=False, norm=True)
    b = _run(_env("orient", 4096, cleats=True), 32, outcomes=True, norm=True)
    assert all(torch.equal(x.view(torch.uint8), y.view(torch.uint8)) for ra, rb in zip(a[0], b[0]) for x, y in
               ((ra[key].contiguous(), rb[key].contiguous()) for key in ra))


def test_folds_match_the_restatement():
    from bez_isaacgym_b200 import ops
    g = torch.Generator().manual_seed(2)
    for task, k in (("kick", 5), ("walk", 4)):
        n = 5000
        w = (n + 31) // 32
        p = torch.randint(0, 3, (70, k, w), generator=g, dtype=torch.int32)
        p[torch.rand(70, generator=g) < 0.2] = 0
        pc = p.cuda()
        mean, size = torch.zeros(k, device="cuda"), torch.zeros(1, dtype=torch.int64, device="cuda")
        for t0 in range(0, 70, 9):
            ops.outcome_meter_update(pc[t0:t0 + 9], n, task, 300, mean, size)
        want, wsize = oo.meter(p.numpy(), 300)
        assert mean.cpu().numpy().tobytes() == want.tobytes() and int(size) == wsize
        games = int(p[:40].sum()) - 3                           # the cutoff lands inside step 39
        want_c, want_per = oo.player_fold(p.numpy(), games)
        for chunk in (1, 7, 32, 70):
            counts = torch.zeros(1 + k, dtype=torch.float64, device="cuda")
            per = torch.zeros(70, k, dtype=torch.float64, device="cuda")
            for t0 in range(0, 70, chunk):
                ops.player_outcome_update(pc[t0:t0 + chunk], n, task, games, counts, per[t0:t0 + chunk])
            assert counts.cpu().numpy().tobytes() == want_c.tobytes() and per.cpu().numpy().tobytes() == want_per.tobytes()
        assert want_per[40:].sum() == 0 and want_per[39].sum() > 0


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


def test_agent_outcomes_change_nothing_else_and_follow_the_meter(tmp_path):
    n, T = 2048, 16
    off, on = _agent(n, T), _agent(n, T, track_outcomes=True)
    assert not hasattr(off, "game_outcomes")
    gm, size = None, 0
    for _ in range(2):
        a, b = off.train_epoch(), on.train_epoch()
        for key in ("a_loss", "c_loss", "kl"):
            assert torch.equal(torch.as_tensor(a[key]), torch.as_tensor(b[key])), key
        assert on.game_outcomes.current_size == on.game_rewards.current_size == off.game_rewards.current_size
        gm, size = oo.meter(on._oc_partials.cpu().numpy(), 100, gm, size)
        assert on.game_outcomes.get_mean().tobytes() == gm.tobytes() and on.game_outcomes.current_size == size
    for pa, pb in zip(off.model.parameters(), on.model.parameters()):
        assert torch.equal(pa, pb)
    assert np.array_equal(off.game_rewards.get_mean(), on.game_rewards.get_mean())
    assert np.array_equal(off.game_lengths.get_mean(), on.game_lengths.get_mean())
    assert torch.equal(off.current_rewards, on.current_rewards)
    (_, _), hist = _agent(n, 8, track_outcomes=True, max_epochs=3, name="K").train(str(tmp_path))
    rows = [h for h in hist if h["outcomes"] is not None]
    assert rows and all(abs(sum(h["outcomes"].values()) - 1.0) <= 1e-6 for h in rows)
    assert list(rows[0]["outcomes"]) == ["fell", "strayed", "wide", "scored", "timeout"]
    (_, _), hist = _agent(n, 8, max_epochs=1, name="K").train(str(tmp_path / "off"))
    assert "outcomes" not in hist[0]


def _player(env, sync_every=32, track_outcomes=False, **config):
    from bez_isaacgym_b200.learner import PpoPlayerContinuous
    torch.manual_seed(11)
    return PpoPlayerContinuous(env, dict(dict(print_stats=False), **config), sync_every=sync_every, track_outcomes=track_outcomes)


def test_player_counts_every_game_once_for_any_sync_every(capsys):
    results = []
    for sync in (1, 7, 32):
        results.append(_player(_env("kick", 4096), sync_every=sync, track_outcomes=True, games_num=3000).run())
    assert results[0] == results[1] == results[2]
    r = results[0]
    assert sum(r["outcomes"].values()) == r["games_played"] >= 3000
    assert abs(sum(r["outcome_rates"].values()) - 1.0) < 1e-12
    out = capsys.readouterr().out
    assert out.count("outcomes: fell") == 3 and out.index("av reward:") < out.index("outcomes:")
    plain = _player(_env("kick", 4096), games_num=3000).run()
    assert set(plain) == {"games_played", "sum_rewards", "sum_steps", "av_reward", "av_steps"}
    assert plain == {k: r[k] for k in plain}
    assert "outcomes:" not in capsys.readouterr().out
    w = _player(_env("walk", 4096), track_outcomes=True, games_num=500).run()
    assert sum(w["outcomes"].values()) == w["games_played"] and list(w["outcomes"]) == ["fell", "reached", "out", "timeout"]


@pytest.mark.parametrize("task", ["kick", "walk", "orient"])
@pytest.mark.parametrize("norm", [False, True])
def test_ops_wrapper_routes_every_argument(task, norm):
    """``ops.post_physics_rollout_ep_outcome`` on a synthetic state against ``ops.post_physics_rollout_ep`` / ``_ep_norm`` on a copy
    of it: every output the same bytes, and the outcome counts consistent with the done counts and the stored rewards."""
    from bez_isaacgym_b200 import ops, synthetic_gym as sg
    n = 4099
    w = (n + 31) // 32
    actors, nb, width = bm.task_dims(task)
    cfg = ops.make_task_cfg(num_bodies=nb)
    runs = []
    for with_outcomes in (False, True):
        st = sg.make_state(n, seed=21, task=task).to("cuda")
        progress, reset = sg.make_bookkeeping(n, seed=22, device="cuda", p_reset=0.1)
        progress[:64] = 899
        t = dict(st=st, progress=progress, reset=reset, timeout=torch.empty(n, dtype=torch.long, device="cuda"),
                 obs=torch.empty(n, width, device="cuda"), rew=torch.empty(n, device="cuda"), prev=torch.zeros(n, 3, device="cuda"),
                 goal=torch.tensor([[1.5, 0.0]] if task == "kick" else [[2.0, 0.5]], device="cuda").repeat(n, 1),
                 shaped=torch.empty(n, device="cuda"), dones=torch.empty(n, dtype=torch.uint8, device="cuda"),
                 ret=torch.rand(n, device="cuda", generator=torch.Generator(device="cuda").manual_seed(1)),
                 len=torch.full((n,), 7.0, device="cuda"), part=torch.full((3, w), float("nan"), dtype=torch.float64, device="cuda"),
                 oc=torch.full((5 if task == "kick" else 4, w), -1, dtype=torch.int32, device="cuda"),
                 obs_norm=torch.empty(n, width, device="cuda"))
        mean = torch.linspace(-1, 1, width, dtype=torch.float64, device="cuda")
        var = torch.linspace(0.1, 2, width, dtype=torch.float64, device="cuda")
        args = (task, st.dof_state, st.rigid_body, st.root_states, st.net_contact, t["goal"], sg.make_initial_root_states(n, "cuda", task=task),
                reset, progress, t["timeout"], cfg, t["obs"], t["rew"])
        kw = dict(rollout_cfg=ops.make_rollout_cfg(), values=torch.ones(n, device="cuda"), shaped_rewards=t["shaped"], dones_u8=t["dones"],
                  goal_angle=torch.full((n,), 1.5708, device="cuda") if task == "orient" else None,
                  ball_init=torch.tensor([[0.175, 0.0]], device="cuda").repeat(n, 1) if task == "kick" else None,
                  prev_lin_vel=t["prev"], seed=5, step=3)
        normkw = dict(obs_mean=mean, obs_var=var, obs_norm=t["obs_norm"]) if norm else {}
        if with_outcomes:
            ops.post_physics_rollout_ep_outcome(*args, t["ret"], t["len"], t["part"], t["oc"], **normkw, **kw)
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
    oc = b["oc"]
    assert int((oc < 0).sum()) == 0 and torch.equal(oc.sum(0).double(), b["part"][0])
    done = b["reset"] != 0
    timeout = done & (b["progress"] >= cfg.max_episode_length)
    assert int(timeout.sum()) > 0
    per_warp = torch.nn.functional.pad(timeout.int(), (0, w * 32 - n)).view(w, 32).sum(1)
    assert torch.equal(oc[-1], per_warp)
