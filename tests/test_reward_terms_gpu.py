"""GPU: the fused step's per-warp reward term sums (``bezk_post_physics_rollout_ep_terms``) against the terms restated op by op
in fp32 torch from the post-step state and summed in the step's shuffle-tree order, the terms against the stored reward, byte
identity of everything else, the fold (``bezk_reward_terms_update``) against ``tests/reward_terms_oracle.py``, and ``A2CAgent``
with ``track_reward_terms``."""
import numpy as np
import pytest
import torch

from bez_isaacgym_b200 import bez_model as bm
from tests import reward_terms_oracle as ro
from tests.test_outcomes_gpu import _env, _mover, _reference

pytestmark = pytest.mark.gpu


def _c(x):
    return torch.tensor(x, dtype=torch.float32)


def _sqrt(x):
    """Correctly rounded fp32 square root, as the kernel's: torch's CPU fp32 sqrt is not (an fp64 root rounded to fp32 is)."""
    return x.double().sqrt().float()


def _restate(env):
    """(K, n) float32 per-env terms in the kernel's operation order, the fired mask, the band mask (envs whose branch or rule hangs
    on a quantity within its documented tie band) and the per-term tolerance class (True: bit-exact)."""
    n, m = env.num_envs, env.max_episode_length
    cls, band = _reference(env)
    fired = cls >= 0
    imu = env.rigid_body.view(n, -1, 13)[:, bm.IMU_BODY].cpu()
    q, v, w = imu[:, 3:7], imu[:, 7:10], imu[:, 10:13]
    dof = env.dof_state.view(n, 18, 2)[..., 0].cpu()
    default = torch.broadcast_to(env.default_dof_pos.cpu().reshape(-1, 18), (n, 18))
    pos_sq = torch.zeros(n)
    for j in range(18):
        d = default[:, j] - dof[:, j]
        pos_sq = pos_sq + d * d
    progress = env.progress_buf.cpu().float()
    zero = torch.zeros(n)
    exact = [True] * len(env.REWARD_TERMS)
    if env.TASK == "kick":
        root = env.root_states.view(n, 2, 13).cpu()
        bez, ball, bv = root[:, 0, 0:3], root[:, 1, 0:2], root[:, 1, 7:9]
        goal, bi = env.goal.cpu(), env.ball_init.cpu()
        dbx, dby = ball[:, 0] - bez[:, 0], ball[:, 1] - bez[:, 1]
        nbb = _sqrt(dbx * dbx + dby * dby)
        vel_fwd = (dbx / nbb) * v[:, 0] + (dby / nbb) * v[:, 1]
        dgx, dgy = goal[:, 0] - ball[:, 0], goal[:, 1] - ball[:, 1]
        n_goal = _sqrt(dgx * dgx + dgy * dgy)
        ball_fwd = (dgx / n_goal) * bv[:, 0] + (dgy / n_goal) * bv[:, 1]
        vs = v[:, 0] * v[:, 0]
        for x in (v[:, 1], v[:, 2], w[:, 0], w[:, 1], w[:, 2]):
            vs = vs + x * x
        vel_r, pos_r = _sqrt(vs) * _c(0.05), _sqrt(pos_sq) * _c(0.05)
        height = (_c(0.325) - bez[:, 2]).abs() * _c(1.0)
        kx, ky = ball[:, 0] - bi[:, 0], ball[:, 1] - bi[:, 1]
        far = _sqrt(kx * kx + ky * ky) > 0.3
        scored = _c(1.0) * (_c(100.0) - _c(100.0) * (progress / _c(float(m))))
        override = torch.where(cls == 3, scored, torch.where(cls == 4, zero, -torch.ones(n)))
        terms = [ball_fwd * _c(0.1), torch.where(far, zero, vel_fwd * _c(0.05)), -height, torch.where(far, -vel_r, zero),
                 torch.where(far, -pos_r, zero)]
    else:
        qx, qy, qz, qw = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
        a_z = _c(1.0) * (_c(2.0) * (qw * qw) - _c(1.0))
        b_z = ((qx * _c(0.0) - qy * _c(0.0)) * qw) * _c(2.0)
        dot = (qx * _c(0.0) + qy * _c(0.0)) + qz * _c(1.0)
        up = (a_z + b_z) + (qz * dot) * _c(2.0)
        s6 = v[:, 0] * v[:, 0]
        for x in (v[:, 1], v[:, 2], w[:, 0], w[:, 1], w[:, 2]):
            s6 = s6 + x * x
        dist_h = (_c(1.0) - up).abs()
        vel_s, pos_s = _sqrt(s6) * _c(0.05), _sqrt(pos_sq) * _c(0.05)
        if env.TASK == "walk":
            goal, bez = env.goal.cpu(), env.root_states.view(n, 13)[:, 0:2].cpu()
            dx, dy = goal[:, 0] - bez[:, 0], goal[:, 1] - bez[:, 1]
            n_goal = _sqrt(dx * dx + dy * dy)
            vel_fwd = (dx / n_goal) * v[:, 0] + (dy / n_goal) * v[:, 1]
            close = n_goal < 0.05
            lead, scale, out_value = vel_fwd * _c(10.0), _c(5.0), -100.0
        else:
            from oracle import task_oracle as to
            _, _, yaw = to.get_euler_xyz(q)
            ang = (env.goal_angle.cpu() - to.normalize_angle(yaw).unsqueeze(-1)).reshape(-1)
            close = ang < 0.05
            lead, scale, out_value = ang.abs() * _c(-0.5), _c(0.05), -5.0
            exact[0] = False                                  # atan2 / sincos: the kernel's and torch's differ in the last bits
        reached = _c(1.0) * (_c(1000.0) - _c(1000.0) * (progress / _c(float(m))))
        override = torch.where(cls == 0, torch.full((n,), -100.0), torch.where(cls == 1, reached,
                               torch.where(cls == 2, torch.full((n,), out_value), zero)))
        terms = [torch.where(close, zero, lead), -dist_h, torch.where(close, -vel_s, zero), torch.where(close, -pos_s, -(scale * pos_s))]
    terms = torch.stack([torch.where(fired, zero, t) for t in terms] + [torch.where(fired, override, zero)])
    return terms, fired, band, exact


def _run(env, steps, terms=True, outcomes=False, check=None, actions_seed=5):
    n = env.num_envs
    w = (n + 31) // 32
    ret, length = torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda")
    part = torch.full((steps, 3, w), float("nan"), dtype=torch.float64, device="cuda")
    oc = torch.full((steps, len(env.OUTCOMES), w), -1, dtype=torch.int32, device="cuda")
    tm = torch.full((steps, len(env.REWARD_TERMS), w), float("nan"), dtype=torch.float64, device="cuda")   # every slot is written
    g = torch.Generator(device="cuda").manual_seed(actions_seed)
    log = []
    for t in range(steps):
        extra = dict(values=torch.randn(n, device="cuda", generator=g), shaped_rewards=torch.empty(n, device="cuda"),
                     dones_u8=torch.empty(n, dtype=torch.uint8, device="cuda"))
        env.set_rollout_targets(**extra, episode_returns=ret, episode_lengths=length, episode_partials=part[t],
                                episode_outcomes=oc[t] if outcomes else None, reward_terms=tm[t] if terms else None)
        env.step(torch.rand(n, 18, device="cuda", generator=g) * 2 - 1)
        log.append(dict(rew=env.rew_buf.clone(), reset=env.reset_buf.clone(), progress=env.progress_buf.clone(),
                        obs=env.obs_buf.clone(), timeout=env.timeout_buf.clone(), ret=ret.clone(), len=length.clone(),
                        shaped=extra["shaped_rewards"], dones=extra["dones_u8"]))
        if check is not None:
            check(t, tm[t])
    env.set_rollout_targets()
    torch.cuda.synchronize()
    return log, part, oc, tm


def _check_step(env, got, stats):
    """The step's (K, W) partials against the restatement, and the restated terms against the stored reward."""
    n = env.num_envs
    w = (n + 31) // 32
    terms, fired, band, exact = _restate(env)
    want = torch.from_numpy(ro.warp_sums(terms.numpy(), n))
    got = got.cpu()
    keep = ~torch.nn.functional.pad(band.int(), (0, w * 32 - n)).view(w, 32).any(1)
    for k in range(terms.shape[0]):
        if exact[k]:
            assert torch.equal(got[k, keep].view(torch.int64), want[k, keep].view(torch.int64)), (env.REWARD_TERMS[k], k)
        else:
            assert torch.allclose(got[k, keep], want[k, keep], rtol=1e-5, atol=1e-5), env.REWARD_TERMS[k]
    rew = env.rew_buf.cpu()
    ok = ~band
    # where a rule fired the termination term IS the stored reward; elsewhere the terms sum to it up to fp32 re-association
    assert torch.equal(terms[-1][fired & ok], rew[fired & ok])
    s = terms.double().sum(0)
    tol = 4 * np.finfo(np.float32).eps * terms.double().abs().sum(0) + 1e-30
    for k in range(terms.shape[0]):
        if not exact[k]:
            tol = tol + 1e-5 * terms[k].double().abs()
    assert bool(((s - rew.double()).abs() <= tol)[~fired & ok].all())
    stats["warps"] += w
    stats["excluded"] += int((~keep).sum())
    stats["fired"] += int(fired.sum())


# 262 144 envs run the L2 variants
@pytest.mark.parametrize("outcomes", [False, True])
@pytest.mark.parametrize("task,n,cleats", [("kick", 4096, False), ("kick", 4096, True), ("walk", 4096, False), ("walk", 4096, True),
                                           ("orient", 4096, False), ("orient", 4096, True), ("kick", 4099, False),
                                           ("walk", 4099, True), ("orient", 4099, False), ("kick", 262144, False),
                                           ("walk", 262144, True), ("orient", 262144, False)])
def test_per_warp_terms_match_the_restatement(task, n, cleats, outcomes):
    env = _env(task, n, cleats)
    stats = dict(warps=0, excluded=0, fired=0)
    _, part, oc, tm = _run(env, 24 if n < 100000 else 8, outcomes=outcomes, check=lambda t, got: _check_step(env, got, stats))
    assert stats["fired"] > 0 and stats["excluded"] <= 0.02 * stats["warps"], stats
    assert not torch.isnan(tm).any()
    if outcomes:
        assert torch.equal(oc.sum(1).double(), part[:, 0])


def _hand_built(task, n):
    """Four groups (env % 4) away from every threshold: kick near / far / fell / scored; walk and orient not close / close /
    fell / out.  Every env moves (IMU linear velocity 0.2) and has a posture error, so every term of its branch is non-zero."""
    grp = torch.arange(n, device="cuda") % 4
    state = {}

    def sel(g):
        return (grp == g).view(-1, 1)

    def hook(sim):
        if "env" not in state:
            return
        env = state["env"]
        rb = sim.rigid_body.view(n, -1, 13)
        rb[:, bm.IMU_BODY, 3:7] = torch.tensor([0.0, 0.0, 0.0, 1.0], device="cuda")
        rb[:, bm.IMU_BODY, 7:13] = torch.tensor([0.2, 0.0, 0.0, 0.0, 0.0, 0.0], device="cuda")
        sim.dof_state.view(n, 18, 2)[..., 0] = env.default_dof_pos + 0.02
        sim.dof_state.view(n, 18, 2)[..., 1] = 0.0
        init = env.bez_init_xy.view(1, 2)
        if task == "kick":
            root = sim.root_states.view(n, 2, 13)
            goal, bi = env.goal, env.ball_init
            u = (goal - bi) / torch.linalg.norm(goal - bi, dim=1, keepdim=True)
            root[:, 0, 0:2], root[:, 0, 2] = init, 0.3
            root[:, 1, 7:9] = 0.4 * u
            root[:, 1, 0:2] = torch.where(sel(1), bi + 0.5 * u, torch.where(sel(3), goal - 0.01 * u, bi + 0.1 * u))
            root[:, 0, 2] = torch.where(sel(2).view(-1), torch.full_like(root[:, 0, 2], 0.2), root[:, 0, 2])
        else:
            root = sim.root_states.view(n, 13)
            root[:, 2] = 0.4
            rb[:, bm.IMU_BODY, 3:7] = torch.where(sel(2), torch.tensor([[1.0, 0.0, 0.0, 0.0]], device="cuda"), rb[:, bm.IMU_BODY, 3:7])
            if task == "walk":
                goal = env.goal
                ug = goal / torch.linalg.norm(goal, dim=1, keepdim=True)
                root[:, 0:2] = torch.where(sel(1), goal - 0.01 * ug, torch.where(sel(3), goal + 0.5 * ug, torch.zeros_like(goal)))
            else:
                root[:, 0:2] = torch.where(sel(3), init + torch.tensor([[0.5, 0.0]], device="cuda"), init.expand(n, 2))

    env = _env(task, n, hook=hook, move=False)
    state["env"] = env
    if task == "walk":
        env.goal.copy_(torch.tensor([[1.0, 1.5]], device="cuda").expand(n, 2))
    if task == "orient":
        env.goal_angle.copy_(torch.where(grp == 1, 0.0, 1.0).view(n, 1))
    env.reset_buf.zero_()
    env.progress_buf.fill_(10)
    return env, grp.cpu()


@pytest.mark.parametrize("task", ["kick", "walk", "orient"])
def test_hand_built_branches_and_overrides(task):
    n = 4096
    env, grp = _hand_built(task, n)
    stats = dict(warps=0, excluded=0, fired=0)
    _, _, _, tm = _run(env, 1, check=lambda t, got: _check_step(env, got, stats))
    assert stats["excluded"] == 0 and stats["fired"] == n // 2, stats
    terms, fired, _, _ = _restate(env)
    assert torch.equal(fired, (grp >= 2))
    rew = env.rew_buf.cpu()
    live = terms[:-1, grp < 2]
    if task == "kick":
        near, far = terms[:, grp == 0], terms[:, grp == 1]
        assert (near[1] != 0).all() and (near[3:5] == 0).all(), "near: approach, no body velocity / posture"
        assert (far[1] == 0).all() and (far[3:5] != 0).all(), "far: body velocity and posture, no approach"
        assert torch.equal(terms[-1, grp == 2], torch.full((n // 4,), -1.0))
    else:
        nc, cl = terms[:, grp == 0], terms[:, grp == 1]
        assert (nc[0] != 0).all() and (nc[2] == 0).all() and (nc[3] != 0).all(), "not close: lead term, no body velocity"
        assert (cl[0] == 0).all() and (cl[2] != 0).all() and (cl[3] != 0).all(), "close: body velocity, no lead term"
        assert torch.equal(terms[-1, grp == 3], torch.full((n // 4,), -100.0 if task == "walk" else -5.0))
    assert torch.isfinite(live).all() and torch.equal(terms[-1, grp >= 2], rew[grp >= 2])
    assert (terms[:-1, grp >= 2] == 0).all() and (terms[-1, grp < 2] == 0).all()
    assert float(tm[0, -1].sum()) == float(rew[grp >= 2].double().sum())


def test_nothing_else_moves_and_terms_repeat():
    for outcomes in (False, True):
        a = _run(_env("kick", 4099), 40, terms=False, outcomes=outcomes)
        b = _run(_env("kick", 4099), 40, terms=True, outcomes=outcomes)
        c = _run(_env("kick", 4099), 40, terms=True, outcomes=outcomes)
        for ra, rb in zip(a[0], b[0]):
            for key in ra:
                assert torch.equal(ra[key].contiguous().view(torch.uint8), rb[key].contiguous().view(torch.uint8)), key
        assert torch.equal(a[1].view(torch.uint8), b[1].view(torch.uint8)), "episode partials"
        assert torch.equal(a[2], b[2]), "outcome partials"
        assert torch.equal(b[3].view(torch.int64), c[3].view(torch.int64)), "term partials repeat"
    for task in ("walk", "orient"):
        a = _run(_env(task, 4096, cleats=True), 16, terms=False, outcomes=True)
        b = _run(_env(task, 4096, cleats=True), 16, terms=True, outcomes=True)
        assert all(torch.equal(ra[k].contiguous().view(torch.uint8), rb[k].contiguous().view(torch.uint8))
                   for ra, rb in zip(a[0], b[0]) for k in ra)
        assert torch.equal(a[1].view(torch.uint8), b[1].view(torch.uint8)) and torch.equal(a[2], b[2])


def test_fold_matches_the_restatement_and_the_mean_reward():
    from bez_isaacgym_b200 import ops
    g = torch.Generator().manual_seed(3)
    for task, k, n in (("kick", 6, 5000), ("walk", 5, 262144), ("orient", 5, 33)):
        w = (n + 31) // 32
        p = torch.randn(32, k, w, generator=g, dtype=torch.float64) * 7
        mean = torch.full((k,), float("nan"), dtype=torch.float64, device="cuda")
        ops.reward_terms_update(p.cuda(), n, task, mean)
        assert mean.cpu().numpy().tobytes() == ro.fold(p.numpy(), n).tobytes(), task
    env = _env("kick", 8192)
    log, _, _, tm = _run(env, 32)
    mean = torch.zeros(6, dtype=torch.float64, device="cuda")
    ops.reward_terms_update(tm, 8192, "kick", mean)
    want = torch.stack([r["rew"] for r in log]).double().mean()
    assert abs(float(mean.sum()) - float(want)) <= 1e-6 * (1 + abs(float(want)))
    assert mean.cpu().numpy().tobytes() == ro.fold(tm.cpu().numpy(), 8192).tobytes()


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


def test_agent_reward_terms_change_nothing_else(tmp_path):
    n, T = 2048, 16
    off, on, both = _agent(n, T), _agent(n, T, track_reward_terms=True), _agent(n, T, track_reward_terms=True, track_outcomes=True)
    assert not hasattr(off, "reward_terms")
    for _ in range(2):
        a, b, c = off.train_epoch(), on.train_epoch(), both.train_epoch()
        for key in ("a_loss", "c_loss", "kl"):
            assert torch.equal(torch.as_tensor(a[key]), torch.as_tensor(b[key])), key
            assert torch.equal(torch.as_tensor(a[key]), torch.as_tensor(c[key])), key
        for ag in (on, both):
            assert ag.reward_terms.mean.cpu().numpy().tobytes() == ro.fold(ag._rt_partials.cpu().numpy(), n).tobytes()
        assert torch.equal(on._rt_partials, both._rt_partials)
    for x in (on, both):
        for pa, pb in zip(off.model.parameters(), x.model.parameters()):
            assert torch.equal(pa, pb)
        assert np.array_equal(off.game_rewards.get_mean(), x.game_rewards.get_mean())
        assert np.array_equal(off.game_lengths.get_mean(), x.game_lengths.get_mean())
        assert torch.equal(off.current_rewards, x.current_rewards)
    (_, _), hist = _agent(n, 8, track_reward_terms=True, track_outcomes=True, max_epochs=2, name="K").train(str(tmp_path))
    assert len(hist) == 2 and all(list(h["reward_terms"]) == list(off.env.REWARD_TERMS) for h in hist)
    assert all(np.isfinite(list(h["reward_terms"].values())).all() and "outcomes" in h for h in hist)
    (_, _), hist = _agent(n, 8, max_epochs=1, name="K").train(str(tmp_path / "off"))
    assert "reward_terms" not in hist[0]
