"""GPU: the exact retry of every kernel that divides and takes square roots through ``Mth<true>`` (``csrc/bezk_common.cuh``).  The
branch-free fast sequences are IEEE-exact only for operands in 2^-60 .. 2^60; outside it they set a sticky flag, and each call site
recomputes its quantities with the plain operators.  Each case below feeds one operand outside that window for which the fast sequence
gives DIFFERENT bits from IEEE (it discriminates), so a missing or partial retry fails the comparison with an fp32 restatement of the
same operations (``tests/exact_retry_reference.py``, ``tests/learner_reference.py``).  Every case asserts in Python that its operand,
formed from the same fp32 inputs, lies outside the window.  Output buffers of the direct kernel calls sit between guard bands.

  site (csrc/)                          operand outside the window            why it discriminates
  1  step observation                   |q|^2 = 1e38 >= 2^126 (IMU quaternion  rcp.approx.ftz flushes 1/|q|^2 = 2e-38 to 0: two_s = 0, so
     bezk_task.cu imu_term /             (0, 1e19, 0, 0), xyzw)                 m22 = 1 instead of -1 and obs column 38 flips sign
     off_orn_term                       walk: robot -> goal distance^2 = 1e-40 rsqrt.approx.ftz flushes the subnormal radicand: the fast
                                        (goal (1e-20, 0), torso at the origin) root is NaN, IEEE gives 1e-20 (obs columns 42:44)
  2  step reward                        walk / orient: |w|^2 = 1e-40 (IMU      fast vel_ang is NaN, IEEE 1e-20 < 0.1: the win rule (and its
     reward_walk / reward_orient /      angular velocity (1e-20, 0, 0), zero   outcome class and termination term) fires only with the retry
     reward_term                        linear velocity, close to the goal)
                                        kick, far branch: the six IMU           fast vel_r is NaN, so is the reward and the body velocity term
                                        velocities 1e-20 -> |v|^2 = 6e-40
                                        walk: goal distance^2 = 1e-40 (above)   fast n_goal NaN: "close" fails and the reward is NaN
  3  in-step observation normaliser     dof velocity +-3e38 / +-inf in columns quotient overflow / infinite numerator: the residual step
     (obs_mean / obs_var armed)         of variance 0; a column of variance inf makes NaN where IEEE gives +-inf -> +-5; den = inf: fast
                                                                               0 * inf = NaN where IEEE gives +-0
  4  rms_normalize_kernel               as 3, statistics given                 as 3 (plain, slabs, the planned batched path)
  5  rms_merge_normalize_kernel         a column of +-1e20 rows: the merged    den = sqrt(inf) = inf: IEEE +-0, fast NaN (the sharded path
                                        variance is inf in fp32                and the c > 1 chain of rms_train_forward)
  6  fused_stats_kernel mode 0          as 5, c = 1, 2 <= m <= B               as 5
  7  ppo_loss_kernel                    logstd[4] = -90: sigma = 8e-40 is      1/sigma flushes: every row's neglogp / KL is NaN without the
                                        subnormal (every row, check_divisor)   retry; IEEE gives 0 / inf
                                        old_sigma = 1.5e19 in one row: the KL  fast NaN, IEEE 0: only the KL sum shows it
                                        divisor 2 (old_sigma^2 + 1e-5) is inf
  8  policy_head_kernel                 logstd[4] = -90 (as 7)                 as 7; neglogp against the restatement with the head's sigmas

Layout of the fused-step cases: retrying envs at lane 0 and lane 31 of a warp, one warp made only of retrying envs and the partial last
warp of n = 4099, among ordinary envs; the same state at 262 144 envs runs the L2 kernels.  Every family of the step (plain, rollout,
episode, normaliser, outcomes, terms, split kick parts 3 + 4) must give the same bytes, and ordinary envs next to a retrying env the same
bytes as when that env is moved back inside the window.
"""
import pytest
import torch

from bez_isaacgym_b200 import bez_model as bm
from tests import exact_retry_reference as X
from tests import learner_reference as R
from tests import reward_terms_oracle as ro
from tests._util import Guarded

pytestmark = pytest.mark.gpu

ORD, QUAT, SLOW, NEAR = 0, 1, 2, 3          # ordinary, |q|^2 = 1e38, subnormal velocity radicand, subnormal goal distance (walk)
TINY = 1e-20
BIG_Q = 1e19
WARP = 32


def _kinds(task, n):
    """Per env: which case it holds.  Retrying envs at lane 0 of warp 3, lane 31 of warp 5, all of warp 7, the partial last warp (or
    the last env) and lane 31 of the last full warp; the rest ordinary."""
    kinds = [QUAT, SLOW] + ([NEAR] if task == "walk" else [])
    k = torch.zeros(n, dtype=torch.long)
    pos = [3 * WARP, 5 * WARP + 31] + list(range(7 * WARP, 8 * WARP)) + [n - 2, n - 1, (n // WARP - 1) * WARP + 31 if n % WARP else n - 33]
    for i, p in enumerate(pos):
        k[p] = kinds[i % len(kinds)]
    return k


def _make_env(task, n, kinds, fusion="fused", clip=None):
    from bez_isaacgym_b200 import tasks
    from bez_isaacgym_b200.synthetic_sim import SyntheticGym
    kd = kinds.cuda()
    state = {}

    def sel(k):
        return (kd == k).view(-1, 1)

    def hook(sim):
        if "env" not in state:
            return
        env = state["env"]
        rb = sim.rigid_body.view(n, -1, 13)
        imu = rb[:, bm.IMU_BODY]
        imu[:, 3:7] = torch.where(sel(QUAT), torch.tensor([[0.0, BIG_Q, 0.0, 0.0]], device="cuda"),
                                  torch.tensor([[0.0, 0.0, 0.0, 1.0]], device="cuda"))
        slow = torch.tensor([[0.0, 0.0, 0.0, TINY, 0.0, 0.0]] if task != "kick" else [[TINY] * 6], device="cuda")
        imu[:, 7:13] = torch.where(sel(SLOW), slow, torch.tensor([[0.2, 0.0, 0.0, 0.0, 0.0, 0.0]], device="cuda"))
        dof = sim.dof_state.view(n, 18, 2)
        still = sel(SLOW) if task != "kick" else torch.zeros_like(sel(SLOW))      # walk / orient: no posture error (win rule)
        dof[..., 0] = torch.where(still, env.default_dof_pos + 0.0, env.default_dof_pos + 0.02)
        dof[..., 1] = torch.linspace(-1.0, 1.0, 18, device="cuda")
        init = env.bez_init_xy.view(1, 2)
        if task == "kick":
            root = sim.root_states.view(n, 2, 13)
            goal, bi = env.goal, env.ball_init
            u = (goal - bi) / torch.linalg.norm(goal - bi, dim=1, keepdim=True)
            root[:, 0, 0:2], root[:, 0, 2] = init, 0.3
            root[:, 1, 7:9] = 0.4 * u
            root[:, 1, 0:2] = torch.where(sel(SLOW), bi + 0.5 * u, bi + 0.1 * u)
        else:
            root = sim.root_states.view(n, 13)
            root[:, 2] = 0.4
            if task == "walk":
                goal = env.goal
                ug = goal / torch.linalg.norm(goal, dim=1, keepdim=True)
                root[:, 0:2] = torch.where(sel(SLOW), goal - 0.01 * ug, torch.zeros_like(goal))
            else:
                root[:, 0:2] = init.expand(n, 2)

    cls = {"kick": tasks.KickEnv, "walk": tasks.WalkEnv, "orient": tasks.OrientEnv}[task]
    sim = SyntheticGym(n, device="cuda:0", seed=3, on_simulate=hook, task=task)
    cfg = bm.default_task_cfg(n, task=task)
    cfg["seed"] = 3
    if clip is not None:
        cfg["env"]["clipObservations"] = clip
    env = cls(cfg, "cuda:0", 0, True, sim=sim, fusion=fusion)
    state["env"] = env
    if task == "walk":
        env.goal.copy_(torch.where((kd == NEAR).view(-1, 1), torch.tensor([[TINY, 0.0]], device="cuda"),
                                   torch.tensor([[1.0, 1.5]], device="cuda")))
    if task == "orient":
        env.goal_angle.copy_(torch.where(kd == SLOW, 0.0, 1.0).view(n, 1))
    env.reset_buf.zero_()
    env.progress_buf.fill_(10)
    return env


def _state(env):
    """The post-step inputs of the restatement, on the CPU."""
    n = env.num_envs
    imu = env.rigid_body.view(n, -1, 13)[:, bm.IMU_BODY].cpu()
    s = dict(q=imu[:, 3:7], v=imu[:, 7:10], w=imu[:, 10:13],
             psq=X.pos_sq(env.dof_state.view(n, 18, 2)[..., 0].cpu(),
                          torch.broadcast_to(env.default_dof_pos.cpu().reshape(-1, 18), (n, 18))),
             progress=env.progress_buf.cpu(), bez_init=tuple(env.bez_init_xy.tolist()))
    if env.TASK == "kick":
        root = env.root_states.view(n, 2, 13).cpu()
        s.update(bez=root[:, 0, 0:3], ball=root[:, 1, 0:2], ball_v=root[:, 1, 7:9], goal=env.goal.cpu(), ball_init=env.ball_init.cpu())
    else:
        s.update(bez=env.root_states.view(n, 13)[:, 0:3].cpu(), goal=env.goal.cpu() if env.TASK == "walk" else None,
                 goal_angle=env.goal_angle.cpu().view(-1) if env.TASK == "orient" else None)
    return s


def _restate(env, s):
    n, m = env.num_envs, env.max_episode_length
    zero = torch.zeros(n, dtype=torch.long)
    if env.TASK == "kick":
        return X.kick_step(s["bez"], s["ball"], s["ball_v"], s["goal"], s["ball_init"], s["v"], s["w"], s["psq"], s["bez_init"],
                           s["progress"], m, zero)
    return X.walk_step(env.TASK, s["bez"], s["q"], s["v"], s["w"], s["psq"], s["goal"], s["goal_angle"], s["bez_init"], s["progress"],
                       m, zero)


def _preconditions(env, kinds, s):
    """Each retrying env's operand, formed from the same fp32 inputs, lies outside 2^-60 .. 2^60."""
    q, v, w = s["q"], s["v"], s["w"]
    norm2 = ((q[:, 0] * q[:, 0] + q[:, 1] * q[:, 1]) + q[:, 2] * q[:, 2]) + q[:, 3] * q[:, 3]
    assert X.outside_window(norm2[kinds == QUAT]).all()
    if env.TASK == "kick":
        vs = X.sumsq(v[:, 0], v[:, 1], v[:, 2], w[:, 0], w[:, 1], w[:, 2])
    else:
        vs = X.sumsq(w[:, 0], w[:, 1], w[:, 2])
    assert X.outside_window(vs[kinds == SLOW]).all() and (vs[kinds == SLOW] > 0).all()
    if env.TASK == "walk":
        d = s["goal"] - s["bez"][:, 0:2]
        r2 = X.sumsq(d[:, 0], d[:, 1])
        assert X.outside_window(r2[kinds == NEAR]).all() and (r2[kinds == NEAR] > 0).all()
    assert not X.outside_window(norm2[kinds == ORD]).any()


FAMILIES = ("plain", "rollout", "ep", "ep_norm", "ep_outcome", "ep_outcome_norm", "ep_terms", "ep_terms_outcome")


def _step(env, family, kinds, norm_stats=None):
    """One step of ``family``; returns every output as CPU tensors."""
    n = env.num_envs
    w, k = (n + 31) // 32, len(env.OUTCOMES)
    out = {}
    extra = {}
    if family != "plain":
        g = torch.Generator(device="cuda").manual_seed(1)
        extra = dict(values=torch.randn(n, device="cuda", generator=g), shaped_rewards=torch.full((n,), float("nan"), device="cuda"),
                     dones_u8=torch.full((n,), 7, dtype=torch.uint8, device="cuda"))
    if family.startswith("ep"):
        extra.update(episode_returns=torch.zeros(n, device="cuda"), episode_lengths=torch.zeros(n, device="cuda"),
                     episode_partials=torch.full((3, w), float("nan"), dtype=torch.float64, device="cuda"))
    if "outcome" in family:
        extra["episode_outcomes"] = torch.full((k, w), -1, dtype=torch.int32, device="cuda")
    if "terms" in family:
        extra["reward_terms"] = torch.full((len(env.REWARD_TERMS), w), float("nan"), dtype=torch.float64, device="cuda")
    if "norm" in family:
        mean, var = norm_stats if norm_stats is not None else _norm_stats(env.num_obs)
        extra.update(obs_norm=torch.full((n, env.num_obs), float("nan"), device="cuda"), obs_mean=mean.cuda(), obs_var=var.cuda())
    if extra:
        env.set_rollout_targets(**extra)
    prev = env.prev_lin_vel.clone().cpu()
    assert not env._prev_is_view
    env.step(torch.zeros(n, 18, device="cuda"))
    if extra:
        env.set_rollout_targets()
    torch.cuda.synchronize()
    out.update(rew=env.rew_buf, reset=env.reset_buf, progress=env.progress_buf, timeout=env.timeout_buf, obs=env.obs_buf)
    if env.obs_clipped_buf is not None:
        out["obs_clipped"] = env.obs_clipped_buf
    for key in ("values", "shaped_rewards", "dones_u8", "episode_returns", "episode_lengths", "episode_partials", "episode_outcomes",
                "reward_terms", "obs_norm", "obs_mean", "obs_var"):
        if key in extra:
            out[key] = extra[key]
    out = {key: t.detach().cpu().clone() for key, t in out.items()}
    out["prev"] = prev
    return out


def _norm_stats(c):
    mean = torch.linspace(-0.5, 0.5, c, dtype=torch.float64)
    var = torch.linspace(0.5, 2.0, c, dtype=torch.float64)
    return mean, var


def _bits(t):
    t = t.contiguous()
    return t.view(torch.uint8) if t.dtype != torch.uint8 else t


def _same_bytes(a, b, what):
    assert a.shape == b.shape, what
    assert torch.equal(_bits(a), _bits(b)), f"{what}: {int((_bits(a) != _bits(b)).sum())} bytes differ"


def _check_against_restatement(env, kinds, out):
    n = env.num_envs
    w = (n + 31) // 32
    s = _state(env)
    _preconditions(env, kinds, s)
    rew, reset, cls, terms = _restate(env, s)
    retry = kinds != ORD
    _same_bytes(out["rew"], rew, "rew")
    _same_bytes(out["reset"], reset, "reset")
    assert torch.equal(out["progress"], s["progress"]) and bool((out["progress"] == 11).all())
    assert not out["timeout"].any()
    # the retrying envs' rules: a fall (|q|^2 = 1e38 has q_w = 0) or the win (walk / orient), nothing for kick
    if env.TASK == "kick":
        assert bool((cls[retry] == -1).all()) and torch.isfinite(rew).all()
    else:
        assert bool((cls[kinds == QUAT] == 0).all()) and bool((cls[kinds == SLOW] == 1).all())
    obs = out["obs"]
    imu = X.imu_lin_acc(s["q"], s["v"], out["prev"], env._kcfg.dt, env._kcfg.imu_max_lin_acc)
    _same_bytes(obs[:, 36:39], imu, "IMU linear acceleration (obs 36:39)")
    assert bool((obs[kinds == QUAT, 38] < 0).all()), "m22 = -1 for |q|^2 = 1e38"
    _same_bytes(obs[:, 39:42], torch.clamp(s["w"], -env._kcfg.imu_max_ang_vel, env._kcfg.imu_max_ang_vel), "IMU angular velocity")
    if env.TASK != "orient":                       # compute_off_orn through atan2f / sincosf: NaN pattern + tolerance
        from oracle import task_oracle as to
        want = to.off_orn(s["bez"], s["q"], s["goal"])
        got = obs[:, 42:44]
        assert torch.equal(torch.isnan(got), torch.isnan(want)) and not torch.isnan(got).any()
        assert torch.allclose(got, want, rtol=1e-5, atol=1e-5)
    if "shaped_rewards" in out:
        timeout = out["timeout"].float()
        shaped = (rew + X.c(0.0)) * X.c(0.01) + (X.c(0.99) * out["values"]) * timeout
        _same_bytes(out["shaped_rewards"], shaped, "shaped rewards")
        _same_bytes(out["dones_u8"], (reset != 0).to(torch.uint8), "dones")
    if "episode_returns" in out:
        done = reset != 0
        r, length = torch.zeros(n) + rew, torch.zeros(n) + X.c(1.0)
        nd = X.c(1.0) - done.float()
        _same_bytes(out["episode_returns"], r * nd, "episode returns")
        _same_bytes(out["episode_lengths"], length * nd, "episode lengths")
        per = torch.stack([done.float(), torch.where(done, r, torch.zeros(n)), torch.where(done, length, torch.zeros(n))])
        want = torch.from_numpy(ro.warp_sums(per.numpy(), n))
        _same_bytes(out["episode_partials"], want, "episode partials")
    if "episode_outcomes" in out:
        z = torch.nn.functional.pad(cls, (0, w * 32 - n), value=-1).view(w, 32)
        want = torch.stack([(z == k).sum(1) for k in range(len(env.OUTCOMES))]).int()
        _same_bytes(out["episode_outcomes"], want, "outcome partials")
    if "reward_terms" in out:
        _same_bytes(out["reward_terms"], torch.from_numpy(ro.warp_sums(terms.numpy(), n)), "reward term partials")
    if "obs_norm" in out:
        x = out.get("obs_clipped", obs)
        ok = R.bits_equal(out["obs_norm"], R.ref_normalize(x, out["obs_mean"], out["obs_var"]))
        assert bool(ok.all()), f"in-step normaliser: {int((~ok).sum())} elements differ"


@pytest.mark.parametrize("task", ["kick", "walk", "orient"])
def test_step_retry_matches_the_restatement_in_every_family(task):
    n = 4099
    kinds = _kinds(task, n)
    ref = {}
    for family in FAMILIES:
        env = _make_env(task, n, kinds)
        out = _step(env, family, kinds)
        _check_against_restatement(env, kinds, out)
        for key, t in out.items():                # every output the families share: the same bytes in all of them
            if key in ref:
                _same_bytes(t, ref[key], f"{family}: {key}")
            else:
                ref[key] = t
        del env
    # the north-star split: kick's parts 3 (bookkeeping + observation) + 4 (reward); walk / orient the same two launches
    env = _make_env(task, n, kinds, fusion="split")
    out = _step(env, "plain", kinds)
    _check_against_restatement(env, kinds, out)
    for key in ("rew", "reset", "progress", "timeout", "obs"):
        _same_bytes(out[key], ref[key], f"split: {key}")


@pytest.mark.parametrize("task", ["kick", "walk", "orient"])
def test_step_retry_on_the_l2_kernels(task):
    n = 262144
    kinds = _kinds(task, n)
    from torch.profiler import ProfilerActivity, profile
    for family in ("ep_terms_outcome", "ep_outcome_norm"):
        env = _make_env(task, n, kinds)
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            out = _step(env, family, kinds)
        names = {e.name for e in prof.events() if "task_tile" in e.name}
        if "B200" in torch.cuda.get_device_name(0):
            assert names and all("_l2_kernel" in x for x in names), names
        _check_against_restatement(env, kinds, out)
        del env


@pytest.mark.parametrize("task", ["kick", "walk", "orient"])
def test_ordinary_neighbours_of_a_retrying_env_keep_their_bytes(task):
    n = 4099
    kinds = _kinds(task, n)
    a = _step(_make_env(task, n, kinds), "ep_terms_outcome", kinds)
    b = _step(_make_env(task, n, torch.zeros_like(kinds)), "ep_terms_outcome", torch.zeros_like(kinds))
    warps = torch.nn.functional.pad((kinds != ORD).int(), (0, (-n) % WARP)).view(-1, WARP).any(1)
    near = torch.repeat_interleave(warps, WARP)[:n] & (kinds == ORD)
    assert int(near.sum()) >= 60
    for key in ("rew", "reset", "progress", "timeout", "obs", "shaped_rewards", "dones_u8", "episode_returns", "episode_lengths"):
        _same_bytes(a[key][near], b[key][near], key)


def _norm_case_stats(c):
    """Statistics of the normaliser cases: columns 20 / 21 / 22 variance 0 (their dof velocities are +-3e38 / +-inf), column 25
    variance inf, the rest ordinary."""
    mean, var = _norm_stats(c)
    var[20:23] = 0.0
    var[25] = float("inf")
    return mean, var


@pytest.mark.parametrize("task,clip", [("kick", None), ("walk", 5.0), ("orient", None), ("kick", 5.0)])
def test_in_step_normaliser_retry(task, clip):
    n = 4099
    kinds = _kinds(task, n)
    retry = kinds != ORD
    big = torch.tensor([3e38, float("-inf"), float("inf")], device="cuda")
    for family in ("ep_norm", "ep_outcome_norm"):
        env = _make_env(task, n, kinds, clip=clip)
        hook = env.sim.on_simulate

        def with_extremes(sim, hook=hook):
            hook(sim)
            dv = sim.dof_state.view(n, 18, 2)[..., 1]           # dof velocities 2:5 = observation columns 20:23
            r = retry.cuda()
            dv[:, 2:5] = torch.where(r.view(-1, 1), big, dv[:, 2:5])
            dv[1::2, 2] = torch.where(r[1::2], -3e38, dv[1::2, 2])
        env.sim.on_simulate = with_extremes
        mean, var = _norm_case_stats(env.num_obs)
        out = _step(env, family, kinds, norm_stats=(mean, var))
        x = out.get("obs_clipped", out["obs"])
        assert bool(torch.isinf(X.sqrt32(var[25].float() + X.c(1e-5))))
        want = R.ref_normalize(x, mean, var)
        if clip is None:
            assert X.outside_window((x[retry, 20] - X.c(float(mean[20]))) / X.sqrt32(X.c(1e-5))).all()
            assert bool((want[retry, 20:23].abs() == 5.0).all())
        assert bool((want[:, 25].abs() == 0).all())
        ok = R.bits_equal(out["obs_norm"], want)
        assert bool(ok.all()), f"{family}: {int((~ok).sum())} elements differ, rows {(~ok).any(1).nonzero().view(-1)[:8].tolist()}"
        _check_against_restatement(env, kinds, out)


# --------------------------------------------------------------------------------------------------------------- learner normalisers
def _special_rows(m, c, seed):
    """(m, c) fp32 ordinary rows with +-3e38 / +-inf in columns 3 / 4 of every 7th row and column 6 of every 5th row."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(m, c, generator=g) * 2
    x[::7, 3] = 3e38
    x[3::7, 3] = -3e38
    x[::7, 4] = float("inf")
    x[2::7, 4] = float("-inf")
    x[::5, 6] = -3e38
    return x


def _special_stats(c):
    g = torch.Generator().manual_seed(9)
    mean = torch.randn(c, generator=g, dtype=torch.float64)
    var = torch.rand(c, generator=g, dtype=torch.float64) + 0.5
    var[3] = var[4] = 0.0
    var[6] = 1e-3
    var[5] = float("inf")
    return mean, var


def _bits_ok(got, want, what):
    ok = R.bits_equal(got, want)
    assert bool(ok.all()), f"{what}: {int((~ok).sum())} of {ok.numel()} elements differ; first {(~ok).nonzero()[0].tolist()}"


@pytest.mark.parametrize("m,c", [(4099, 54), (1, 54), (4096, 52), (333, 7)])
def test_rms_normalize_retry(m, c):
    from bez_isaacgym_b200 import ops
    x = _special_rows(m, c, m)
    mean, var = _special_stats(c)
    den = X.sqrt32(var.float() + X.c(1e-5))
    assert X.outside_window((x[:, 3] - mean[3].float()) / den[3])[::7].all() and bool(torch.isinf(den[5]))
    g = Guarded()
    y = g.make((m, c))
    ops.rms_normalize(x.cuda(), mean.cuda(), var.cuda(), y)
    want = R.ref_normalize(x, mean, var)
    _bits_ok(y, want, "rms_normalize")
    if m > 1:
        assert bool((want[::7, 3] == 5).all()) and bool((want[:, 5] == 0).all())
    yu = g.make((m, c))
    ops.rms_normalize(x.cuda(), mean.cuda(), var.cuda(), yu, unnorm=True)
    _bits_ok(yu, R.ref_normalize(x, mean, var, unnorm=True), "rms_normalize unnorm")
    # slab view of time-major storage: rows t * E + (env - e0)
    T, N, e0, E = 4, 1100, 50, 1000
    st = torch.randn(T, N, c) * 2
    st[:, e0:e0 + E] = _special_rows(T * E, c, 7).view(T, E, c)
    ys = g.make((T * E, c))
    ops.rms_normalize_slabs(st.cuda()[:, e0:e0 + E], mean.cuda(), var.cuda(), ys)
    _bits_ok(ys, R.ref_normalize(st[:, e0:e0 + E].reshape(-1, c), mean, var), "rms_normalize_slabs")
    # the planned path: several minibatches, each with its own statistics, in one launch
    nb = 3
    seq = torch.stack([torch.stack([mean + b, var]) for b in range(nb)])
    ds = _special_rows(nb * 256, c, 11).cuda()
    yb = g.make((nb, 256, c))
    ops.rms_normalize_slabs_batched([ds[b * 256:(b + 1) * 256] for b in range(nb)], seq.cuda(), 0, yb)
    for b in range(nb):
        _bits_ok(yb[b], R.ref_normalize(ds[b * 256:(b + 1) * 256], seq[b, 0], seq[b, 1]), f"batched {b}")
    g.check()


def _huge_column(m, c, seed, col=5):
    """Ordinary rows with column ``col`` = +-1e20 alternating: the merged variance of that column is ~1e40, inf in fp32."""
    g = torch.Generator().manual_seed(seed)
    x = torch.randn(m, c, generator=g) * 2 + 1
    x[:, col] = torch.where(torch.arange(m) % 2 == 0, 1e20, -1e20)
    return x


@pytest.mark.parametrize("c", [1, 54])
def test_train_forward_retry(c):
    """c = 1: the cooperative fused_stats_kernel; c = 54: the chain ending in rms_merge_normalize_kernel."""
    from bez_isaacgym_b200 import ops
    m = 4099
    x = _huge_column(m, c, 5, col=0 if c == 1 else 5)
    g = Guarded()
    mean = g.make((c,), torch.float64, fill=torch.zeros(c, dtype=torch.float64, device="cuda"))
    var = g.make((c,), torch.float64, fill=torch.full((c,), 2.0, dtype=torch.float64, device="cuda"))
    count = g.make((1,), torch.float64, fill=torch.tensor([1000.0], dtype=torch.float64, device="cuda"))
    scratch = g.make((ops.rms_scratch_doubles(c),), torch.float64)
    y = g.make((m, c))
    ops.rms_train_forward(x.cuda().view(m) if c == 1 else x.cuda(), mean, var, count, y.view(m) if c == 1 else y, scratch)
    g.check()
    col = 0 if c == 1 else 5
    assert bool(torch.isinf(var.cpu().float()[col])) and X.outside_window(X.sqrt32(var.cpu().float()[col:col + 1] + X.c(1e-5))).all()
    want = R.ref_normalize(x, mean.cpu(), var.cpu())
    assert bool((want[:, col] == 0).all())
    _bits_ok(y, want, f"rms_train_forward c={c}")


def test_sharded_merge_normalize_retry():
    from bez_isaacgym_b200 import ops
    c = 54
    shards = [_huge_column(m, c, 20 + m) for m in (2048, 2051)]
    g = Guarded()
    mean = torch.zeros(c, dtype=torch.float64, device="cuda")
    var = torch.full((c,), 2.0, dtype=torch.float64, device="cuda")
    count = torch.tensor([1000.0], dtype=torch.float64, device="cuda")
    accs = []
    for x in shards:
        acc = torch.empty(2 + 4 * c, dtype=torch.float64, device="cuda")
        ops.rms_moments_ext(x.cuda(), mean, var, count, acc, torch.empty(ops.rms_scratch_doubles(c), dtype=torch.float64, device="cuda"))
        accs.append(acc)
    acc = accs[0].clone()
    acc[:1 + 2 * c] = accs[0][:1 + 2 * c] + accs[1][:1 + 2 * c]       # the all-reduce (SUM) of the heads
    for x in shards:
        rm, rv, rc = mean.clone(), var.clone(), count.clone()
        y = g.make((x.shape[0], c))
        ops.rms_merge_normalize(x.cuda(), acc, rm, rv, rc, y)
        assert bool(torch.isinf(rv.cpu().float()[5]))
        want = R.ref_normalize(x, rm.cpu(), rv.cpu())
        assert bool((want[:, 5] == 0).all())
        _bits_ok(y, want, "rms_merge_normalize")
    g.check()


# --------------------------------------------------------------------------------------------------------------- PPO loss / policy head
def _ppo_inputs(m, seed, bad_col=None, bad_row=None):
    g = torch.Generator().manual_seed(seed)
    mu = torch.randn(m, 18, generator=g) * 0.5
    logstd = torch.randn(18, generator=g) * 0.3 - 0.5
    if bad_col is not None:
        logstd[bad_col] = -90.0
    actions = mu + torch.randn(m, 18, generator=g) * 0.4
    if bad_col is not None:
        actions[::2, bad_col] = mu[::2, bad_col]                 # 0 / sigma: IEEE 0; the rest overflow to inf
    old_mu = mu + torch.randn(m, 18, generator=g) * 0.05
    old_sigma = torch.exp(logstd).expand(m, 18).clone() * (1 + 0.1 * torch.rand(m, 18, generator=g))
    if bad_col is not None:
        old_sigma[:, bad_col] = 1e-3                             # old / new sigma = 1.2e36: the KL stays finite in fp32
    if bad_row is not None:
        old_sigma[bad_row, 2] = 1.5e19
    values, old_values = torch.randn(m, generator=g), torch.randn(m, generator=g)
    returns, advantages = torch.randn(m, generator=g), torch.randn(m, generator=g)
    old_neglogp = torch.randn(m, generator=g) + 20
    return dict(actions=actions, mu=mu, logstd=logstd, old_mu=old_mu, old_sigma=old_sigma, values=values, old_values=old_values,
                returns=returns, old_neglogp=old_neglogp, advantages=advantages)


def _sigmas(logstd, m):
    """The per-row sigma the policy head writes (its expf), the divisor the kernels use."""
    from bez_isaacgym_b200 import ops
    sig = torch.empty(m, 18, device="cuda")
    ops.policy_head(torch.zeros(m, 18, device="cuda"), logstd.cuda(), noise=torch.zeros(m, 18, device="cuda"), sigmas=sig)
    return sig.cpu()


def _kl_mean(d, sigma):
    """torch_ext.policy_kl in float64 from the fp32 inputs: mean over rows of sum_j log(s1 / s0 + 1e-5) + (s0^2 + (m1 - m0)^2) /
    (2 (s1^2 + 1e-5)) - 0.5 with (m0, s0) the new and (m1, s1) the old policy."""
    s0, s1 = sigma.double(), d["old_sigma"].double()
    dm = d["old_mu"].double() - d["mu"].double()
    kl = torch.log(s1 / s0 + 1e-5) + (s0 * s0 + dm * dm) / (2 * (s1 * s1 + 1e-5)) - 0.5
    return kl.sum(1).mean()


@pytest.mark.parametrize("slabs", [False, True])
@pytest.mark.parametrize("case", ["bad_column", "bad_row"])
def test_ppo_loss_retry(case, slabs):
    from bez_isaacgym_b200 import ops
    m = 4099 if not slabs else 4 * 1000
    bad_col, bad_row = (4, None) if case == "bad_column" else (None, 1234)
    d = _ppo_inputs(m, 3, bad_col, bad_row)
    sigma = _sigmas(d["logstd"], m)
    if bad_col is not None:
        assert X.outside_window(sigma[:, bad_col]).all()
    else:
        os_ = d["old_sigma"][bad_row, 2]
        assert X.outside_window(X.c(2.0) * (os_ * os_ + X.c(1e-5)).view(1)).all()
    g = Guarded()
    stats = g.make((8,), torch.float64)
    nlp = g.make((m,))
    grad_mu, grad_values, grad_logstd = g.make((m, 18)), g.make((m,)), g.make((18,))
    partials = torch.empty(ops.ppo_scratch_doubles(), dtype=torch.float64, device="cuda")
    dev = {k: v.cuda() for k, v in d.items()}
    if slabs:
        T, N, e0, E = 4, 1100, 50, 1000

        def slab(t):
            st = torch.zeros((T, N) + tuple(t.shape[1:]), device="cuda")
            st[:, e0:e0 + E] = t.view((T, E) + tuple(t.shape[1:]))
            return st[:, e0:e0 + E]
        for k in ("actions", "old_mu", "old_sigma", "old_values", "returns", "old_neglogp", "advantages"):
            dev[k] = slab(dev[k])
        fn = ops.ppo_loss_slabs
    else:
        fn = ops.ppo_loss
    fn(dev["actions"], dev["mu"], dev["logstd"], dev["old_mu"], dev["old_sigma"], dev["values"], dev["old_values"], dev["returns"],
       dev["old_neglogp"], dev["advantages"], ops.make_ppo_cfg(), stats, partials, grad_mu=grad_mu, grad_values=grad_values,
       grad_logstd=grad_logstd, neglogp_out=nlp)
    g.check()
    want = X.neglogp(d["actions"], d["mu"], sigma, d["logstd"])
    _bits_ok(nlp, want, "neglogp")
    kl = _kl_mean(d, sigma)
    got = float(stats[5].cpu())
    assert (got != got) == bool(torch.isnan(kl)), (got, float(kl))
    if torch.isfinite(kl):
        assert abs(got - float(kl)) <= 1e-5 * abs(float(kl)) + 1e-6, (got, float(kl))
    else:
        assert got == float(kl), (got, float(kl))
    if case == "bad_row":
        assert torch.isfinite(stats.cpu()).all() and torch.isfinite(grad_mu.cpu()).all() and torch.isfinite(grad_logstd.cpu()).all()


def test_policy_head_retry():
    from bez_isaacgym_b200 import ops
    m = 4099
    g0 = torch.Generator().manual_seed(4)
    mu = torch.randn(m, 18, generator=g0) * 0.5
    logstd = torch.randn(18, generator=g0) * 0.3 - 0.5
    logstd[4] = -90.0
    noise = torch.randn(m, 18, generator=g0)
    noise[::3, 4] = 0.0                                         # action == mu: 0 / sigma
    g = Guarded()
    act, nlp, sig = g.make((m, 18)), g.make((m,)), g.make((m, 18))
    ops.policy_head(mu.cuda(), logstd.cuda(), noise=noise.cuda(), actions=act, neglogp=nlp, sigmas=sig)
    g.check()
    sig_c = sig.cpu()
    assert X.outside_window(sig_c[:, 4]).all() and bool((sig_c[:, 4] > 0).all())
    want = X.neglogp(act.cpu(), mu, sig_c, logstd)
    assert not torch.isnan(want).any()
    _bits_ok(nlp, want, "policy head neglogp")
    # Philox noise (no noise tensor): the same restatement from the sampled actions
    nlp2, act2, sig2 = g.make((m,)), g.make((m, 18)), g.make((m, 18))
    ops.policy_head(mu.cuda(), logstd.cuda(), seed=7, step=3, actions=act2, neglogp=nlp2, sigmas=sig2)
    g.check()
    _bits_ok(nlp2, X.neglogp(act2.cpu(), mu, sig2.cpu(), logstd), "policy head neglogp (Philox)")
