"""GPU: the unaligned memory paths of the hot-path kernels.  The fused step, the policy head, the DR noise pass,
``swap_and_flatten01`` and ``quat_rotate`` pick their loads and stores from pointer alignment at launch; training reaches the
unaligned ones without asking (an obs row is 216 B and an action row 72 B, so at an odd env count every odd experience slot
starts at 8 mod 16).  Every case here

* places the buffers at a byte residue mod 16 with ``_util.Guarded`` (stores past a row or a buffer hit a guard band),
* asserts the alignment clause that routes the launch to its fallback,
* compares every output with the same call on fresh aligned tensors from clones of the same state, bit for bit (NaN equal
  to NaN) -- the aligned path is pinned to ``oracle/`` elsewhere -- and, once per task, with the oracle or the reference's
  goldens directly."""
import math

import numpy as np
import pytest
import torch

from bez_isaacgym_b200 import bez_model as bm
from bez_isaacgym_b200 import synthetic_gym as sg
from tests import _util as U

pytestmark = pytest.mark.gpu


def _ops():
    from bez_isaacgym_b200 import ops
    return ops


def _same(a, b):
    if a.dtype.is_floating_point:
        return a.shape == b.shape and bool(((a == b) | (a.isnan() & b.isnan())).all())
    return torch.equal(a, b)


def _res(t):
    return t.data_ptr() % 16


def _assert_same(got, want, what=""):
    for k in want:
        assert _same(got[k], want[k]), f"{what}: {k} differs from the aligned call"


# ============================================================================================ 1. the fused step
N = 4099                                     # 128 full warps and a 3-env tail
MAX_LEN = 900


def _inputs(task, cleats, n, seed=17, clip=math.inf):
    """CPU tensors of one step: simulator state, carried state, outputs pre-filled with sentinels."""
    st = sg.make_state(n, seed=seed, task=task, cleats=cleats, filler=n < 100000)
    g = torch.Generator().manual_seed(seed)
    width = bm.task_dims(task)[2]
    progress = torch.randint(0, MAX_LEN, (n,), generator=g)
    progress = torch.where(torch.rand(n, generator=g) < 0.25, torch.randint(MAX_LEN - 3, MAX_LEN, (n,), generator=g), progress)
    t = dict(dof_state=st.dof_state, rigid_body=st.rigid_body, root_states=st.root_states, net_contact=st.net_contact,
             initial_root_states=sg.make_initial_root_states(n, task=task),
             prev_lin_vel=0.3 * torch.randn(n, 3, generator=g),
             reset_buf=(torch.rand(n, generator=g) < 0.05).long(), progress_buf=progress,
             timeout_buf=torch.full((n,), -1, dtype=torch.long), randomize_buf=torch.randint(0, 9, (n,), generator=g),
             obs=torch.full((n, width), float("nan")), obs_clipped=torch.full((n, width), float("nan")),
             rew=torch.full((n,), float("nan")), values=torch.randn(n, generator=g),
             shaped_rewards=torch.full((n,), float("nan")), dones_u8=torch.full((n,), 0xAB, dtype=torch.uint8),
             episode_returns=torch.randn(n, generator=g), episode_lengths=torch.randint(0, 50, (n,), generator=g).float(),
             obs_mean=torch.randn(width, generator=g, dtype=torch.float64), obs_var=torch.rand(width, generator=g, dtype=torch.float64) + 0.1,
             obs_norm=torch.full((n, width), float("nan")))
    w = (n + 31) // 32
    t["episode_partials"] = torch.full((3, w), float("nan"), dtype=torch.float64)
    t["outcome_partials"] = torch.full((5 if task == "kick" else 4, w), -1, dtype=torch.int32)
    t["term_partials"] = torch.full((6 if task == "kick" else 5, w), float("nan"), dtype=torch.float64)
    # a few envs of the rarest outcome classes: the ball beyond the goal (kick: wide) and the robot beyond its goal (walk: out)
    rare = torch.rand(n, generator=g) < 0.02
    if task == "kick":
        goal, ball_init, _, _, _ = sg.make_constants(n)
        ball = st.root_states.view(n, 2, 13)[:, 1]
        ball[:, 0] = torch.where(rare, 1.8 + 0.2 * torch.rand(n, generator=g), ball[:, 0])
        t.update(goal=goal, ball_init=ball_init)
    else:
        bez = st.root_states.view(n, 13)[:, 0:2]
        t["goal"] = torch.where(rare.unsqueeze(1), 0.5 * bez, torch.tensor([2.0, 0.0]).expand(n, 2))
        if task == "orient":
            t["goal_angle"] = 1.5708 + 0.02 * torch.randn(n, generator=g)
    cfg = _ops().make_task_cfg(num_bodies=st.num_bodies, cleats=cleats, max_episode_length=MAX_LEN, clip_obs=clip)
    return t, cfg


def _place(t, G, offsets):
    return {k: G.make(tuple(v.shape), v.dtype, fill=v.cuda(), offset=offsets.get(k, 0)) for k, v in t.items()}


def _launch(fam, task, b, cfg, step=3, env_base=0, lo=0, hi=None):
    """One launch of family ``fam`` on the buffers ``b`` (envs [lo, hi) when chunked, Philox keyed from ``env_base``)."""
    ops = _ops()
    hi = b["progress_buf"].shape[0] if hi is None else hi
    actors = bm.task_dims(task)[0]
    s = {k: (v if k in ("obs_mean", "obs_var") or k.endswith("_partials") else v.view(-1, *v.shape[1:])) for k, v in b.items()}
    rows = lambda k, per=1: s[k][lo * per:hi * per]          # noqa: E731
    sl = dict(dof_state=rows("dof_state", 18), rigid_body=rows("rigid_body", cfg.num_bodies), root_states=rows("root_states", actors),
              net_contact=rows("net_contact", cfg.num_bodies), initial_root_states=rows("initial_root_states", actors))
    for k in ("prev_lin_vel", "reset_buf", "progress_buf", "timeout_buf", "randomize_buf", "obs", "obs_clipped", "rew", "values",
              "shaped_rewards", "dones_u8", "episode_returns", "episode_lengths", "obs_norm", "goal", "goal_angle", "ball_init"):
        if k in s:
            sl[k] = rows(k)
    clip = None if math.isinf(cfg.clip_obs) else sl["obs_clipped"]
    pos = (task, sl["dof_state"], sl["rigid_body"], sl["root_states"], sl["net_contact"], sl["goal"], sl["initial_root_states"],
           sl["reset_buf"], sl["progress_buf"], sl["timeout_buf"], cfg, sl["obs"], sl["rew"])
    kw = dict(goal_angle=sl.get("goal_angle"), ball_init=sl.get("ball_init"), prev_lin_vel=sl["prev_lin_vel"], seed=11, step=step,
              randomize_buf=sl["randomize_buf"], obs_clipped=clip)
    if fam.startswith("parts"):
        p = int(fam[5:])
        if task == "kick":
            ops.post_physics(*pos[1:6], sl["ball_init"], *pos[6:], prev_lin_vel=sl["prev_lin_vel"], seed=11, step=step,
                             randomize_buf=sl["randomize_buf"], obs_clipped=clip, parts=p)
        else:
            ops.post_physics_task(*pos, goal_angle=sl.get("goal_angle"), prev_lin_vel=sl["prev_lin_vel"], seed=11, step=step,
                                  randomize_buf=sl["randomize_buf"], obs_clipped=clip, parts=p)
        return
    kw.update(rollout_cfg=ops.make_rollout_cfg(), values=sl["values"], shaped_rewards=sl["shaped_rewards"], dones_u8=sl["dones_u8"],
              env_base=env_base)
    if fam == "rollout":
        return ops.post_physics_rollout(*pos, **kw)
    ep = (sl["episode_returns"], sl["episode_lengths"], s["episode_partials"])
    if fam == "ep":
        ops.post_physics_rollout_ep(*pos, *ep, **kw)
    elif fam == "ep_norm":
        ops.post_physics_rollout_ep_norm(*pos, *ep, s["obs_mean"], s["obs_var"], sl["obs_norm"], **kw)
    elif fam in ("ep_outcome", "ep_norm_outcome"):
        norm = dict(obs_mean=s["obs_mean"], obs_var=s["obs_var"], obs_norm=sl["obs_norm"]) if "norm" in fam else {}
        ops.post_physics_rollout_ep_outcome(*pos, *ep, s["outcome_partials"], **norm, **kw)
    elif fam in ("ep_terms", "ep_outcome_terms"):
        oc = s["outcome_partials"] if "outcome" in fam else None
        ops.post_physics_rollout_ep_terms(*pos, *ep, s["term_partials"], outcome_partials=oc, **kw)
    else:
        raise ValueError(fam)


def _run(fam, task, cleats, t, cfg, offsets=None, chunk=None):
    G = U.Guarded()
    b = _place(t, G, offsets or {})
    if chunk is None:
        _launch(fam, task, b, cfg)
    else:                                    # two launches, the second starting at env `chunk` with pointers offset to it
        _launch(fam, task, b, cfg, env_base=0, lo=0, hi=chunk)
        _launch(fam, task, b, cfg, env_base=chunk, lo=chunk)
    G.check()
    return b, {k: v.cpu() for k, v in b.items()}


def _use_tma(b):
    return all(_res(b[k]) == 0 for k in ("dof_state", "root_states", "obs", "obs_clipped"))


FAMILIES = ["rollout", "ep", "ep_outcome", "ep_terms", "ep_outcome_terms", "ep_norm", "ep_norm_outcome"]
PARTS = {"kick": [1, 2, 3, 4, 5, 6], "walk": [2, 3, 4], "orient": [2, 3, 4]}
TASKS = [("kick", False), ("kick", True), ("walk", False), ("orient", False)]
TRIGGERS = [(task, cleats, trig) for task, cleats in TASKS for trig in ("obs", "obs_clipped", "chunk", "rb4", "rb8", "cf4")
            if not (trig == "rb8" and task == "kick") and not (trig == "cf4" and (task != "kick" or cleats))]


@pytest.mark.parametrize("task,cleats,trigger", TRIGGERS)
def test_fused_step_on_unaligned_buffers_equals_the_aligned_step(task, cleats, trigger):
    """(a) obs at +8 (the odd-N slot); (b) obs_clipped at +8 with a finite clip_obs; (c) a second launch starting at an odd
    env (root_states / obs at +8 for kick, root_states at +4 for walk / orient); (d) rigid_body at +4 / +8: the scalar IMU
    gather; (e) net_contact at +4: the scalar foot gather and the in-place contact filter."""
    clip = 1.5 if trigger == "obs_clipped" else math.inf
    t, cfg = _inputs(task, cleats, N, clip=clip)
    assert 0 < int(t["reset_buf"][:4096].sum()), "resets inside full warps: the reset write-back runs in a full warp"
    offsets = {"obs": {"obs": 8}, "obs_clipped": {"obs_clipped": 8}, "rb4": {"rigid_body": 4}, "rb8": {"rigid_body": 8},
               "cf4": {"net_contact": 4}}.get(trigger, {})
    chunk = 1281 if trigger == "chunk" else None
    fams = FAMILIES + [f"parts{p}" for p in PARTS[task]] if chunk is None else ["rollout"]
    seen = None
    for fam in fams:
        ref_b, want = _run(fam, task, cleats, t, cfg)
        assert _use_tma(ref_b) and _res(ref_b["rigid_body"]) == 0 and _res(ref_b["net_contact"]) == 0
        b, got = _run(fam, task, cleats, t, cfg, offsets, chunk)
        # the precondition that routes this launch to its fallback
        if trigger in ("obs", "obs_clipped"):
            assert _res(b[trigger]) == 8 and not _use_tma(b)
        elif trigger == "chunk":
            root = b["root_states"].view(N, -1)[chunk]
            assert chunk % 2 == 1 and _res(root) == (8 if task == "kick" else 4)
            if task == "kick":
                assert _res(b["obs"][chunk]) == 8
        elif trigger.startswith("rb"):
            # rb_vec2 needs an 8-byte aligned base, an even row stride and offset; rb_win (walk / orient) a 16-byte aligned base
            stride = cfg.num_bodies * 13
            assert _res(b["rigid_body"]) == int(trigger[2:])
            assert not (b["rigid_body"].data_ptr() % 8 == 0 and stride % 2 == 0)
        else:
            assert _res(b["net_contact"]) == 4 and b["net_contact"].data_ptr() % 8 != 0      # cf_vec2 off
        _assert_same(got, want, f"{task} cleats={cleats} {trigger} {fam}")
        if "outcome" in fam:
            seen = want["outcome_partials"].sum(1)
        if fam == "rollout":
            assert int(want["dones_u8"].sum()) > 0
    if seen is not None:
        assert bool((seen > 0).all()), f"done envs of every outcome class: {seen.tolist()}"


def test_large_kick_with_obs_at_8_runs_the_l2_kernel_and_equals_the_aligned_step():
    from torch.profiler import ProfilerActivity, profile
    n = 262145
    t, cfg = _inputs("kick", False, n, seed=5)
    _, want = _run("ep", "kick", False, t, cfg)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        b, got = _run("ep", "kick", False, t, cfg, {"obs": 8})
    assert _res(b["obs"]) == 8 and not _use_tma(b)
    names = [e.name for e in prof.events() if "task_tile" in e.name]
    if "B200" in torch.cuda.get_device_name(0):
        assert any("_l2_kernel" in s for s in names), names
    _assert_same(got, want, "262145 kick envs, obs at +8")


def test_unaligned_kick_step_matches_the_reference_goldens():
    """The observation and reward kernels with obs at +8, rigid_body and net_contact at +4 against the reference's own
    functions (``fn_n257.npz``), with the tolerances of ``test_golden_gpu``."""
    from tests.test_oracle_pinning import _eq, _load, _state
    ops = _ops()
    g = _load("fn_n257.npz")
    st = _state(g)
    n = st.num_envs
    goal, ball_init, default, _, _ = U.constants(n)
    cfg = ops.make_task_cfg(num_bodies=st.num_bodies)
    G = U.Guarded()
    rb = G.make(st.rigid_body.shape, fill=st.rigid_body.cuda(), offset=4)
    cf = G.make(st.net_contact.shape, fill=st.net_contact.cuda(), offset=4)
    obs = G.make((n, 54), fill=torch.full((n, 54), float("nan")), offset=8)
    rew = G.make((n,), offset=4)
    reset = G.make((n,), torch.long, offset=8)
    prev = g["in_prev_lin_vel"].cuda().contiguous()
    assert _res(obs) == 8 and rb.data_ptr() % 8 and cf.data_ptr() % 8
    ops.compute_observations(st.dof_state.cuda(), rb, st.root_states.cuda(), cf, goal.cuda(), ball_init.cuda(), cfg, obs, prev_lin_vel=prev)
    ops.compute_reward(st.dof_state.cuda(), rb, st.root_states.cuda(), goal.cuda(), ball_init.cuda(), g["in_reset"].cuda(),
                       g["in_progress"].cuda(), cfg, rew, reset)
    G.check()
    got, want = obs.cpu(), g["ref_obs"]
    assert _eq(got[:, 0:36], want[:, 0:36]) and _eq(got[:, 39:42], want[:, 39:42]) and _eq(got[:, 44:54], want[:, 44:54])
    assert _eq(cf.cpu(), g["ref_net_contact_after"]), "in-place contact filter"
    U.assert_close(got[:, 36:39], want[:, 36:39], scale=U.imu_term_scale(st, g["in_prev_lin_vel"]), what="imu lin_acc")
    U.assert_close(got[:, 42:44], want[:, 42:44], what="off_orn")
    band = U.reward_tie_band(st, goal, ball_init)
    assert not bool(((reset.cpu() != g["ref_reset"]) & ~band).any())
    U.assert_close(rew.cpu()[~band], g["ref_rew"][~band], scale=U.reward_scale(st, goal, ball_init, default)[~band], what="reward")


@pytest.mark.parametrize("task", ["walk", "orient"])
def test_unaligned_sibling_step_matches_the_reference_goldens(task):
    """WalkEnv / OrientEnv kernels with obs at +8 and rigid_body at +4 against ``fn_{task}_n257.npz``."""
    from tests.test_oracle_pinning import _load, _sibling_state
    from tests.test_sibling_tasks_gpu import _check
    ops = _ops()
    g = _load(f"fn_{task}_n257.npz")
    st = _sibling_state(g)
    n = st.num_envs
    cfg = ops.make_task_cfg(num_bodies=st.num_bodies, max_episode_length=600, cleats=st.num_bodies > 21)
    G = U.Guarded()
    rb = G.make(st.rigid_body.shape, fill=st.rigid_body.cuda(), offset=4)
    cf = G.make(st.net_contact.shape, fill=st.net_contact.cuda(), offset=4)
    obs = G.make((n, 52), fill=torch.full((n, 52), float("nan")), offset=8)
    rew = G.make((n,), offset=4)
    reset = G.make((n,), torch.long, fill=g["in_reset"].cuda(), offset=8)
    gl = g["in_goal"].cuda().contiguous()
    ga = torch.full((n,), 1.5708, device="cuda")
    p = g["in_prev_lin_vel"].cuda().contiguous()
    assert _res(obs) == 8 and _res(rb) == 4
    d = st.to("cuda")
    ops.post_physics_task(task, d.dof_state, rb, d.root_states, cf, gl, None, None, None, None, cfg, obs, None, goal_angle=ga,
                          prev_lin_vel=p, parts=2)
    ops.post_physics_task(task, d.dof_state, rb, d.root_states, None, gl, None, reset, g["in_progress"].cuda(), None, cfg, None, rew,
                          goal_angle=ga, parts=4)
    G.check()
    _check(task, st, g["in_prev_lin_vel"], g["in_goal"], (obs.cpu(), rew.cpu(), reset.cpu(), cf.cpu(), p.cpu()), g["ref_obs"],
           g["ref_rew"], g["ref_reset"], g["ref_net_contact_after"])


# ============================================================================================ 2. training at an odd env count
def _train_env(task, n, randomize):
    from bez_isaacgym_b200 import tasks
    from bez_isaacgym_b200.synthetic_sim import SyntheticGym
    from tests.test_outcomes_gpu import _mover
    cls = {"kick": tasks.KickEnv, "walk": tasks.WalkEnv}[task]
    cfg = bm.default_task_cfg(n, task=task)
    cfg["seed"] = 3
    if randomize:
        cfg["task"] = {"randomize": True, "randomization_params": {
            "frequency": 1, "observations": {"range": [0, .05], "operation": "additive", "distribution": "gaussian"}}}
    mv = _mover(3)
    env = cls(cfg, "cuda:0", 0, True, sim=SyntheticGym(n, device="cuda:0", seed=3, on_simulate=mv, task=task))
    m = env.max_episode_length
    env.progress_buf.copy_(torch.randint(int(m) - 6, int(m), (n,), generator=torch.Generator().manual_seed(3)).cuda())
    return env


@pytest.mark.parametrize("task,randomize", [("kick", False), ("walk", False), ("kick", True)])
def test_rollout_into_odd_env_count_experience_slots_equals_fresh_tensors(task, randomize):
    """N = 1025, T = 8: the env and the policy head write the slots of an ExperienceBuffer (odd slots at +8); a twin env and a
    twin head with the same state, inputs and seeds write fresh aligned tensors.  Every output, every step, bit for bit."""
    from bez_isaacgym_b200.learner import experience as ex
    from bez_isaacgym_b200.learner.policy_head import policy_head

    class Box:
        def __init__(self, k):
            self.shape = (k,)
    n, T = 1025, 8
    envs = [_train_env(task, n, randomize), _train_env(task, n, randomize)]
    if randomize:
        assert set(envs[0].dr_randomizations) == {"observations"}
    width = envs[0]._obs_width
    buf = ex.ExperienceBuffer(dict(observation_space=Box(width), action_space=Box(18)), dict(num_actors=n, horizon_length=T), "cuda")
    shaped = torch.zeros(T, n, 1, device="cuda")
    ep = [(torch.zeros(n, device="cuda"), torch.zeros(n, device="cuda"), torch.zeros(T, 3, (n + 31) // 32, dtype=torch.float64,
                                                                                     device="cuda")) for _ in envs]
    g = torch.Generator(device="cuda").manual_seed(9)
    logstd = 0.2 * torch.randn(18, device="cuda", generator=g)
    last_obs = torch.empty(n, width, device="cuda")
    dones = 0
    for t in range(T):
        mu = 0.6 * torch.randn(n, 18, device="cuda", generator=g)
        value = torch.randn(n, 1, device="cuda", generator=g)
        # slot t starts t * n rows in: at n = 1025 an odd slot of 72 B action rows (216 B kick obs rows) is at +8, of 4 B rows at +4
        for k, row in (("obses", 4 * width), ("actions", 72), ("mus", 72), ("sigmas", 72), ("values", 4), ("neglogpacs", 4)):
            assert _res(buf.slot(k, t)) == (t * n * row) % 16, (k, t)
        if t % 2:
            assert _res(buf.slot("actions", t)) == 8 and (task != "kick" or _res(buf.slot("obses", t)) == 8)
        res = [policy_head(mu, logstd, value, experience=buf, t=t, seed=21, step=t, env=envs[0]),
               policy_head(mu, logstd, value, seed=21, step=t, env=envs[1])]
        for k in ("actions", "neglogpacs", "values", "mus", "sigmas", "env_actions"):
            assert _same(res[0][k], res[1][k]), (t, k)
        assert _same(envs[0].targets, envs[1].targets), t
        outs = [(buf.slot("obses", t + 1) if t + 1 < T else last_obs, shaped[t],
                 buf.slot("dones", t + 1) if t + 1 < T else torch.empty(n, dtype=torch.uint8, device="cuda")),
                (torch.empty(n, width, device="cuda"), torch.empty(n, 1, device="cuda"), torch.empty(n, dtype=torch.uint8, device="cuda"))]
        if t + 1 < T:
            assert _res(outs[0][0]) == ((t + 1) * n * 4 * width) % 16
        for env, r, (o, sh, d), (ret, length, part) in zip(envs, res, outs, ep):
            env.set_obs_target(o)
            env.set_rollout_targets(values=r["values"], shaped_rewards=sh, dones_u8=d, episode_returns=ret, episode_lengths=length,
                                    episode_partials=part[t])
            env.step_precomputed_targets(r["env_actions"])
        for a, b in zip(outs[0], outs[1]):
            assert _same(a.view(b.shape), b), t
        for name in ("rew_buf", "reset_buf", "progress_buf", "timeout_buf", "dof_state", "root_states", "net_contact"):
            assert _same(getattr(envs[0], name), getattr(envs[1], name)), (t, name)
        dones += int(envs[0].reset_buf.sum())
    for a, b in zip(ep[0], ep[1]):
        assert _same(a, b)
    assert dones > 0
    torch.cuda.synchronize()


def test_slab_minibatches_at_odd_env_offsets_equal_the_aligned_slab_and_the_oracle():
    """minibatch_size = 8 * 41 on 1025 envs: E = 41, so minibatch 1 starts at env 41 (obs and action rows at +8, values at +4).
    RunningMeanStd train forward and the PPO loss on those slab views equal, bit for bit, the same calls on an aligned copy of
    the storage with the same slab geometry (its minibatch starts at env 42 of 1026), and the oracle within the tolerances of
    ``test_slab_normalize_and_moments_match_flattened_minibatch`` / ``test_slab_ppo_loss_matches_flattened_minibatch``."""
    from bez_isaacgym_b200.learner import experience as ex
    from oracle import rl_games_oracle as rg
    from tests.test_rollout_gpu import _rollout
    ops = _ops()

    class Box:
        def __init__(self, k):
            self.shape = (k,)
    T, n, mb = 8, 1025, 8 * 41
    ro = _rollout(T, n, seed=13)
    buf = ex.ExperienceBuffer(dict(observation_space=Box(54), action_space=Box(18)), dict(num_actors=n, horizon_length=T), "cuda")
    for k in ("obses", "actions", "mus", "sigmas", "values", "neglogpacs"):
        buf.tensor_dict[k].copy_(ro[k].cuda())
    extra = dict(returns=ro["returns"].cuda(), advantages=ro["advantages"].cuda())
    sds = ex.SlabDataset(buf, mb, extra=extra)
    E = sds.envs_per_batch
    i = 1
    v = sds[i]
    assert E % 2 == 1 and _res(v["obses"]) == 8 and _res(v["actions"]) == 8 and _res(v["values"]) == 4
    # the twin: one env column in front of the storage shifts minibatch 1 to env 42, where every row starts 16-byte aligned
    twin = {}
    for k, t in v.items():
        full = sds.tensors[k]
        pad = torch.zeros((T, n + 1) + tuple(full.shape[2:]), dtype=full.dtype, device="cuda")
        pad[:, 1:] = full
        twin[k] = pad[:, i * E + 1:(i + 1) * E + 1]
    assert _res(twin["obses"]) == 0 and _res(twin["actions"]) == 0
    outs = []
    for src in (v, twin):
        mean = torch.zeros(54, dtype=torch.float64, device="cuda"); var = torch.ones(54, dtype=torch.float64, device="cuda")
        count = torch.ones(1, dtype=torch.float64, device="cuda")
        y = torch.empty(T * E, 54, device="cuda")
        ops.rms_train_forward(src["obses"], mean, var, count, y,
                              torch.empty(ops.rms_scratch_doubles(54), dtype=torch.float64, device="cuda"))
        outs.append((mean, var, count, y))
    for a, b in zip(*outs):
        assert _same(a, b)
    perm = sds.permutation_to_env_major()
    flat = {k: rg.swap_and_flatten01(t)[i * mb:(i + 1) * mb] for k, t in ro.items()}
    rms = rg.RunningMeanStd(54)
    want_y = rms(flat["obses"])
    torch.testing.assert_close(outs[0][0].cpu(), rms.running_mean, rtol=2e-6, atol=1e-7)
    torch.testing.assert_close(outs[0][1].cpu(), rms.running_var, rtol=2e-5, atol=1e-7)
    U.assert_close(outs[0][3].cpu()[perm], want_y, rtol=2e-5, atol=2e-6, what="normalised minibatch")
    # PPO loss
    g = torch.Generator().manual_seed(5)
    logstd = torch.randn(18, generator=g) * 0.1
    mu_new = (flat["mus"] + 0.05 * torch.randn(mb, 18, generator=g)).requires_grad_(True)
    val_new = (flat["values"] + 0.1 * torch.randn(mb, 1, generator=g)).requires_grad_(True)
    logstd_p = logstd.clone().requires_grad_(True)
    out = rg.ppo_loss(dict(mu=mu_new, logstd=logstd_p, values=val_new, actions=flat["actions"], old_mu=flat["mus"],
                           old_sigma=flat["sigmas"], old_values=flat["values"], returns=flat["returns"],
                           old_neglogp=flat["neglogpacs"], advantages=flat["advantages"]), bound_form="outside")
    out["loss"].backward()
    inv = torch.empty_like(perm); inv[perm] = torch.arange(mb)
    mu_slab = mu_new.detach()[inv].contiguous().cuda()
    val_slab = val_new.detach().view(-1)[inv].contiguous().cuda()
    cfg = ops.make_ppo_cfg(bound_form="outside")
    part = torch.empty(ops.ppo_scratch_doubles(), dtype=torch.float64, device="cuda")
    res = []
    for src in (v, twin):
        stats = torch.empty(8, dtype=torch.float64, device="cuda")
        gmu = torch.empty(mb, 18, device="cuda"); gv = torch.empty(mb, device="cuda"); gls = torch.empty(18, device="cuda")
        nlp = torch.empty(mb, device="cuda")
        ops.ppo_loss_slabs(src["actions"], mu_slab, logstd.cuda(), src["mus"], src["sigmas"], val_slab, src["values"], src["returns"],
                           src["neglogpacs"], src["advantages"], cfg, stats, part, grad_mu=gmu, grad_values=gv, grad_logstd=gls,
                           neglogp_out=nlp)
        res.append((stats, gmu, gv, gls, nlp))
    for a, b in zip(*res):
        assert _same(a, b)
    s = res[0][0].cpu()
    for k, idx in (("loss", 0), ("a_loss", 1), ("c_loss", 2), ("entropy", 3), ("b_loss", 4), ("kl", 5)):
        assert math.isclose(float(s[idx]), float(out[k]), rel_tol=2e-5, abs_tol=2e-6), (k, float(s[idx]), float(out[k]))
    U.assert_close(res[0][4].cpu()[perm], out["neglogp"].detach(), rtol=2e-5, atol=2e-5, what="neglogp")
    U.assert_close(res[0][1].cpu()[perm], mu_new.grad, rtol=2e-4, atol=2e-9, what="grad_mu")
    U.assert_close(res[0][2].cpu()[perm], val_new.grad.view(-1), rtol=2e-4, atol=2e-9, what="grad_values")
    U.assert_close(res[0][3].cpu(), logstd_p.grad, rtol=2e-4, atol=2e-7, what="grad_logstd")


# ============================================================================================ 3. kernels called directly
@pytest.mark.parametrize("n", [4099, 128 * 33])
@pytest.mark.parametrize("philox", [False, True])
def test_policy_head_on_unaligned_slots_equals_the_aligned_call_and_the_oracle(n, philox):
    from oracle import rl_games_oracle as rg
    from oracle import task_oracle as to
    ops = _ops()
    g = torch.Generator().manual_seed(n + philox)
    mu = torch.randn(n, 18, generator=g) * 0.8
    logstd = torch.randn(18, generator=g) * 0.3
    vnorm = torch.randn(n, generator=g) * 3
    noise = ops.normal_noise(5, 6, torch.empty(n, 18, device="cuda")) if philox else torch.randn(n, 18, generator=g).cuda()
    mean, var = torch.tensor([0.37], dtype=torch.float64), torch.tensor([2.5], dtype=torch.float64)
    cfg = ops.make_task_cfg()
    wide, narrow = ("actions", "mus", "sigmas", "env_actions", "targets"), ("neglogp", "values")
    runs = []
    for off_w, off_n in ((0, 0), (8, 4)):
        G = U.Guarded()
        o = {k: G.make((n, 18), fill=torch.full((n, 18), float("nan")), offset=off_w) for k in wide}
        o.update({k: G.make((n,), fill=torch.full((n,), float("nan")), offset=off_n) for k in narrow})
        nz = None if philox else G.make((n, 18), fill=noise, offset=off_w)
        if off_w:                            # launch_policy_head: use_tma needs every row pointer 16-byte aligned
            assert all(_res(o[k]) == 8 for k in wide) and all(_res(o[k]) == 4 for k in narrow) and (philox or _res(nz) == 8)
        ops.policy_head(mu.cuda(), logstd.cuda(), vnorm.cuda(), mean.cuda(), var.cuda(), 1e-5, noise=nz, seed=5, step=6, task_cfg=cfg,
                        **o)
        G.check()
        runs.append({k: v.cpu() for k, v in o.items()})
    _assert_same(runs[1], runs[0], "policy head")
    vr = rg.RunningMeanStd(1)
    vr.running_mean, vr.running_var = mean, var
    want = rg.policy_head(mu, logstd, vnorm.view(-1, 1), vr, noise.cpu())
    env_act = rg.preprocess_actions(want["actions"])
    _, _, default, lower, upper = sg.make_constants(n)
    _, want_targets = to.pre_physics(env_act, default, lower, upper, clip_actions=3.9)
    got = runs[1]
    assert torch.equal(got["mus"], mu)
    U.assert_close(got["sigmas"], want["sigmas"], what="sigmas")
    U.assert_close(got["actions"], want["actions"], what="actions")
    U.assert_close(got["neglogp"], want["neglogpacs"], rtol=2e-5, atol=2e-5, what="neglogp")
    U.assert_close(got["values"], want["values"].view(-1), what="values")
    U.assert_close(got["env_actions"], env_act, what="env actions")
    U.assert_close(got["targets"], want_targets, what="targets")


DR_NAMES = ("x", "corr", "white", "y", "y_clip")


@pytest.mark.parametrize("dist,op", [("gaussian", "additive"), ("gaussian", "scaling"), ("uniform", "additive"), ("uniform", "scaling")])
@pytest.mark.parametrize("philox", [False, True])
def test_dr_noise_on_unaligned_buffers_equals_the_aligned_call(dist, op, philox):
    """Every buffer at +4 / +8 / +12 alone, then all together, on totals = 0, 1, 2, 3 (mod 4): the scalar quad path with
    all four elements present and with the ragged tail.  The Philox draw is keyed by the quad index: alignment changes no bit."""
    ops = _ops()
    cfg = ops.make_noise_cfg(dist, op, a=0.3, b=0.9 if op == "scaling" else 0.05, a_corr=0.2, b_corr=0.1)
    names = [k for k in DR_NAMES if not (philox and k == "white")]
    places = [{k: r} for k in names for r in (4, 8, 12)] + [{k: r for k in names} for r in (4, 8, 12)]
    for total in (4100, 4101, 4102, 4103):
        g = torch.Generator().manual_seed(total)
        src = dict(x=torch.randn(total, generator=g), corr=torch.randn(total, generator=g),
                   white=torch.randn(total, generator=g) if dist == "gaussian" else torch.rand(total, generator=g),
                   y=torch.full((total,), float("nan")), y_clip=torch.full((total,), float("nan")))
        want = None
        for place in [{}] + places:
            G = U.Guarded()
            b = {k: G.make((total,), fill=src[k].cuda(), offset=place.get(k, 0)) for k in DR_NAMES}
            assert all(_res(b[k]) == place.get(k, 0) for k in DR_NAMES)
            ops.dr_noise(b["x"], cfg, corr=b["corr"], white=None if philox else b["white"], seed=(7 << 32) + 3, step=(5 << 32) + 11,
                         out=b["y"], out_clipped=b["y_clip"], clip=0.7)
            G.check()
            got = {k: b[k].cpu() for k in ("y", "y_clip")}
            if want is None:
                want = got
            else:
                _assert_same(got, want, f"dr_noise total={total} {place}")


def _dr_fill_reference(seed, step, total, dist):
    """numpy restatement of ``dr_fill``: quad q draws Philox4x32-10 with ctr = (q_lo, q_hi, step_lo, step_hi) and key =
    (seed_lo ^ 0x2545F491, seed_hi); uniform: (x >> 8) * 2^-24 per word; gaussian: Box-Muller on the word pairs (x, y) and
    (z, w), each giving (r cos 2 pi u2, r sin 2 pi u2) with u1 = ((a >> 8) + 1) * 2^-24, u2 = (b >> 8) * 2^-24."""
    from oracle.philox_ref import philox4x32_10
    q = np.arange((total + 3) // 4, dtype=np.uint64)
    ctr = np.zeros((q.size, 4), dtype=np.uint32)
    ctr[:, 0] = (q & np.uint64(0xFFFFFFFF)).astype(np.uint32)
    ctr[:, 1] = (q >> np.uint64(32)).astype(np.uint32)
    ctr[:, 2] = np.uint32(step & 0xFFFFFFFF)
    ctr[:, 3] = np.uint32((step >> 32) & 0xFFFFFFFF)
    key = np.zeros((q.size, 2), dtype=np.uint32)
    key[:, 0] = np.uint32((seed & 0xFFFFFFFF) ^ 0x2545F491)
    key[:, 1] = np.uint32((seed >> 32) & 0xFFFFFFFF)
    x = philox4x32_10(ctr, key)
    scale = np.float32(1.0 / 16777216.0)
    if dist == "uniform":
        w = (x >> np.uint32(8)).astype(np.float32) * scale
    else:
        p = x.reshape(-1, 2)
        u1 = ((p[:, 0] >> np.uint32(8)) + np.uint32(1)).astype(np.float32) * scale
        u2 = (p[:, 1] >> np.uint32(8)).astype(np.float32) * scale
        r = np.sqrt(np.float32(-2.0) * np.log(u1)).astype(np.float32)
        th = (np.float32(6.283185307179586) * u2).astype(np.float32)
        w = np.stack((r * np.cos(th), r * np.sin(th)), axis=-1).astype(np.float32)
    return w.reshape(-1)[:total].astype(np.float32)


@pytest.mark.parametrize("dist", ["gaussian", "uniform"])
def test_dr_fill_stream_matches_the_numpy_philox_restatement(dist):
    ops = _ops()
    total = 3 * 4099 + 2
    for seed, step in ((0x1234_5678_9ABC_DEF0, (3 << 32) + 77), ((9 << 32) + 1, (0x7FFF_0001 << 32) + 5)):
        got = ops.dr_fill(seed, step, torch.empty(total, device="cuda"), dist).cpu()
        want = torch.from_numpy(_dr_fill_reference(seed, step, total, dist))
        if dist == "uniform":
            assert torch.equal(got, want)
        else:
            U.assert_close(got, want, rtol=1e-5, atol=3e-5, what="gaussian draws (SFU Box-Muller)")


def _swap_case(T, N, tail, dtype, off_src=0, off_dst=0, env0=0, envs=None):
    from oracle import rl_games_oracle as rg
    ops = _ops()
    g = torch.Generator().manual_seed(T * 7 + N)
    shape = (T, N) + tail
    src = torch.randn(shape, generator=g, dtype=dtype) if dtype.is_floating_point else torch.randint(0, 120, shape, generator=g, dtype=dtype)
    envs = N - env0 if envs is None else envs
    want = rg.swap_and_flatten01(src[:, env0:env0 + envs].contiguous())
    G = U.Guarded()
    s = G.make(shape, dtype, fill=src.cuda(), offset=off_src)
    out = G.make(tuple(want.shape), dtype, offset=off_dst)
    assert _res(s) == off_src and _res(out) == off_dst
    ops.swap_and_flatten01(s, out=out, env0=env0, envs=envs)
    G.check()
    assert torch.equal(out.cpu(), want)
    return s, out


@pytest.mark.parametrize("T,N,tail,dtype,off", [
    (8, 1025, (3,), torch.float32, 0), (32, 1025, (4,), torch.float32, 0), (4, 257, (3,), torch.float32, 4),
    (8, 1025, (3,), torch.uint8, 0), (8, 1025, (5,), torch.uint8, 0), (8, 1025, (16,), torch.uint8, 0),
    (8, 1025, (3,), torch.int16, 0), (8, 1025, (4,), torch.float32, 4), (8, 1025, (8,), torch.uint8, 1),
    (32, 37, (200,), torch.float64, 0)])
def test_swap_and_flatten01_narrow_wide_and_unaligned_rows(T, N, tail, dtype, off):
    """Rows of at most 16 bytes with an even tile width leave the tile through the odd-pitch strided store; src / dst at +4
    run the uint32 kernel and at +1 the uint8 kernel with w > 1; float64 rows of 200 need a 51 KB tile (shared-memory opt-in
    beyond 48 KB).  Whole tensor and an env0 / envs sub-range."""
    # launch_swap_flatten: the uint64 kernel needs both pointers 8-byte aligned, the uint32 kernel 4-byte aligned
    assert off % 8 or not off
    assert off != 1 or off % 4
    _swap_case(T, N, tail, dtype, off, off)
    _swap_case(T, N, tail, dtype, off, off, env0=3, envs=N // 2 + 1)


def test_swap_and_flatten01_refuses_a_tile_beyond_200_kb():
    from bez_isaacgym_b200._lib import BezkError
    ops = _ops()
    src = torch.zeros(32, 2, 1700, device="cuda")
    with pytest.raises(BezkError):
        ops.swap_and_flatten01(src)


@pytest.mark.parametrize("q_off", [4, 8, 12])
def test_quat_rotate_on_unaligned_quaternions_equals_the_aligned_call_and_the_goldens(q_off):
    import os
    ops = _ops()
    gd = {k: torch.from_numpy(v) for k, v in np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden",
                                                                 "fn_jit_utils.npz")).items()}
    q, v = gd["in_q"], gd["in_v"]
    n = q.shape[0]
    for inverse in (False, True):
        want = ops.quat_rotate(q.cuda(), v.cuda(), inverse=inverse).cpu()
        G = U.Guarded()
        qd = G.make(tuple(q.shape), fill=q.cuda(), offset=q_off)
        vd = G.make(tuple(v.shape), fill=v.cuda(), offset=4)
        out = G.make((n, 3), fill=torch.full((n, 3), float("nan")), offset=4)
        assert _res(qd) == q_off                           # launch_quat_rotate: q_vec4 only when q is 16-byte aligned
        ops.quat_rotate(qd, vd, out=out, inverse=inverse)
        G.check()
        assert _same(out.cpu(), want), (q_off, inverse)
        if inverse:
            scale = (v.abs().sum(1, keepdim=True) * (q ** 2).sum(1, keepdim=True) * 2).clamp_min(1.0)
            U.assert_close(out.cpu(), gd["ref_vel_loc"], scale=scale, what="quat_rotate_inverse vs compute_rot vel_loc")
