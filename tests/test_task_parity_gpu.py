"""GPU parity of the task-side CUDA kernels (through the C ABI) against the CPU oracle.

Oracle = ``oracle.task_oracle`` (bit-identical on CPU to the reference's own jit functions, see
tests/test_oracle_pinning.py).  Tolerances and the tie-band policy are documented in tests/_util.py.
"""
import math

import numpy as np
import pytest
import torch

from bez_isaacgym_b200 import bez_model as bm
from bez_isaacgym_b200 import synthetic_gym as sg
from tests import _util as U

pytestmark = pytest.mark.gpu

SIZES = [1, 31, 64, 127, 128, 129, 4096, 20011]


def _ops():
    from bez_isaacgym_b200 import ops
    return ops


# ----------------------------------------------------------------------------------------------- K0
@pytest.mark.parametrize("n", [1, 2, 3, 64, 4097])
def test_pre_physics_matches_oracle_bit_exact(n):
    from oracle import task_oracle as to
    ops = _ops()
    g = torch.Generator().manual_seed(n)
    actions = 3.0 * torch.randn(n, 18, generator=g)            # beyond +-3.9 clip and joint limits
    actions.view(-1)[:: 7] = float("nan")
    actions.view(-1)[3:: 11] = float("inf")
    actions.view(-1)[5:: 13] = -float("inf")
    _, _, default, lower, upper = U.constants(n)
    want_a, want_t = to.pre_physics(actions, default, lower, upper, 3.9)
    cfg = ops.make_task_cfg()
    d = actions.cuda()
    targets, stored = torch.empty_like(d), torch.empty_like(d)
    ops.pre_physics(d, targets, cfg, actions_out=stored)
    assert torch.equal(torch.nan_to_num(targets.cpu(), nan=123.0), torch.nan_to_num(want_t, nan=123.0))
    assert torch.equal(torch.nan_to_num(stored.cpu(), nan=123.0), torch.nan_to_num(want_a, nan=123.0))
    # unaligned input pointer (scalar path) gives the same answer
    pad = torch.empty(n * 18 + 1, device="cuda")
    pad[1:] = d.view(-1)
    t2 = torch.empty_like(d)
    ops.pre_physics(pad[1:].view(n, 18), t2, cfg)
    assert torch.equal(torch.nan_to_num(t2, nan=123.0), torch.nan_to_num(targets, nan=123.0))


# ----------------------------------------------------------------------------------------------- K1
def _run_obs(st, goal, ball_init, prev, cleats=False, clip_obs=math.inf, write_filter=True):
    ops = _ops()
    n = st.num_envs
    cfg = ops.make_task_cfg(num_bodies=st.num_bodies, cleats=cleats, clip_obs=clip_obs, write_contact_filter=write_filter)
    d = st.to("cuda")
    obs = torch.full((n, 54), float("nan"), device="cuda")
    clipped = torch.full((n, 54), float("nan"), device="cuda") if math.isfinite(clip_obs) else None
    prev_d = None if prev is None else prev.cuda().contiguous()
    ops.compute_observations(d.dof_state, d.rigid_body, d.root_states, d.net_contact, goal.cuda(), ball_init.cuda(),
                             cfg, obs, prev_lin_vel=prev_d, obs_clipped=clipped)
    torch.cuda.synchronize()
    return obs.cpu(), d, prev_d, clipped


@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("alias", [False, True])
def test_observations_match_oracle(n, alias):
    st = sg.make_state(n, seed=100 + n)
    goal, ball_init, *_ = U.constants(n)
    prev = None if alias else 0.3 * torch.randn(n, 3, generator=torch.Generator().manual_seed(5))
    want, want_cf, want_prev = U.oracle_observations(st, prev, goal, ball_init)
    got, d, prev_d, _ = _run_obs(st, goal, ball_init, prev)
    # raw copies and bit logic are bit-exact
    assert torch.equal(got[:, 0:36], want[:, 0:36]), "dof_pos / dof_vel copy"
    assert torch.equal(got[:, 39:42], want[:, 39:42]), "clamped angular velocity"
    assert torch.equal(got[:, 44:52], want[:, 44:52]), "foot pressure bits"
    assert torch.equal(got[:, 52:54], want[:, 52:54]), "ball_init"
    # in-place contact noise filter written back bit-exactly (kick_env.py:987-990)
    assert torch.equal(d.net_contact.cpu(), want_cf)
    # IMU linear term: condition-aware tolerance on the mat-vec; heading: plain tolerance
    U.assert_close(got[:, 36:39], want[:, 36:39], scale=U.imu_term_scale(st, prev), what="imu lin_acc")
    U.assert_close(got[:, 42:44], want[:, 42:44], what="off_orn")
    if not alias:
        assert torch.equal(prev_d.cpu(), want_prev), "prev_lin_vel <- current IMU-link velocity"
    # the other state tensors are untouched
    assert torch.equal(d.dof_state.cpu(), st.dof_state) and torch.equal(d.root_states.cpu(), st.root_states)
    assert torch.equal(d.rigid_body.cpu(), st.rigid_body)


def test_observations_literal_tolerance_fraction():
    """How many IMU entries meet the LITERAL rtol 1e-5 / atol 1e-6 (no condition-aware scale): reported,
    and required to be the overwhelming majority."""
    n = 20000
    st = sg.make_state(n, seed=7)
    goal, ball_init, *_ = U.constants(n)
    prev = 0.3 * torch.randn(n, 3, generator=torch.Generator().manual_seed(5))
    want, _, _ = U.oracle_observations(st, prev, goal, ball_init)
    got, *_ = _run_obs(st, goal, ball_init, prev)
    ok = (got - want).abs() <= U.ATOL + U.RTOL * want.abs()
    frac = ok.float().mean().item()
    print(f"literal-tolerance pass fraction over all obs entries: {frac:.6f}")
    assert frac > 0.999


def test_observations_aliasing_gives_unit_gravity_column():
    """In the reference's steady state prev_lin_vel aliases the velocity view, so lin_acc == R(q)(0,0,1)."""
    n = 1000
    st = sg.make_state(n, seed=3)
    goal, ball_init, *_ = U.constants(n)
    got, *_ = _run_obs(st, goal, ball_init, None)
    from oracle import task_oracle as to
    col = to.wxyz_matrix(U.views(st)["quat"])[:, :, 2]
    U.assert_close(got[:, 36:39], col, what="third column of R")


def test_observations_cleats_variant():
    n = 4099
    st = sg.make_state(n, seed=11, cleats=True)
    goal, ball_init, *_ = U.constants(n)
    want, want_cf, _ = U.oracle_observations(st, None, goal, ball_init, cleats=True)
    got, d, _, _ = _run_obs(st, goal, ball_init, None, cleats=True)
    v = U.views(st, cleats=True)
    norms = torch.cat((torch.linalg.norm(v["left_c"], dim=-1), torch.linalg.norm(v["right_c"], dim=-1)), 1)
    tie = (norms - 1.0).abs() <= 2 * U.ulp(1.0)
    mism = got[:, 44:52] != want[:, 44:52]
    assert not bool((mism & ~tie).any()), "cleat bits differ outside the |f| = 1 N tie band"
    print(f"cleat bits inside tie band: {int(tie.sum())}, mismatching: {int(mism.sum())}")
    assert torch.equal(d.net_contact.cpu(), st.net_contact), "cleats path must not filter the contact buffer"
    U.assert_close(got[:, 42:44], want[:, 42:44], what="off_orn")


def test_observations_edge_cases():
    """Contact-filter thresholds, NaN forces, fz around 1 N, zero distance to goal, non-unit quaternions."""
    n = 64
    st = sg.make_state(n, seed=21)
    goal, ball_init, *_ = U.constants(n)
    cf = st.net_contact.view(n, -1, 3)
    f32 = lambda x: float(torch.tensor(x, dtype=torch.float32))
    vals = [0.0, -0.0, f32(0.01), -f32(0.01), float(np.nextafter(np.float32(0.01), np.float32(1.0))), 0.005, -0.005, 2.0, -2.0, float("nan"),
            float("inf"), -float("inf")]
    fz = [0.5, f32(0.999), 1.0, float(np.nextafter(np.float32(1.0), np.float32(2.0))), 2.0, 0.005, float("nan"), f32(0.99), f32(1.01)]
    k = 0
    for e in range(n):
        for body in (bm.LEFT_FOOT_BODY, bm.RIGHT_FOOT_BODY):
            cf[e, body, 0] = vals[k % len(vals)]
            cf[e, body, 1] = vals[(k // len(vals) + k) % len(vals)]
            cf[e, body, 2] = fz[k % len(fz)]
            k += 1
    root = st.root_states.view(n, 2, 13)
    root[0, 0, 0:2] = goal[0]                                   # ||d|| = 0 -> NaN heading terms
    rb = st.rigid_body.view(n, -1, 13)
    rb[1, bm.IMU_BODY, 3:7] = torch.tensor([0.0, 0.0, 0.0, 1.0])     # identity
    rb[2, bm.IMU_BODY, 3:7] = torch.tensor([0.0, 0.0, 1.0, 0.0])     # 180 deg about z
    rb[3, bm.IMU_BODY, 3:7] = torch.tensor([0.3, -0.2, 0.1, 2.5])    # non-unit
    rb[4, bm.IMU_BODY, 10:13] = torch.tensor([100.0, -100.0, float("nan")])
    rb[5, bm.IMU_BODY, 7:10] = torch.tensor([1e3, -1e3, 0.0])        # lin-acc clamp
    prev = torch.zeros(n, 3)
    want, want_cf, _ = U.oracle_observations(st, prev, goal, ball_init)
    got, d, _, _ = _run_obs(st, goal, ball_init, prev)
    assert torch.equal(got[:, 44:52], want[:, 44:52])
    assert torch.equal(torch.nan_to_num(d.net_contact.cpu(), nan=7.0), torch.nan_to_num(want_cf, nan=7.0))
    assert torch.isnan(got[0, 42:44]).all() and torch.isnan(want[0, 42:44]).all()
    U.assert_close(got[:, 36:42], want[:, 36:42], scale=U.imu_term_scale(st, prev), what="imu")
    U.assert_close(got[1:, 42:44], want[1:, 42:44], what="off_orn")


def test_observations_clip_obs_and_filter_flag():
    n = 300
    st = sg.make_state(n, seed=31)
    goal, ball_init, *_ = U.constants(n)
    want, _, _ = U.oracle_observations(st, None, goal, ball_init)
    got, d, _, clipped = _run_obs(st, goal, ball_init, None, clip_obs=1.0, write_filter=False)
    assert torch.equal(clipped.cpu(), torch.clamp(got, -1.0, 1.0))
    assert torch.equal(d.net_contact.cpu(), st.net_contact), "filter write-back disabled"
    assert torch.equal(got[:, 44:52], want[:, 44:52])


# ----------------------------------------------------------------------------------------------- K2
def _run_reward(st, goal, ball_init, reset_in, progress):
    ops = _ops()
    n = st.num_envs
    cfg = ops.make_task_cfg(num_bodies=st.num_bodies)
    d = st.to("cuda")
    rew = torch.full((n,), float("nan"), device="cuda")
    reset_out = torch.full((n,), -7, dtype=torch.long, device="cuda")
    ops.compute_reward(d.dof_state, d.rigid_body, d.root_states, goal.cuda(), ball_init.cuda(), reset_in.cuda(),
                       progress.cuda(), cfg, rew, reset_out)
    torch.cuda.synchronize()
    return rew.cpu(), reset_out.cpu()


def _oracle_reward(st, goal, ball_init, default, reset_in, progress):
    from oracle import task_oracle as to
    v = U.views(st)
    return to.reward(v["dof_pos"], default, v["lin"], v["ang"], v["bez_pos"], v["ball_pos"], v["ball_vel"], goal,
                     ball_init, torch.tensor([0.0, 0.0]), reset_in, progress, 900)


def _check_reward(st, goal, ball_init, default, reset_in, progress):
    want_r, want_m = _oracle_reward(st, goal, ball_init, default, reset_in, progress)
    got_r, got_m = _run_reward(st, goal, ball_init, reset_in, progress)
    band = U.reward_tie_band(st, goal, ball_init)
    mism = got_m != want_m
    assert not bool((mism & ~band).any()), f"reset mask differs outside the tie band at {(mism & ~band).nonzero()[:5]}"
    keep = ~band
    U.assert_close(got_r[keep], want_r[keep], scale=U.reward_scale(st, goal, ball_init, default)[keep], what="reward")
    return int(band.sum()), int(mism.sum())


@pytest.mark.parametrize("n", SIZES + [200003])
def test_reward_and_reset_mask_match_oracle(n):
    st = sg.make_state(n, seed=300 + n)
    goal, ball_init, default, _, _ = U.constants(n)
    progress, reset_in = sg.make_bookkeeping(n, seed=n)
    progress[: min(n, 6)] = torch.tensor([898, 899, 900, 901, 0, 450])[: min(n, 6)]
    in_band, mismatched = _check_reward(st, goal, ball_init, default, reset_in, progress)
    print(f"n={n}: envs in tie band {in_band}, mask mismatches (all inside band) {mismatched}")


def test_reward_each_rule_alone_and_override_order():
    """One env per rule, then all rules at once (later rules override the reward, SURVEY A.1)."""
    n = 8
    st = sg.make_state(n, seed=1)
    goal, ball_init, default, _, _ = U.constants(n)
    root = st.root_states.view(n, 2, 13)
    root[:, 0, 0:3] = torch.tensor([0.0, 0.0, 0.34])
    root[:, 1, 0:3] = torch.tensor([0.4, 0.1, 0.1])
    progress = torch.full((n,), 10, dtype=torch.long)
    root[1, 0, 2] = 0.27                                        # rule 1
    root[2, 0, 0:2] = torch.tensor([0.4, 0.4])                  # rule 2
    root[3, 1, 0:2] = torch.tensor([1.6, 1.0])                  # rule 3 (ball behind the goal line, wide angle)
    root[4, 1, 0:2] = torch.tensor([1.49, 0.01])                # rule 4
    progress[5] = 900                                           # rule 5
    root[6, 0, 2] = 0.2; root[6, 0, 0:2] = torch.tensor([0.6, 0.0])
    root[6, 1, 0:2] = torch.tensor([1.5, 0.02]); progress[6] = 450   # rules 1, 2, 4 -> rule 4's reward
    root[7, 1, 0:2] = torch.tensor([1.5, 0.02]); progress[7] = 900   # rules 4, 5 -> 0
    reset_in = torch.zeros(n, dtype=torch.long)
    want_r, want_m = _oracle_reward(st, goal, ball_init, default, reset_in, progress)
    got_r, got_m = _run_reward(st, goal, ball_init, reset_in, progress)
    assert want_m.tolist() == [0, 1, 1, 1, 1, 1, 1, 1]
    assert torch.equal(got_m, want_m)
    U.assert_close(got_r, want_r, scale=U.reward_scale(st, goal, ball_init, default), what="reward")
    assert got_r[1] == -1.0 and got_r[2] == -1.0 and got_r[3] == -1.0 and got_r[5] == 0.0 and got_r[7] == 0.0
    assert got_r[6] == want_r[6] == 50.0
    # reset_in = 1 survives when no rule fires
    got_r2, got_m2 = _run_reward(st, goal, ball_init, torch.ones(n, dtype=torch.long), progress)
    assert got_m2.tolist() == [1] * n


def test_reward_nan_inputs_fall_through():
    n = 4
    st = sg.make_state(n, seed=2)
    goal, ball_init, default, _, _ = U.constants(n)
    root = st.root_states.view(n, 2, 13)
    root[:, 0, 0:3] = torch.tensor([0.0, 0.0, 0.34])
    root[0, 0, 2] = float("nan")
    root[1, 1, 0:2] = goal[1]                                   # n_goal = 0 -> division by zero, rule 4 fires
    root[2, 1, 0] = float("nan")
    progress = torch.full((n,), 5, dtype=torch.long)
    reset_in = torch.zeros(n, dtype=torch.long)
    want_r, want_m = _oracle_reward(st, goal, ball_init, default, reset_in, progress)
    got_r, got_m = _run_reward(st, goal, ball_init, reset_in, progress)
    assert torch.equal(got_m, want_m)
    assert torch.equal(torch.isnan(got_r), torch.isnan(want_r))
    ok = ~torch.isnan(want_r)
    U.assert_close(got_r[ok], want_r[ok], scale=U.reward_scale(st, goal, ball_init, default)[ok], what="reward")


# ----------------------------------------------------------------------------------------------- K3 / Philox
def test_philox_matches_numpy_reference():
    from oracle.philox_ref import reset_uniforms
    ops = _ops()
    for n, seed, step in [(1, 0, 0), (1000, 42, 7), (257, 2 ** 40 + 3, 2 ** 33 + 5)]:
        out = torch.empty(n, 36, device="cuda")
        ops.philox_uniforms(seed, step, out)
        want = torch.from_numpy(reset_uniforms(seed, step, n))
        assert torch.equal(out.cpu(), want)
        assert float(out.min()) >= 0.0 and float(out.max()) < 1.0


@pytest.mark.parametrize("use_philox", [False, True])
def test_reset_idx_matches_oracle(use_philox):
    from oracle import task_oracle as to
    from oracle.philox_ref import reset_uniforms
    ops = _ops()
    n = 500
    st = sg.make_state(n, seed=77)
    _, _, default, lower, upper = U.constants(n)
    env_ids = torch.tensor(sorted(set(torch.randint(0, n, (60,), generator=torch.Generator().manual_seed(1)).tolist())))
    k = env_ids.numel()
    if use_philox:
        u = torch.from_numpy(reset_uniforms(9, 4, n))[env_ids]
    else:
        u = torch.rand(k, 36, generator=torch.Generator().manual_seed(2))
    pos, vel = to.reset_idx_dof(default[env_ids], lower, upper, u[:, 0:18], u[:, 18:36])
    want_dof = st.dof_state.clone().view(n, 18, 2)
    want_dof[env_ids, :, 0] = pos
    want_dof[env_ids, :, 1] = vel
    init_root = torch.zeros(n, 2, 13)
    init_root[:, 0, 0:3] = torch.tensor([0.0, 0.0, 0.34]); init_root[:, 0, 6] = 1.0
    init_root[:, 1, 0:3] = torch.tensor([0.175, 0.0, 0.1]); init_root[:, 1, 6] = 1.0
    want_root = st.root_states.clone().view(n, 2, 13)
    want_root[env_ids] = init_root[env_ids]
    d = st.to("cuda")
    progress = torch.arange(n, device="cuda")
    reset = torch.ones(n, dtype=torch.long, device="cuda")
    cfg = ops.make_task_cfg()
    ops.reset_idx(env_ids.cuda(), d.dof_state, d.root_states, init_root.view(n * 2, 13).cuda(), progress, reset, cfg,
                  uniforms=None if use_philox else u.cuda().contiguous(), seed=9, step=4)
    assert torch.equal(d.dof_state.cpu().view(n, 18, 2), want_dof)
    assert torch.equal(d.root_states.cpu().view(n, 2, 13), want_root)
    keep = torch.ones(n, dtype=torch.bool); keep[env_ids] = False
    assert torch.equal(progress.cpu()[env_ids], torch.zeros(k, dtype=torch.long))
    assert torch.equal(progress.cpu()[keep], torch.arange(n)[keep])
    assert torch.equal(reset.cpu(), keep.long())


# ----------------------------------------------------------------------------------------------- fused step
@pytest.mark.parametrize("n,parts_mode", [(64, "fused"), (4096, "fused"), (4099, "fused"), (4099, "split"), (33000, "fused")])
@pytest.mark.parametrize("alias", [True, False])
def test_fused_post_physics_follows_step_oracle(n, parts_mode, alias):
    """Several VecTask.step post-physics phases in a row (state perturbed in between the way a simulator
    would) against oracle.task_oracle.KickStepOracle: timeout / progress / masked reset / obs / reward."""
    from oracle import task_oracle as to
    from oracle.philox_ref import reset_uniforms
    ops = _ops()
    seed = 1234
    st = sg.make_state(n, seed=500 + n)
    goal, ball_init, default, lower, upper = U.constants(n)
    init_root = torch.zeros(n, 2, 13)
    init_root[:, 0, 0:3] = torch.tensor([0.0, 0.0, 0.34]); init_root[:, 0, 6] = 1.0
    init_root[:, 1, 0:3] = torch.tensor([0.175, 0.0, 0.1]); init_root[:, 1, 6] = 1.0
    init_root = init_root.view(n * 2, 13)
    cpu = st.clone()
    orc = to.KickStepOracle(n, cpu.root_states, cpu.dof_state, cpu.rigid_body, cpu.net_contact, default, lower, upper,
                            goal, ball_init, torch.tensor([0.0, 0.0]), init_root, alias_prev_lin_vel=alias,
                            reset_uniforms=lambda step: torch.from_numpy(reset_uniforms(seed, step, n)))
    progress0, reset0 = sg.make_bookkeeping(n, seed=n + 1)
    progress0[: min(n, 4)] = torch.tensor([897, 898, 899, 900])[: min(n, 4)]
    orc.progress_buf[:] = progress0
    orc.reset_buf[:] = reset0
    if not alias:
        orc.prev_lin_vel = torch.zeros(n, 3)

    d = st.to("cuda")
    cfg = ops.make_task_cfg(num_bodies=st.num_bodies)
    obs = torch.zeros(n, 54, device="cuda"); rew = torch.zeros(n, device="cuda")
    reset = reset0.cuda(); progress = progress0.cuda(); timeout = torch.zeros(n, dtype=torch.long, device="cuda")
    randomize = torch.zeros(n, dtype=torch.long, device="cuda")
    # the reference starts from zeros (kick_env.py:183) and aliases the velocity view from the second
    # observation on (:930): step 0 always reads a zero buffer, later steps pass NULL in aliasing mode
    prev_d = torch.zeros(n, 3, device="cuda")
    g_d, b_d, ir_d = goal.cuda(), ball_init.cuda(), init_root.cuda()

    total_band = 0
    for step in range(4):
        if step > 0:                                            # "simulate": move the state, identically on both sides
            fresh = sg.make_state(n, seed=900 + step)
            for name in ("root_states", "rigid_body", "net_contact"):
                getattr(cpu, name).copy_(getattr(fresh, name)); getattr(d, name).copy_(getattr(fresh, name).cuda())
            drift = 0.01 * torch.randn(n * 18, 2, generator=torch.Generator().manual_seed(step))
            cpu.dof_state.add_(drift); d.dof_state.add_(drift.cuda())
        before = sg.SimState(cpu.root_states.clone(), cpu.dof_state.clone(), cpu.rigid_body.clone(),
                             cpu.net_contact.clone(), n, st.num_bodies)
        prev_before = None if (alias and step > 0) else orc.prev_lin_vel.clone().float()
        want_obs, want_rew, want_reset, want_timeout = orc.post_physics_step()
        kw = dict(prev_lin_vel=None if (alias and step > 0) else prev_d, seed=seed, step=step, randomize_buf=randomize)
        if parts_mode == "fused":
            ops.post_physics(d.dof_state, d.rigid_body, d.root_states, d.net_contact, g_d, b_d, ir_d, reset, progress,
                             timeout, cfg, obs, rew, **kw)
        else:                                                   # the north-star's two kernels
            ops.post_physics(d.dof_state, d.rigid_body, d.root_states, d.net_contact, g_d, b_d, ir_d, reset, progress,
                             timeout, cfg, obs, None, parts=3, **kw)
            ops.post_physics(d.dof_state, d.rigid_body, d.root_states, None, g_d, b_d, ir_d, reset, progress,
                             None, cfg, None, rew, parts=4, seed=seed, step=step)
        torch.cuda.synchronize()
        # bookkeeping: bit-exact
        assert torch.equal(timeout.cpu(), want_timeout), f"timeout step {step}"
        assert torch.equal(progress.cpu(), orc.progress_buf), f"progress step {step}"
        assert torch.equal(randomize.cpu(), orc.randomize_buf)
        # reset write-back into the simulator tensors: bit-exact
        assert torch.equal(d.dof_state.cpu(), cpu.dof_state), f"dof_state after masked reset, step {step}"
        assert torch.equal(d.root_states.cpu(), cpu.root_states)
        assert torch.equal(d.net_contact.cpu(), cpu.net_contact)
        after = sg.SimState(cpu.root_states, cpu.dof_state, cpu.rigid_body, cpu.net_contact, n, st.num_bodies)
        band = U.reward_tie_band(after, goal, ball_init)
        total_band += int(band.sum())
        mism = reset.cpu() != want_reset
        assert not bool((mism & ~band).any()), f"reset mask outside tie band, step {step}"
        got = obs.cpu()
        assert torch.equal(got[:, 0:36], want_obs[:, 0:36]) and torch.equal(got[:, 44:54], want_obs[:, 44:54])
        U.assert_close(got[:, 36:42], want_obs[:, 36:42], scale=U.imu_term_scale(after, prev_before), what="imu")
        U.assert_close(got[:, 42:44], want_obs[:, 42:44], what="off_orn")
        keep = ~band
        U.assert_close(rew.cpu()[keep], want_rew[keep], scale=U.reward_scale(after, goal, ball_init, default)[keep],
                       what=f"reward step {step}")
        # keep both sides on the oracle's mask so that a tie-band env cannot fork the trajectories
        reset.copy_(want_reset.cuda())
    print(f"n={n} {parts_mode} alias={alias}: envs inside tie band over 4 steps: {total_band}")


def test_cpu_tensors_raise_no_fallback():
    ops = _ops()
    cfg = ops.make_task_cfg()
    a = torch.zeros(4, 18)
    with pytest.raises(Exception, match="CUDA only"):
        ops.pre_physics(a, torch.zeros(4, 18), cfg)


@pytest.mark.parametrize("task", ["kick", "walk", "orient"])
@pytest.mark.parametrize("host_mode", ["zero_copy", "staged", "staged_ce", "staged_pack", "staged_pack+dof", "staged_pack+cleats", "auto"])
def test_host_pipeline_equals_gpu_pipeline(host_mode, task):
    """``use_gpu_pipeline: False`` (simulator tensors in pinned host memory; BASELINE configs[0] sim_device=cpu pipeline=cpu;
    the reference's device selection ``tasks/base/vec_task.py:51-98`` serves every task): same kernels, so results are
    bit-identical to the GPU pipeline, and resets land in the HOST dof_state.  ``staged_ce`` = chunked copy-engine pipeline
    (strided cudaMemcpy2DAsync pulls of the sparse rows); it cannot write the contact filter back, so the filter is off there.
    ``staged_pack`` = the same pipeline with the sparse rows gathered by host worker threads (``bezk_host_pack_*``)."""
    from bez_isaacgym_b200.synthetic_sim import SyntheticGym
    from bez_isaacgym_b200 import tasks as T
    cls = {"kick": T.KickEnv, "walk": T.WalkEnv, "orient": T.OrientEnv}[task]
    n = 4099
    host_mode, _, variant = host_mode.partition("+")
    cleats = variant == "cleats"
    if cleats and task != "kick":
        pytest.skip("cleats variant: BezKick only")
    st = sg.make_state(n, seed=77, task=task, cleats=cleats)
    envs = {}
    for kind in ("gpu", "host"):
        cfg = bm.default_task_cfg(n, cleats=cleats, use_gpu_pipeline=(kind == "gpu"), rl_device="cuda:0" if kind == "gpu" else "cpu",
                                  task=task)
        cfg["seed"] = 5
        cfg["env"]["hostPipeline"] = host_mode
        cfg["env"]["hostPipelineChunks"] = [1, 2, 1] if variant == "dof" else 3
        cfg["env"]["hostPackDof"] = variant == "dof"
        cfg["env"]["writeContactFilter"] = host_mode not in ("staged_ce", "staged_pack", "auto")
        sim = SyntheticGym(n, device="cuda:0", cleats=cleats, state=st.clone(), host=(kind == "host"), task=task)
        envs[kind] = cls(cfg, "cuda:0", 0, True, sim=sim)
        envs[kind].progress_buf.copy_(torch.arange(n, device="cuda") % envs[kind].max_episode_length)
    # rl_games' per-step reward path in the step's epilogue (a16): also served by the copy-engine / packed host pipelines, with
    # the critic values arriving from pinned HOST memory (the outputs are device rollout slots on both sides)
    epilogue = True
    sh = {k: torch.zeros(n, device="cuda") for k in envs}
    dn = {k: torch.zeros(n, dtype=torch.uint8, device="cuda") for k in envs}
    for step in range(4):
        a = sg.make_actions(n, seed=step)
        if epilogue:
            vals = torch.randn(n, generator=torch.Generator().manual_seed(step))
            envs["gpu"].set_rollout_targets(values=vals.cuda(), shaped_rewards=sh["gpu"], dones_u8=dn["gpu"])
            envs["host"].set_rollout_targets(values=vals.pin_memory() if step != 2 else vals.cuda(), shaped_rewards=sh["host"],
                                             dones_u8=dn["host"])
        o_g, r_g, d_g, e_g = envs["gpu"].step(a.cuda())
        o_h, r_h, d_h, e_h = envs["host"].step(a.pin_memory() if step % 2 else a)
        assert o_h["obs"].device.type == "cpu" and r_h.device.type == "cpu"
        torch.cuda.synchronize()
        og, oh = o_g["obs"].cpu(), o_h["obs"]
        assert bool(((og == oh) | (og.isnan() & oh.isnan())).all()) and torch.equal(r_g.cpu(), r_h)
        assert torch.equal(d_g.cpu(), d_h) and torch.equal(e_g["time_outs"].cpu(), e_h["time_outs"])
        if epilogue:
            assert torch.equal(sh["gpu"], sh["host"]) and torch.equal(dn["gpu"], dn["host"]) and torch.equal(dn["host"].cpu().long(), d_h)
            assert float(sh["host"].abs().sum()) > 0
        assert torch.equal(envs["gpu"].dof_state.cpu(), envs["host"].dof_state), "resets written into the host dof_state"
        assert torch.equal(envs["gpu"].net_contact.cpu(), envs["host"].net_contact), "contact filter written back (or left alone)"
        assert torch.equal(envs["gpu"].root_states.cpu(), envs["host"].root_states)
        assert torch.equal(envs["gpu"].targets.cpu(), envs["host"].targets.cpu())
        if task != "kick":
            assert torch.equal(envs["gpu"].goal.cpu(), envs["host"].goal.cpu()), "goal redraw on reset"
    assert int(d_g.sum()) > 0
    link = envs["host"].link_counters()
    assert link["h2d_bytes"] > 0 and link["d2h_bytes"] > 0
    if host_mode == "staged_pack" and task == "kick" and not cleats and variant == "":
        # the byte counts bench.py reports are those of the copies issued: per env-step dof_state 144 + record 96 + actions 72 in,
        # obs 216 + rew 4 + reset 8 + time_outs 8 + PD targets 72 out
        assert link["h2d_bytes"] == 4 * n * (144 + 96 + 72) and link["d2h_bytes"] == 4 * n * (216 + 4 + 8 + 8 + 72)
    if host_mode == "auto":
        assert envs["host"].host_pipeline == "zero_copy"          # a small task: two zero-copy launches beat any staged pipeline


def test_chunked_step_equals_one_launch():
    """``bezk_post_physics_chunk``: a step launched as chunks [env_base, env_base + n) with offset pointers gives, bit for bit,
    the results of one launch -- the Philox reset noise stays keyed by the GLOBAL env id."""
    import ctypes as C
    from bez_isaacgym_b200 import _lib
    ops = _ops()
    n = 4099
    cfg = ops.make_task_cfg()
    goal, ball_init, default, _, _ = U.constants(n, "cuda")
    init_root = sg.make_initial_root_states(n, "cuda")
    outs = []
    for chunks in (None, [(0, 1280), (1280, 2560), (2560, 4099)]):
        st = sg.make_state(n, seed=31).to("cuda")
        progress, reset = sg.make_bookkeeping(n, seed=4, device="cuda", p_reset=0.2)
        timeout = torch.empty(n, dtype=torch.long, device="cuda")
        obs = torch.empty(n, 54, device="cuda"); rew = torch.empty(n, device="cuda")
        prev = torch.zeros(n, 3, device="cuda")
        if chunks is None:
            ops.post_physics(st.dof_state, st.rigid_body, st.root_states, st.net_contact, goal, ball_init, init_root, reset, progress,
                             timeout, cfg, obs, rew, prev_lin_vel=prev, seed=9, step=3)
        else:
            lib = _lib.load()
            stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
            p4 = lambda t, k: C.c_void_p(t.data_ptr() + 4 * k)        # noqa: E731
            p8 = lambda t, k: C.c_void_p(t.data_ptr() + 8 * k)        # noqa: E731
            for lo, hi in chunks:
                rc = lib.bezk_post_physics_chunk(p4(st.dof_state, lo * 36), p4(st.rigid_body, lo * 22 * 13), p4(st.root_states, lo * 26),
                                                 p4(st.net_contact, lo * 66), p4(prev, lo * 3), p4(goal, lo * 2), p4(ball_init, lo * 2),
                                                 p4(init_root, lo * 26), None, 9, 3, p8(reset, lo), p8(progress, lo), p8(timeout, lo),
                                                 None, C.byref(cfg), p4(obs, lo * 54), None, p4(rew, lo), 7, hi - lo, lo, None, None,
                                                 stream)
                _lib.check(rc, "bezk_post_physics_chunk")
        torch.cuda.synchronize()
        outs.append([t.clone() for t in (obs, rew, reset, progress, timeout, st.dof_state, st.root_states, st.net_contact, prev)])
    for a, b in zip(*outs):
        assert torch.equal(a, b) or bool(((a == b) | (a.isnan() & b.isnan())).all())
    assert int(outs[0][2].sum()) > 0


def test_branch_free_division_and_sqrt_are_ieee_exact():
    """The task kernels' division / square root (Mth<true>: NVIDIA's fast sequences with a sticky validity flag instead of a
    branch per operation) against the built-in IEEE operators: all 2^32 radicands, 2^31 random quotients (a quarter of them in
    the exponent window the task math lives in) and a 24 x 24 cross of special values -- zero mismatches wherever the fast path
    accepts its operands."""
    import ctypes as C
    from bez_isaacgym_b200 import _lib
    lib = _lib.load()
    counts = torch.zeros(4, dtype=torch.int64, device="cuda")
    _lib.check(lib.bezk_selftest_fastmath(1 << 31, 12345, C.c_void_p(counts.data_ptr()), C.c_void_p(torch.cuda.current_stream().cuda_stream)))
    torch.cuda.synchronize()
    sq_bad, div_bad, sq_ok, div_ok = counts.tolist()
    assert sq_bad == 0 and div_bad == 0, (sq_bad, div_bad)
    # positive floats in [2^-60, 2^60] + the two zeros; a good share of the random quotients
    assert sq_ok == 120 * (1 << 23) + 1 + 2 and div_ok > (1 << 27)


def test_default_host_pipeline_resolves_to_a_mode_that_serves_the_configuration():
    """``env.hostPipeline`` defaults to ``auto``: ``zero_copy`` for small tasks (two launches, nothing staged) and when the caller
    asks for what only that mode does (the two-kernel split, the in-place contact filter); a staged pipeline for the fused step of
    a large task -- packed when the process has host cores to gather with -- in chunks of >= 32 768 envs."""
    from bez_isaacgym_b200.synthetic_sim import SyntheticGym
    from bez_isaacgym_b200 import tasks as T

    def make(n, st, fusion="fused", **env):
        cfg = bm.default_task_cfg(n, use_gpu_pipeline=False, rl_device="cpu")
        cfg["env"].update(env)
        return T.KickEnv(cfg, "cuda:0", 0, True, sim=SyntheticGym(n, device="cuda:0", state=st.clone(), host=True), fusion=fusion)

    n = 100352                                                    # >= 98 304: staged whatever the host's core count
    st = sg.make_state(n, seed=5, filler=False)
    a = sg.make_actions(n, seed=1)
    e_auto, e_split, e_filter = make(n, st), make(n, st, "split"), make(n, st, writeContactFilter=True)
    assert e_auto.host_pipeline in ("staged_pack", "staged_ce") and len(e_auto._ce_chunks) == 3
    assert e_split.host_pipeline == "zero_copy" and e_filter.host_pipeline == "zero_copy"
    outs = [e.step(a) for e in (e_auto, e_split, e_filter)]
    torch.cuda.synchronize()
    for o, r, d, _ in outs[1:]:
        same = (o["obs"] == outs[0][0]["obs"]) | (o["obs"].isnan() & outs[0][0]["obs"].isnan())
        assert bool(same.all()) and torch.equal(r, outs[0][1]) and torch.equal(d, outs[0][2])
    assert not torch.equal(e_filter.net_contact, e_auto.net_contact), "only the zero-copy mode filters the simulator's tensor in place"
    small = make(1000, sg.make_state(1000, seed=5))
    assert small.host_pipeline == "zero_copy"


def test_packed_host_pipeline_at_the_baseline_size_is_bit_identical_to_the_gpu_pipeline():
    """The configuration ``bench.py``'s e2e leg runs (262 144 envs, ``staged_pack``, 4 chunks, critic values arriving from pinned
    host memory, reward epilogue in the step): every output of two steps equals the GPU pipeline's bit for bit."""
    from bez_isaacgym_b200.synthetic_sim import SyntheticGym
    from bez_isaacgym_b200 import tasks as T
    n = 262144
    st = sg.make_state(n, seed=11, filler=False)

    class OwnedRootSim(SyntheticGym):
        owns_root_reset = True

    envs = {}
    for kind in ("gpu", "host"):
        cfg = bm.default_task_cfg(n, use_gpu_pipeline=(kind == "gpu"), rl_device="cuda:0" if kind == "gpu" else "cpu")
        cfg["env"]["hostPipeline"] = "staged_pack"
        cfg["env"]["imuPrevVelAliasing"] = False
        envs[kind] = T.KickEnv(cfg, "cuda:0", 0, True, sim=OwnedRootSim(n, device="cuda:0", state=st.clone(), host=(kind == "host")))
        envs[kind].progress_buf.copy_(torch.arange(n, device="cuda") % envs[kind].max_episode_length)
    assert envs["host"].host_pipeline == "staged_pack" and len(envs["host"]._ce_chunks) == 4
    sh = {k: torch.zeros(n, device="cuda") for k in envs}
    dn = {k: torch.zeros(n, dtype=torch.uint8, device="cuda") for k in envs}
    for step in range(2):
        a = sg.make_actions(n, seed=step)
        vals = torch.randn(n, generator=torch.Generator().manual_seed(step))
        envs["gpu"].set_rollout_targets(values=vals.cuda(), shaped_rewards=sh["gpu"], dones_u8=dn["gpu"])
        envs["host"].set_rollout_targets(values=vals.pin_memory(), shaped_rewards=sh["host"], dones_u8=dn["host"])
        o_g, r_g, d_g, e_g = envs["gpu"].step(a.cuda())
        o_h, r_h, d_h, e_h = envs["host"].step(a.pin_memory())
        torch.cuda.synchronize()
        og, oh = o_g["obs"].cpu(), o_h["obs"]
        assert bool(((og == oh) | (og.isnan() & oh.isnan())).all()) and torch.equal(r_g.cpu(), r_h) and torch.equal(d_g.cpu(), d_h)
        assert torch.equal(e_g["time_outs"].cpu(), e_h["time_outs"]) and torch.equal(sh["gpu"], sh["host"]) and torch.equal(dn["gpu"], dn["host"])
        assert torch.equal(envs["gpu"].dof_state.cpu(), envs["host"].dof_state) and torch.equal(envs["gpu"].targets.cpu(), envs["host"].targets)
    assert int(d_g.sum()) > 100
    from tests.test_parity_report_gpu import record
    record("host_pipeline_staged_pack_262144_envs", {
        "compared_with": "KickEnv.step of the GPU pipeline on the same state, 2 steps", "chunks": 4,
        "bit_identical": ["obs", "rew", "reset", "time_outs", "shaped_rewards", "dones_u8", "dof_state (reset rows)", "PD targets"],
        "resets_in_last_step": int(d_g.sum())})
