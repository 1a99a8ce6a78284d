"""Parity at the BASELINE sizes, with the numbers RECORDED (VERDICT r1, item 3): the fused step through the C ABI against the CPU
oracle at 4 096 (configs[1]), 262 144 (configs[3]) and 1 048 576 (configs[4]) envs, ``KickEnv.step`` at 4 096 envs, and the
learner kernels at their BASELINE shapes.  Every test also asserts; what it measures goes to the JSON file named by
``BEZK_PARITY_REPORT`` when that is set (``profiles/parity_r02.json`` is such a report; a run without it writes nothing, so the
suite leaves the tree as it found it): per output the literal rtol 1e-5 / atol 1e-6 pass
fraction, the condition-aware pass fraction where one is used, the maximum error in ulp, and for the masks the population of
every tie band and how many of those envs actually flipped."""
import json
import math
import os

import numpy as np
import pytest
import torch

from bez_isaacgym_b200 import bez_model as bm
from bez_isaacgym_b200 import synthetic_gym as sg
from tests import _util as U

pytestmark = pytest.mark.gpu

REPORT = os.environ.get("BEZK_PARITY_REPORT")


def record(section, payload):
    if not REPORT:
        return
    data = {}
    if os.path.exists(REPORT):
        with open(REPORT) as f:
            data = json.load(f)
    data[section] = payload
    data["_tolerance"] = {"rtol": U.RTOL, "atol": U.ATOL, "literal": "|got - want| <= atol + rtol * |want|",
                          "condition_aware": "|got - want| <= atol + rtol * max(|want|, sum of |terms|) (tests/_util.py)"}
    with open(REPORT, "w") as f:
        json.dump(data, f, indent=1, sort_keys=True)


def _ops():
    from bez_isaacgym_b200 import ops
    return ops


def ulp_err(got, want):
    g, w = got.double().numpy(), want.double().numpy()
    sp = np.spacing(np.abs(want.numpy()).astype(np.float32)).astype(np.float64)
    e = np.abs(g - w) / sp
    e[np.isnan(g) & np.isnan(w)] = 0.0
    e[(g == w)] = 0.0
    return e


def float_stats(got, want, scale=None):
    got, want = got.detach().cpu().float(), want.detach().cpu().float()
    both_nan = got.isnan() & want.isnan()
    diff = (got - want).abs()
    lit = (diff <= U.ATOL + U.RTOL * want.abs()) | both_nan | (got == want)
    out = {"elements": int(got.numel()), "literal_pass_fraction": float(lit.double().mean()), "literal_failures": int((~lit).sum()),
           "bit_identical_fraction": float(((got == want) | both_nan).double().mean()),
           "max_abs_err": float(torch.nan_to_num(diff, nan=0.0, posinf=0.0).max()) if got.numel() else 0.0,
           "max_ulp_err": float(np.nanmax(ulp_err(got, want))) if got.numel() else 0.0}
    if scale is not None:
        ref = torch.maximum(want.abs(), scale.expand_as(want))
        cond = (diff <= U.ATOL + U.RTOL * ref) | both_nan | (got == want)
        out["condition_aware_pass_fraction"] = float(cond.double().mean())
        out["condition_aware_failures"] = int((~cond).sum())
    return out


def tie_bands(st, goal, ball_init):
    """Per-rule tie-band membership (documented bands: 2 ulp for norm-fed thresholds, 4 ulp for the atan2-fed one)."""
    v = U.views(st)
    n_goal = torch.linalg.norm(goal - v["ball_pos"][:, 0:2], dim=1)
    strayed = torch.linalg.norm(v["bez_pos"][:, 0:2], dim=1)
    kicked = torch.linalg.norm(v["ball_pos"][:, 0:2] - ball_init, dim=1)
    u = (goal - v["ball_pos"][:, 0:2]) / n_goal.unsqueeze(1)
    ui = (goal - ball_init) / torch.linalg.norm(goal - ball_init, dim=1, keepdim=True)
    ang = (torch.atan2(ui[:, 1], ui[:, 0]) - torch.atan2(u[:, 1], u[:, 0])).abs()
    return {"rule2_strayed_gt_0.5 (2 ulp)": (strayed - 0.5).abs() <= 2 * U.ulp(0.5),
            "rule4_ball_to_goal_lt_0.05 (2 ulp)": (n_goal - 0.05).abs() <= 2 * U.ulp(0.05),
            "branch_kicked_gt_0.3 (2 ulp)": (kicked - 0.3).abs() <= 2 * U.ulp(0.3),
            "rule3_goal_angle_gt_1.5708 (4 ulp)": (ang - 1.5708).abs() <= 4 * U.ulp(1.5708)}


# ----------------------------------------------------------------------------------------------- the fused step, C ABI
@pytest.mark.parametrize("n", [4096, 262144, 1048576])
def test_fused_step_parity_at_baseline_sizes(n):
    from oracle import task_oracle as to
    from oracle.philox_ref import reset_uniforms
    ops = _ops()
    seed = 17
    st = sg.make_state(n, seed=500 + (n % 97), filler=(n <= 262144))
    goal, ball_init, default, lower, upper = U.constants(n)
    init_root = sg.make_initial_root_states(n)
    cpu = st.clone()
    orc = to.KickStepOracle(n, cpu.root_states, cpu.dof_state, cpu.rigid_body, cpu.net_contact, default, lower, upper, goal, ball_init,
                            torch.tensor([0.0, 0.0]), init_root,
                            reset_uniforms=lambda step: torch.from_numpy(reset_uniforms(seed, step, n)))
    progress0, reset0 = sg.make_bookkeeping(n, seed=n + 1, p_reset=0.02)
    progress0[:4] = torch.tensor([897, 898, 899, 900])
    orc.progress_buf[:] = progress0
    orc.reset_buf[:] = reset0
    d = st.to("cuda")
    cfg = ops.make_task_cfg(num_bodies=st.num_bodies)
    obs = torch.zeros(n, 54, device="cuda"); rew = torch.zeros(n, device="cuda")
    reset, progress = reset0.cuda(), progress0.cuda()
    timeout = torch.zeros(n, dtype=torch.long, device="cuda")
    prev_d = torch.zeros(n, 3, device="cuda")
    g_d, b_d, ir_d = goal.cuda(), ball_init.cuda(), init_root.cuda()
    steps = []
    for step in range(2):                 # step 0 reads the zero prev_lin_vel buffer, step 1 the reference's aliasing
        if step > 0:
            fresh = sg.make_state(n, seed=900 + step + (n % 89), filler=False)
            for name in ("root_states", "net_contact"):
                getattr(cpu, name).copy_(getattr(fresh, name)); getattr(d, name).copy_(getattr(fresh, name).cuda())
            imu = fresh.rigid_body.view(n, -1, 13)[:, bm.IMU_BODY]
            cpu.rigid_body.view(n, -1, 13)[:, bm.IMU_BODY] = imu
            d.rigid_body.view(n, -1, 13)[:, bm.IMU_BODY] = imu.cuda()
        prev_before = orc.prev_lin_vel.clone().float() if step == 0 else None
        want_obs, want_rew, want_reset, want_timeout = orc.post_physics_step()
        ops.post_physics(d.dof_state, d.rigid_body, d.root_states, d.net_contact, g_d, b_d, ir_d, reset, progress, timeout, cfg,
                         obs, rew, prev_lin_vel=prev_d if step == 0 else None, seed=seed, step=step)
        torch.cuda.synchronize()
        after = sg.SimState(cpu.root_states, cpu.dof_state, cpu.rigid_body, cpu.net_contact, n, st.num_bodies)
        bands = tie_bands(after, goal, ball_init)
        band = torch.zeros(n, dtype=torch.bool)
        for b in bands.values():
            band |= b
        got, got_rew, got_reset = obs.cpu(), rew.cpu(), reset.cpu()
        mism = got_reset != want_reset
        rew_scale = U.reward_scale(after, goal, ball_init, default)
        rew_lit = ((got_rew - want_rew).abs() <= U.ATOL + U.RTOL * want_rew.abs()) | (got_rew == want_rew)
        rec = {
            "bit_exact": {
                "dof_pos_vel (obs 0:36)": bool(torch.equal(got[:, 0:36], want_obs[:, 0:36])),
                "imu_ang_vel (obs 39:42)": bool(torch.equal(got[:, 39:42], want_obs[:, 39:42])),
                "feet_bits (obs 44:52)": bool(torch.equal(got[:, 44:52], want_obs[:, 44:52])),
                "ball_init (obs 52:54)": bool(torch.equal(got[:, 52:54], want_obs[:, 52:54])),
                "timeout_buf": bool(torch.equal(timeout.cpu(), want_timeout)),
                "progress_buf": bool(torch.equal(progress.cpu(), orc.progress_buf)),
                "dof_state after masked reset": bool(torch.equal(d.dof_state.cpu(), cpu.dof_state)),
                "root_states after masked reset": bool(torch.equal(d.root_states.cpu(), cpu.root_states)),
                "net_contact after in-place filter": bool(torch.equal(d.net_contact.cpu(), cpu.net_contact))},
            "imu_lin_acc (obs 36:39)": float_stats(got[:, 36:39], want_obs[:, 36:39], U.imu_term_scale(after, prev_before)),
            "off_orn (obs 42:44)": float_stats(got[:, 42:44], want_obs[:, 42:44]),
            "reward (outside tie bands)": float_stats(got_rew[~band], want_rew[~band], rew_scale[~band]),
            "reward (all envs) literal failures": int((~rew_lit).sum()),
            "reset_mask": {"envs": n, "resets_fired": int(want_reset.sum()), "mismatches": int(mism.sum()),
                           "mismatches_outside_tie_bands": int((mism & ~band).sum()),
                           "tie_band_population": {k: int(b.sum()) for k, b in bands.items()},
                           "tie_band_flipped": {k: int((b & mism).sum()) for k, b in bands.items()},
                           "reward_branch_or_rule_flipped_in_band": int((band & ~rew_lit).sum())},
        }
        steps.append(rec)
        assert all(rec["bit_exact"].values()), rec["bit_exact"]
        assert rec["reset_mask"]["mismatches_outside_tie_bands"] == 0
        assert rec["imu_lin_acc (obs 36:39)"]["condition_aware_failures"] == 0
        assert rec["off_orn (obs 42:44)"]["literal_failures"] == 0
        assert rec["reward (outside tie bands)"]["condition_aware_failures"] == 0
        assert rec["imu_lin_acc (obs 36:39)"]["literal_pass_fraction"] > 0.999
        reset.copy_(want_reset.cuda())        # a tie-band env must not fork the trajectories
    record(f"fused_step_c_abi_{n}_envs", {"steps": steps, "oracle": "oracle.task_oracle.KickStepOracle (pinned bit-exact to the "
                                          "reference's own jit functions and KickEnv.step, tests/test_oracle_pinning.py)"})


def test_observation_kernel_with_random_prev_lin_vel_262144_envs():
    """``compute_imu`` in its general contract (an arbitrary ``prev_lin_vel`` buffer, |a| = |v - prev| / dt ~ 25): the mat-vec's
    terms are ~50x its result, the case the condition-aware bound was introduced for.  The literal pass fraction is recorded."""
    ops = _ops()
    n = 262144
    st = sg.make_state(n, seed=7)
    goal, ball_init, *_ = U.constants(n)
    prev = 0.3 * torch.randn(n, 3, generator=torch.Generator().manual_seed(5))
    want, _, _ = U.oracle_observations(st, prev, goal, ball_init)
    d = st.to("cuda")
    obs = torch.empty(n, 54, device="cuda")
    ops.compute_observations(d.dof_state, d.rigid_body, d.root_states, d.net_contact, goal.cuda(), ball_init.cuda(),
                             ops.make_task_cfg(num_bodies=st.num_bodies), obs, prev_lin_vel=prev.cuda())
    got = obs.cpu()
    imu = float_stats(got[:, 36:39], want[:, 36:39], U.imu_term_scale(st, prev))
    assert imu["condition_aware_failures"] == 0 and imu["literal_pass_fraction"] > 0.999
    record("observation_kernel_random_prev_lin_vel_262144_envs", {"imu_lin_acc (obs 36:39)": imu,
                                                                  "off_orn (obs 42:44)": float_stats(got[:, 42:44], want[:, 42:44])})


def test_kick_env_step_parity_4096_envs():
    """BASELINE configs[1]: 8 steps of ``KickEnv.step`` at the repo-default 4 096 envs against the oracle stepping the same
    state (the simulator stand-in moves the state between steps identically on both sides)."""
    from bez_isaacgym_b200.synthetic_sim import SyntheticGym
    from bez_isaacgym_b200.tasks import KickEnv
    from oracle import task_oracle as to
    from oracle.philox_ref import reset_uniforms
    n = 4096
    goal, ball_init, default, lower, upper = U.constants(n)
    init_root = sg.make_initial_root_states(n)
    cfg = bm.default_task_cfg(n)
    cfg["seed"] = 23
    st = sg.make_state(n, seed=61)
    frame = [0]

    def move(sim):                            # gym.simulate + refresh_*: new root / rigid-body / contact state, dof drift
        frame[0] += 1
        fresh = sg.make_state(n, seed=7000 + frame[0])
        drift = 0.01 * torch.randn(n * 18, 2, generator=torch.Generator().manual_seed(frame[0]))
        for tgt, is_gpu in ((sim, True), (cpu, False)):
            for name in ("root_states", "rigid_body", "net_contact"):
                getattr(tgt, name).copy_(getattr(fresh, name).cuda() if is_gpu else getattr(fresh, name))
            tgt.dof_state.add_(drift.cuda() if is_gpu else drift)

    env = KickEnv(cfg, "cuda:0", 0, True, sim=SyntheticGym(n, device="cuda:0", state=st.clone()))
    cpu = sg.SimState(env.root_states.cpu(), env.dof_state.cpu(), env.rigid_body.cpu(), env.net_contact.cpu(), n, st.num_bodies)
    orc = to.KickStepOracle(n, cpu.root_states, cpu.dof_state, cpu.rigid_body, cpu.net_contact, default, lower, upper, goal,
                            ball_init, torch.tensor([0.0, 0.0]), init_root)
    progress0, _ = sg.make_bookkeeping(n, seed=3)
    env.progress_buf.copy_(progress0); orc.progress_buf[:] = progress0
    orc.reset_buf[:] = env.reset_buf.cpu()
    env.sim.on_simulate = move
    out = []
    for step in range(8):
        actions = sg.make_actions(n, seed=200 + step)
        orc.pre_physics_step(actions)
        orc.reset_uniforms = lambda _s, k=env._rng_step + 1: torch.from_numpy(reset_uniforms(env._seed, k, n))
        prev_before = orc.prev_lin_vel.clone().float() if step == 0 else None
        od, rew, done, extras = env.step(actions.cuda())          # moves BOTH states inside sim.simulate()
        want_obs, want_rew, want_reset, want_timeout = orc.post_physics_step()
        torch.cuda.synchronize()
        after = sg.SimState(cpu.root_states, cpu.dof_state, cpu.rigid_body, cpu.net_contact, n, st.num_bodies)
        bands = tie_bands(after, goal, ball_init)
        band = torch.zeros(n, dtype=torch.bool)
        for b in bands.values():
            band |= b
        got = od["obs"].cpu()
        assert torch.equal(env.targets.cpu(), orc.targets)
        assert torch.equal(got[:, 0:36], want_obs[:, 0:36]) and torch.equal(got[:, 39:42], want_obs[:, 39:42])
        assert torch.equal(got[:, 44:54], want_obs[:, 44:54])
        assert torch.equal(extras["time_outs"].cpu(), want_timeout) and torch.equal(env.progress_buf.cpu(), orc.progress_buf)
        assert torch.equal(env.dof_state.cpu(), cpu.dof_state)
        mism = done.cpu() != want_reset
        assert not bool((mism & ~band).any())
        imu = float_stats(got[:, 36:39], want_obs[:, 36:39], U.imu_term_scale(after, prev_before))
        orn = float_stats(got[:, 42:44], want_obs[:, 42:44])
        rw = float_stats(rew.cpu()[~band], want_rew[~band], U.reward_scale(after, goal, ball_init, default)[~band])
        assert imu["condition_aware_failures"] == 0 and orn["literal_failures"] == 0 and rw["condition_aware_failures"] == 0
        out.append({"imu_lin_acc": imu, "off_orn": orn, "reward": rw, "resets_fired": int(want_reset.sum()),
                    "reset_mismatches": int(mism.sum()), "tie_band_population": {k: int(b.sum()) for k, b in bands.items()}})
        env.reset_buf.copy_(want_reset.cuda())
    assert sum(o["resets_fired"] for o in out) > 0
    record("kick_env_step_4096_envs_8_steps", {"steps": out})


# ----------------------------------------------------------------------------------------------- learner kernels
def test_learner_parity_at_baseline_shapes():
    from oracle import rl_games_oracle as rg
    ops = _ops()
    rep = {}
    # GAE at 262 144 x 32 (configs[3]) and 4 096 x 32 (configs[2])
    for n in (4096, 262144):
        T = 32
        rewards, values, dones, last_values, last_dones = sg.make_rollout(n, T, seed=n, p_done=0.01)
        want = rg.discount_values(last_dones.float(), last_values, dones.float(), values, rewards, 0.99, 0.95)
        advs = torch.empty(T, n, 1, device="cuda"); rets = torch.empty_like(advs)
        ops.gae(rewards.cuda(), values.cuda(), dones.cuda(), last_values.cuda(), last_dones.cuda(), 0.99, 0.95, advs, rets)
        scale = values.abs() + rewards.abs() + 1.0
        a, r = float_stats(advs, want, scale), float_stats(rets, want + values, scale)
        assert a["condition_aware_failures"] == 0 and r["condition_aware_failures"] == 0
        rep[f"gae_{n}x{T}"] = {"advantages": a, "returns": r}
    # RunningMeanStd train forward, three successive minibatches of 32 768 x 54
    m, c = 32768, 54
    g = torch.Generator().manual_seed(1)
    orc = rg.RunningMeanStd(c)
    mean = torch.zeros(c, dtype=torch.float64, device="cuda"); var = torch.ones(c, dtype=torch.float64, device="cuda")
    count = torch.ones(1, dtype=torch.float64, device="cuda")
    acc = torch.empty(1 + 2 * c, dtype=torch.float64, device="cuda")
    part = torch.empty(ops.rms_scratch_doubles(c), dtype=torch.float64, device="cuda")
    allx = []
    for it in range(3):
        x = torch.randn(m, c, generator=g) * (torch.rand(c, generator=g) * 3 + 0.1) + torch.randn(c, generator=g) + it
        allx.append(x)
        want = orc(x)
        pivot = mean.clone()
        xd = x.cuda()
        ops.rms_moments(xd, pivot, acc, part); ops.rms_merge(acc, pivot, mean, var, count)
        y = torch.empty_like(xd)
        ops.rms_normalize(xd, mean, var, y)
    cat = torch.cat(allx).double()
    # restatement-free reference for the mean: the (0, 1, 1) start is one pseudo-sample at 0, so mean = sum(x) / (1 + N) in fp64
    tot = 1.0 + cat.shape[0]
    mu2 = cat.sum(0) / tot
    rep["running_mean_std_3x32768x54"] = {
        "running_mean_max_rel_err_vs_oracle": float(((mean.cpu() - orc.running_mean).abs() / orc.running_mean.abs().clamp_min(1e-12)).max()),
        "running_var_max_rel_err_vs_oracle": float(((var.cpu() - orc.running_var).abs() / orc.running_var).max()),
        "running_mean_max_abs_err_vs_fp64_two_pass": float((mean.cpu() - mu2).abs().max()),
        "count": float(count.item()), "normalised_output": float_stats(y, want)}
    assert count.item() == tot and float((mean.cpu() - mu2).abs().max()) < 1e-9
    assert torch.allclose(var.cpu(), orc.running_var, rtol=2e-5, atol=1e-7)
    # PPO loss at the reference minibatch
    mb = sg.make_minibatch(m, seed=4)
    mu = mb["mu"].clone().requires_grad_(True); vals = mb["values"].clone().requires_grad_(True)
    logstd = mb["logstd"].clone().requires_grad_(True)
    o = rg.ppo_loss(dict(mb, mu=mu, values=vals, logstd=logstd))
    o["loss"].backward()
    dv = {k: v.cuda().contiguous() for k, v in mb.items()}
    stats = torch.empty(8, dtype=torch.float64, device="cuda")
    pp = torch.empty(ops.ppo_scratch_doubles(), dtype=torch.float64, device="cuda")
    g_mu = torch.empty(m, 18, device="cuda"); g_v = torch.empty(m, device="cuda"); g_ls = torch.empty(18, device="cuda")
    nlp = torch.empty(m, device="cuda")
    ops.ppo_loss(dv["actions"], dv["mu"], dv["logstd"], dv["old_mu"], dv["old_sigma"], dv["values"].view(-1), dv["old_values"].view(-1),
                 dv["returns"].view(-1), dv["old_neglogp"], dv["advantages"], ops.make_ppo_cfg(), stats, pp, grad_mu=g_mu,
                 grad_values=g_v, grad_logstd=g_ls, neglogp_out=nlp)
    s = stats.cpu()
    terms = {k: {"got": float(s[i]), "want": float(o[k]), "rel_err": abs(float(s[i]) - float(o[k])) / max(abs(float(o[k])), 1e-12)}
             for i, k in [(0, "loss"), (1, "a_loss"), (2, "c_loss"), (3, "entropy"), (4, "b_loss"), (5, "kl")]}
    for k, t in terms.items():
        assert math.isclose(t["got"], t["want"], rel_tol=2e-5, abs_tol=2e-6), (k, t)
    rep["ppo_loss_32768"] = {"terms": terms, "neglogp": float_stats(nlp, o["neglogp"].detach()),
                             "grad_mu_max_rel_err": float(((g_mu.cpu() - mu.grad).abs().max() / mu.grad.abs().max())),
                             "grad_values_max_rel_err": float(((g_v.cpu() - vals.grad.view(-1)).abs().max() / vals.grad.abs().max())),
                             "grad_logstd_max_rel_err": float(((g_ls.cpu() - logstd.grad).abs().max() / logstd.grad.abs().max()))}
    record("learner_kernels", rep)
