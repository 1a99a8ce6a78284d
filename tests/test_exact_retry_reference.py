"""CPU: the kernel-order restatements of ``tests/exact_retry_reference.py`` against the oracle (``oracle/task_oracle.py``,
``oracle/rl_games_oracle.py``) on ordinary inputs, and bit for bit on the hand-made extremes the GPU retry tests rely on."""
import torch

from bez_isaacgym_b200 import bez_model as bm
from oracle import rl_games_oracle as rg
from oracle import task_oracle as to
from tests import _util as U
from tests import exact_retry_reference as X

DT, MAX_ACC = 0.01667, 2.0 * 9.81
NB = bm.BODIES_NO_CLEATS


def _unit_quats(n, g):
    q = torch.randn(n, 4, generator=g)
    return q / torch.linalg.norm(q, dim=1, keepdim=True)


def test_imu_matches_the_oracle():
    g = torch.Generator().manual_seed(1)
    n = 4096
    q = _unit_quats(n, g) * (1 + 0.1 * torch.rand(n, 1, generator=g))            # non-unit quaternions too
    v, prev, w = torch.randn(n, 3, generator=g), torch.randn(n, 3, generator=g), torch.randn(n, 3, generator=g)
    want, _ = to.imu(q, v, w, prev, torch.tensor([[0.0, 0.0, -1.0]]).repeat(n, 1), DT)
    got = X.imu_lin_acc(q, v, prev, DT, MAX_ACC)
    scale = ((v - prev) / DT + torch.tensor([0.0, 0.0, 1.0])).abs().sum(1, keepdim=True) * 2
    U.assert_close(got, want[:, 0:3], scale=scale, what="imu")


def test_imu_extremes_are_ieee():
    """|q|^2 = 1e38: two_s = 2e-38 (a normal number), so m22 = 1 - 2 = -1 and the z acceleration of a resting body is -1."""
    q = torch.tensor([[0.0, 1e19, 0.0, 0.0]])
    z = torch.zeros(1, 3)
    got = X.imu_lin_acc(q, z, z, DT, MAX_ACC)
    assert got.tolist() == [[0.0, 0.0, -1.0]]
    assert bool(X.outside_window(((q * q).sum(1))).all())


def _kick_inputs(n, g):
    bez = torch.cat((torch.randn(n, 2, generator=g) * 0.2, 0.25 + 0.1 * torch.rand(n, 1, generator=g)), 1)
    ball = torch.randn(n, 2, generator=g) * 0.5 + torch.tensor([1.0, 0.0])
    ball_v = torch.randn(n, 2, generator=g)
    goal = torch.tensor([[4.5, 0.0]]).repeat(n, 1)
    ball_init = torch.tensor([[1.0, 0.0]]).repeat(n, 1)
    v, w = torch.randn(n, 3, generator=g), torch.randn(n, 3, generator=g)
    dof = torch.randn(n, 18, generator=g) * 0.1
    progress = torch.randint(800, 905, (n,), generator=g)
    return bez, ball, ball_v, goal, ball_init, v, w, dof, progress


def test_kick_reward_matches_the_oracle():
    g = torch.Generator().manual_seed(2)
    n, m = 8192, 900
    bez, ball, ball_v, goal, ball_init, v, w, dof, progress = _kick_inputs(n, g)
    default = torch.zeros(n, 18)
    reset_in = torch.zeros(n, dtype=torch.long)
    rew, reset, cls, terms = X.kick_step(bez, ball, ball_v, goal, ball_init, v, w, X.pos_sq(dof, default), (0.0, 0.0), progress, m,
                                         reset_in)
    want_rew, want_reset = to.reward(dof, default, v, w, bez, torch.cat((ball, torch.zeros(n, 1)), 1),
                                     torch.cat((ball_v, torch.zeros(n, 1)), 1), goal, ball_init, torch.zeros(2), reset_in, progress, m)
    root = torch.zeros(n, 2, 13)
    root[:, 0, 0:3], root[:, 1, 0:2], root[:, 1, 7:9] = bez, ball, ball_v
    st = type("S", (), dict(root_states=root.view(-1), dof_state=torch.zeros(n * 36), rigid_body=torch.zeros(n * NB * 13),
                            net_contact=torch.zeros(n * NB * 3), num_envs=n))
    ok = ~(U.reward_tie_band(st, goal, ball_init) | ((bez[:, 2] - 0.275).abs() <= 4 * U.ulp(0.275)))
    assert torch.equal(reset[ok], want_reset[ok])
    assert bool((cls >= 0).any()) and bool((cls == -1).any())
    U.assert_close(rew[ok], want_rew[ok], scale=terms[:, ok].abs().sum(0), what="kick reward")
    assert torch.equal(terms[-1][cls >= 0], rew[cls >= 0])


def test_walk_and_orient_rewards_match_the_oracle():
    g = torch.Generator().manual_seed(3)
    n, m = 8192, 900
    q = _unit_quats(n, g)
    q[: n // 2] = torch.tensor([0.0, 0.0, 0.0, 1.0]) + 0.05 * torch.randn(n // 2, 4, generator=g)
    v, w = torch.randn(n, 3, generator=g) * 0.1, torch.randn(n, 3, generator=g) * 0.1
    dof = torch.randn(n, 18, generator=g) * 0.05
    default = torch.zeros(n, 18)
    bez = torch.cat((torch.randn(n, 2, generator=g) * 0.3, torch.full((n, 1), 0.4)), 1)
    goal = torch.randn(n, 2, generator=g)
    goal_angle = torch.rand(n, generator=g) * 2 - 1
    progress = torch.randint(800, 905, (n,), generator=g)
    reset_in = torch.zeros(n, dtype=torch.long)
    psq = X.pos_sq(dof, default)
    for task in ("walk", "orient"):
        rew, reset, cls, terms = X.walk_step(task, bez, q, v, w, psq, goal, goal_angle, (0.0, 0.0), progress, m, reset_in)
        if task == "walk":
            want_rew, want_reset = to.reward_walk(dof, default, v, w, bez, q, goal, reset_in, progress, m)
        else:
            want_rew, want_reset = to.reward_orient(dof, default, v, w, bez, q, goal_angle.view(n, 1), reset_in, progress,
                                                    torch.zeros(2), m)
        up, _, vel_lin, vel_ang, pos = to._walk_terms(dof, default, v, w, q, n)
        band = torch.zeros(n, dtype=torch.bool)
        for x, thr in ((up, 0.7), (pos, 0.15), (vel_lin, 0.1), (vel_ang, 0.1)):
            band |= (x - thr).abs() <= 4 * U.ulp(thr)
        assert torch.equal(reset[~band], want_reset.view(-1)[~band]), task
        assert bool((cls >= 0).any()) and bool((cls == -1).any())
        U.assert_close(rew[~band], want_rew.view(-1)[~band], scale=terms[:, ~band].abs().sum(0), what=task)


def test_win_rule_with_a_subnormal_angular_velocity():
    """The IEEE result the GPU tests expect for |w|^2 = 1e-40: vel_ang = 1e-20 < 0.1, so a close, still, upright robot has won."""
    n = 2
    q = torch.tensor([[0.0, 0.0, 0.0, 1.0]] * n)
    v, w = torch.zeros(n, 3), torch.tensor([[1e-20, 0.0, 0.0]] * n)
    assert bool(X.outside_window(w[:, 0] * w[:, 0]).all())
    bez = torch.tensor([[0.99, 1.49, 0.4]] * n)
    rew, reset, cls, _ = X.walk_step("walk", bez, q, v, w, torch.zeros(n), torch.tensor([[1.0, 1.5]] * n), None, (0.0, 0.0),
                                     torch.tensor([11, 11]), 900, torch.zeros(n, dtype=torch.long))
    assert cls.tolist() == [1, 1] and reset.tolist() == [1, 1]
    assert rew[0].item() == X.c(1000.0) - X.c(1000.0) * (X.c(11.0) / X.c(900.0))


def test_neglogp_matches_the_oracle():
    g = torch.Generator().manual_seed(4)
    m = 4096
    mu, logstd = torch.randn(m, 18, generator=g), torch.randn(18, generator=g) * 0.3
    sigma = torch.exp(logstd)
    a = mu + torch.randn(m, 18, generator=g) * sigma
    want = rg.neglogp(a, mu, sigma.expand(m, 18), logstd.expand(m, 18))
    U.assert_close(X.neglogp(a, mu, sigma, logstd), want, what="neglogp")
