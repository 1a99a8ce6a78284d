"""fp32 restatements of the fused step's IMU / reward math and of the PPO neglogp in the kernels' operation order: every ``*``, ``+``,
``-`` and ``/`` is one correctly rounded fp32 torch op (the library is built with ``-fmad=false``) and every square root is a float64
root rounded once, so where a kernel promises IEEE results these agree with it bit for bit -- also for operands outside the branch-free
fast sequences' range (``Mth`` in ``csrc/bezk_common.cuh``), where only the kernels' exact retry gets the IEEE answer.  ``atan2`` /
``sin`` / ``cos`` are torch's, which can differ from the device's in the last bits; the callers keep inputs away from the thresholds
those feed.  Pinned against ``oracle/`` on ordinary inputs by ``tests/test_exact_retry_reference.py``."""
import torch

KICK_OUTCOMES = ("fell", "strayed", "wide", "scored", "timeout")
WALK_OUTCOMES = ("fell", "reached", "out", "timeout")
TWO_PI = torch.tensor(6.283185307179586, dtype=torch.float32)


def c(x):
    return torch.tensor(x, dtype=torch.float32)


def sqrt32(x):
    """Correctly rounded fp32 square root (torch's CPU fp32 sqrt is not always)."""
    return x.double().sqrt().float()


def imu_lin_acc(q, v, prev, dt, max_acc):
    """Observation columns 36:39 (``imu_term``): the real-first rotation matrix of the xyzw quaternion ``q`` (n, 4) times
    (v - prev) / dt - gravity, clamped to +-max_acc with NaN propagating."""
    dt = c(dt)
    a = [(v[:, 0] - prev[:, 0]) / dt - c(0.0), (v[:, 1] - prev[:, 1]) / dt - c(0.0), (v[:, 2] - prev[:, 2]) / dt - c(-1.0)]
    r, i, j, k = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    two_s = c(2.0) / (((r * r + i * i) + j * j) + k * k)
    one = c(1.0)
    m = [[one - two_s * (j * j + k * k), two_s * (i * j - k * r), two_s * (i * k + j * r)],
         [two_s * (i * j + k * r), one - two_s * (i * i + k * k), two_s * (j * k - i * r)],
         [two_s * (i * k - j * r), two_s * (j * k + i * r), one - two_s * (i * i + j * j)]]
    t = [(m[row][0] * a[0] + m[row][1] * a[1]) + m[row][2] * a[2] for row in range(3)]
    return torch.stack([torch.clamp(x, -max_acc, max_acc) for x in t], 1)


def pos_sq(dof_pos, default):
    """sum_j (default_j - pos_j)^2, accumulated j = 0..17 in order."""
    s = torch.zeros(dof_pos.shape[0])
    for j in range(dof_pos.shape[1]):
        d = default[:, j] - dof_pos[:, j]
        s = s + d * d
    return s


def _atan2_z(y, x):
    """``atan2f_z``: atan2 with atan2(+-0, x > 0) = +-0."""
    return torch.where((y == 0) & (x > 0), y, torch.atan2(y, x))


def sumsq(*xs):
    s = xs[0] * xs[0]
    for x in xs[1:]:
        s = s + x * x
    return s


def _fire(rules, rew, reset_cur):
    """Apply the termination rules in order: ``rules`` = [(mask, value)], the last firing rule sets the reward and the class."""
    n = rew.shape[0]
    reset = reset_cur.clone()
    cls = torch.full((n,), -1, dtype=torch.long)
    for k, (mask, value) in enumerate(rules):
        reset = torch.where(mask, torch.ones_like(reset), reset)
        rew = torch.where(mask, value, rew)
        cls = torch.where(mask, torch.full_like(cls, k), cls)
    return rew, reset, cls


def kick_step(bez, ball, ball_v, goal, ball_init, v, w, psq, bez_init, progress, max_len, reset_cur):
    """``reward_term``: (rew, reset, outcome class (-1: none), terms (6, n))."""
    dbx, dby = ball[:, 0] - bez[:, 0], ball[:, 1] - bez[:, 1]
    nbb = sqrt32(sumsq(dbx, dby))
    vel_fwd = (dbx / nbb) * v[:, 0] + (dby / nbb) * v[:, 1]
    dgx, dgy = goal[:, 0] - ball[:, 0], goal[:, 1] - ball[:, 1]
    n_goal = sqrt32(sumsq(dgx, dgy))
    ugx, ugy = dgx / n_goal, dgy / n_goal
    ball_fwd = ugx * ball_v[:, 0] + ugy * ball_v[:, 1]
    dix, diy = goal[:, 0] - ball_init[:, 0], goal[:, 1] - ball_init[:, 1]
    n_init = sqrt32(sumsq(dix, diy))
    angle_diff = (_atan2_z(diy / n_init, dix / n_init) - _atan2_z(ugy, ugx)).abs()
    vel_r = sqrt32(sumsq(v[:, 0], v[:, 1], v[:, 2], w[:, 0], w[:, 1], w[:, 2])) * c(0.05)
    pos_r = sqrt32(psq) * c(0.05)
    height = (c(0.325) - bez[:, 2]).abs() * c(1.0)
    kx, ky = ball[:, 0] - ball_init[:, 0], ball[:, 1] - ball_init[:, 1]
    far = sqrt32(sumsq(kx, ky)) > 0.3
    far_r = ball_fwd * c(0.1) - (height + (vel_r + pos_r))
    near_r = ball_fwd * c(0.1) + (vel_fwd * c(0.05) - height)
    rew = torch.where(far, far_r, near_r)
    tx, ty = bez[:, 0] - c(bez_init[0]), bez[:, 1] - c(bez_init[1])
    p = progress.float()
    minus1 = torch.full_like(rew, -1.0)
    rules = [(bez[:, 2] < 0.275, minus1), (sqrt32(sumsq(tx, ty)) > 0.5, minus1), (angle_diff > 1.5708, minus1),
             (n_goal < 0.05, c(1.0) * (c(100.0) - c(100.0) * (p / c(float(max_len))))), (progress >= max_len, torch.zeros_like(rew))]
    rew, reset, cls = _fire(rules, rew, reset_cur)
    fired, zero = cls >= 0, torch.zeros_like(rew)
    terms = [ball_fwd * c(0.1), torch.where(far, zero, vel_fwd * c(0.05)), -height, torch.where(far, -vel_r, zero),
             torch.where(far, -pos_r, zero)]
    terms = torch.stack([torch.where(fired, zero, t) for t in terms] + [torch.where(fired, rew, zero)])
    return rew, reset, cls, terms


def yaw_mod_2pi(q):
    x, y, z, w = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    yaw = _atan2_z(c(2.0) * (w * z + x * y), ((w * w + x * x) - y * y) - z * z)
    return torch.where(yaw < 0, yaw + TWO_PI, yaw)


def walk_step(task, bez, q, v, w, psq, goal, goal_angle, bez_init, progress, max_len, reset_cur):
    """``reward_walk`` (task "walk", ``goal`` (n, 2)) / ``reward_orient`` (task "orient", ``goal_angle`` (n,)): (rew, reset, outcome
    class, terms (5, n))."""
    qx, qy, qz, qw = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    a_z = c(1.0) * (c(2.0) * (qw * qw) - c(1.0))
    b_z = ((qx * c(0.0) - qy * c(0.0)) * qw) * c(2.0)
    dot = (qx * c(0.0) + qy * c(0.0)) + qz * c(1.0)
    up = (a_z + b_z) + (qz * dot) * c(2.0)
    vel6 = sqrt32(sumsq(v[:, 0], v[:, 1], v[:, 2], w[:, 0], w[:, 1], w[:, 2]))
    vel_lin, vel_ang = sqrt32(sumsq(v[:, 0], v[:, 1], v[:, 2])), sqrt32(sumsq(w[:, 0], w[:, 1], w[:, 2]))
    pos = sqrt32(psq)
    dist_h = (c(1.0) - up).abs()
    vel_s, pos_s = vel6 * c(0.05), pos * c(0.05)
    hvp = -((vel_s + pos_s) + dist_h)
    if task == "walk":
        dx, dy = goal[:, 0] - bez[:, 0], goal[:, 1] - bez[:, 1]
        n_goal = sqrt32(sumsq(dx, dy))
        ux, uy = dx / n_goal, dy / n_goal
        lead = (ux * v[:, 0] + uy * v[:, 1]) * c(10.0)
        scale, close = c(5.0), n_goal < 0.05
        ix, iy = goal[:, 0] - c(0.0), goal[:, 1] - c(0.0)
        n_i = sqrt32(sumsq(ix, iy))
        out = (_atan2_z(iy / n_i, ix / n_i) - _atan2_z(uy, ux)).abs() > 1.5708
        out_value = -100.0
    else:
        yaw = yaw_mod_2pi(q)
        ang = goal_angle - _atan2_z(torch.sin(yaw), torch.cos(yaw))
        lead, scale, close = ang.abs() * c(-0.5), c(0.05), ang < 0.05
        tx, ty = bez[:, 0] - c(bez_init[0]), bez[:, 1] - c(bez_init[1])
        out, out_value = sqrt32(sumsq(tx, ty)) > 0.3, -5.0
    rew = torch.where(close, hvp, (lead - (dist_h + scale * pos_s)) * c(1.0))
    state = close.float() + (pos < 0.15).float() + (vel_ang < 0.1).float() + (vel_lin < 0.1).float()
    p = progress.float()
    rules = [(up < 0.7, torch.full_like(rew, -100.0)),
             (state == 4.0, c(1.0) * (c(1000.0) - c(1000.0) * (p / c(float(max_len))))),
             (out, torch.full_like(rew, out_value)), (progress >= max_len, torch.zeros_like(rew))]
    rew, reset, cls = _fire(rules, rew, reset_cur)
    fired, zero = cls >= 0, torch.zeros_like(rew)
    terms = [torch.where(close, zero, lead), -dist_h, torch.where(close, -vel_s, zero), torch.where(close, -pos_s, -(scale * pos_s))]
    terms = torch.stack([torch.where(fired, zero, t) for t in terms] + [torch.where(fired, rew, zero)])
    return rew, reset, cls, terms


NLP_CONST = torch.tensor(0.5 * 1.8378770664093453 * 18.0, dtype=torch.float64).float()


def neglogp(actions, mu, sigma, logstd):
    """models.py neglogp as the kernels form it: zz = (a - mu) / sigma, sq = sum_j zz * zz in order j = 0..17, then
    (0.5 * sq + 0.5 * log(2 pi) * 18) + sum_j logstd_j (summed in order).  ``sigma``: (18,) or (m, 18) fp32."""
    sigma = torch.broadcast_to(sigma, actions.shape)
    sq = torch.zeros(actions.shape[0])
    lsum = c(0.0)
    for j in range(actions.shape[1]):
        zz = (actions[:, j] - mu[:, j]) / sigma[:, j]
        sq = sq + zz * zz
        lsum = lsum + logstd[j]
    return (c(0.5) * sq + NLP_CONST) + lsum


def outside_window(x):
    """True where |x| lies outside the branch-free operators' range 2^-60 .. 2^60 (NaN and inf are outside)."""
    a = x.double().abs()
    return ~((a >= 2.0 ** -60) & (a <= 2.0 ** 60))

