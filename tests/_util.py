"""Shared helpers for the parity tests: synthetic inputs, oracle views, tolerances, tie bands.

Tolerances (BASELINE.json north_star): fp32 rtol 1e-5 / atol 1e-6 for observations, rewards, advantages,
returns; masks bit-exact.  Two documented refinements:

* condition-aware sums: where a result is a sum of products whose terms are much larger than the result
  (IMU mat-vec with |v/dt| ~ 50, reward sums), fp32 evaluation order alone (BLAS FMA vs separate
  mul/add) moves the result by ~1 ulp of the LARGEST TERM, so the bound is
  |a-b| <= atol + rtol * max(|b|, scale) with `scale` = sum of |terms| (the textbook forward error bound);
* threshold ties: masks must be bit-exact OUTSIDE a tie band |value - thr| <= k ulp(thr) (k = 2 for
  norm-fed rules, 4 for the atan2-fed rule); in-band envs are counted and reported (SURVEY 8a).
"""
import math

import numpy as np
import torch

from bez_isaacgym_b200 import bez_model as bm
from bez_isaacgym_b200 import synthetic_gym as sg

RTOL, ATOL = 1e-5, 1e-6


def views(st, cleats=False):
    n = st.num_envs
    root = st.root_states.view(n, 2, 13)
    rb = st.rigid_body.view(n, -1, 13)
    cf = st.net_contact.view(n, -1, 3)
    dof = st.dof_state.view(n, 18, 2)
    d = dict(dof_pos=dof[..., 0], dof_vel=dof[..., 1], bez_pos=root[:, 0, 0:3], ball_pos=root[:, 1, 0:3],
             ball_vel=root[:, 1, 7:10], quat=rb[:, bm.IMU_BODY, 3:7], lin=rb[:, bm.IMU_BODY, 7:10],
             ang=rb[:, bm.IMU_BODY, 10:13])
    if cleats:
        d["left_c"] = cf[:, bm.LEFT_CLEATS[0]:bm.LEFT_CLEATS[1], :]
        d["right_c"] = cf[:, bm.RIGHT_CLEATS[0]:bm.RIGHT_CLEATS[1], :]
    else:
        d["left_f"] = cf[:, bm.LEFT_FOOT_BODY, :]
        d["right_f"] = cf[:, bm.RIGHT_FOOT_BODY, :]
    return d


def constants(n, device="cpu"):
    return sg.make_constants(n, device)


def oracle_observations(st, prev_lin_vel, goal, ball_init, cleats=False, dt=0.01667):
    """Oracle obs on (a clone of) the CPU state; returns obs, filtered contact buffer, new prev."""
    from oracle import task_oracle as to
    st = st.clone()
    v = views(st, cleats)
    n = st.num_envs
    g = torch.tensor([[0.0, 0.0, -1.0]]).repeat(n, 1)
    prev = v["lin"] if prev_lin_vel is None else prev_lin_vel
    imu6, _ = to.imu(v["quat"], v["lin"], v["ang"], prev, g, dt)
    orn = to.off_orn(v["bez_pos"], v["quat"], goal)
    if cleats:
        feet = to.feet_cleats(v["left_c"], v["right_c"])
    else:
        feet = torch.cat((to.feet_no_cleats(v["left_f"]), to.feet_no_cleats(v["right_f"])), 1)
    obs = to.observations(v["dof_pos"], v["dof_vel"], imu6, orn, feet, ball_init)
    return obs, st.net_contact, v["lin"].clone()


def imu_term_scale(st, prev_lin_vel, dt=0.01667):
    """sum_j |R_ij a_j| bound (<= sqrt(3)|a| for a rotation-like R): scale of the IMU mat-vec terms."""
    v = views(st)
    prev = v["lin"] if prev_lin_vel is None else prev_lin_vel
    a = (v["lin"] - prev) / dt
    a = a - torch.tensor([0.0, 0.0, -1.0])
    return a.abs().sum(1, keepdim=True)


def assert_close(actual, expected, scale=None, rtol=RTOL, atol=ATOL, what=""):
    actual, expected = actual.detach().cpu(), expected.detach().cpu()
    assert actual.shape == expected.shape, f"{what}: shape {tuple(actual.shape)} vs {tuple(expected.shape)}"
    both_nan = torch.isnan(actual) & torch.isnan(expected)
    same_inf = torch.isinf(expected) & (actual == expected)
    ref = expected.abs()
    if scale is not None:
        ref = torch.maximum(ref, scale.expand_as(ref))
    ok = ((actual - expected).abs() <= atol + rtol * ref) | both_nan | same_inf
    if not bool(ok.all()):
        bad = (~ok).nonzero()
        i = tuple(bad[0].tolist())
        raise AssertionError(f"{what}: {bad.shape[0]} of {ok.numel()} elements outside rtol={rtol} atol={atol}; "
                             f"first at {i}: got {actual[i].item()!r} want {expected[i].item()!r}")


GUARD = 4096          # bytes each side


class Guarded:
    """Out-of-bounds WRITE canaries: every buffer ``make`` hands out lives between two guard bands filled with a sentinel;
    ``check`` asserts that the bands came back untouched."""

    def __init__(self):
        self.bufs = []

    def make(self, shape, dtype=torch.float32, fill=None):
        numel = 1
        for s in shape:
            numel *= s
        nbytes = numel * torch.empty((), dtype=dtype).element_size()
        pad = (-nbytes) % 16
        raw = torch.full((GUARD + nbytes + pad + GUARD,), 0x5A, dtype=torch.uint8, device="cuda")
        view = raw[GUARD:GUARD + nbytes].view(dtype).view(shape)
        if fill is not None:
            view.copy_(fill)
        self.bufs.append((raw, nbytes))
        return view

    def check(self):
        torch.cuda.synchronize()
        for raw, nbytes in self.bufs:
            assert bool((raw[:GUARD] == 0x5A).all()), "write BEFORE an output buffer"
            assert bool((raw[GUARD + nbytes:] == 0x5A).all()), "write PAST an output buffer"


def ulp(x):
    return float(np.spacing(np.float32(x)))


def reward_tie_band(st, goal, ball_init, bez_init_xy=(0.0, 0.0)):
    """Envs whose mask / reward branch hangs on a computed quantity within the documented tie band."""
    v = views(st)
    n_goal = torch.linalg.norm(goal - v["ball_pos"][:, 0:2], dim=1)
    strayed = torch.linalg.norm(v["bez_pos"][:, 0:2] - torch.tensor(bez_init_xy), dim=1)
    kicked = torch.linalg.norm(v["ball_pos"][:, 0:2] - ball_init, dim=1)
    u = (goal - v["ball_pos"][:, 0:2]) / n_goal.unsqueeze(1)
    ui = (goal - ball_init) / torch.linalg.norm(goal - ball_init, dim=1, keepdim=True)
    ang = (torch.atan2(ui[:, 1], ui[:, 0]) - torch.atan2(u[:, 1], u[:, 0])).abs()
    band = ((strayed - 0.5).abs() <= 2 * ulp(0.5)) | ((n_goal - 0.05).abs() <= 2 * ulp(0.05)) | \
           ((kicked - 0.3).abs() <= 2 * ulp(0.3)) | ((ang - 1.5708).abs() <= 4 * ulp(1.5708))
    return band


def reward_scale(st, goal, ball_init, default):
    """Sum of |terms| of the reward expression (condition-aware tolerance)."""
    v = views(st)
    vel_r = 0.05 * torch.linalg.norm(torch.cat((v["lin"], v["ang"]), 1), dim=1)
    pos_r = 0.05 * torch.linalg.norm(default - v["dof_pos"], dim=1)
    height = (0.325 - v["bez_pos"][:, 2]).abs()
    ball_fwd = 0.1 * torch.linalg.norm(v["ball_vel"][:, 0:2], dim=1)
    vel_fwd = 0.05 * torch.linalg.norm(v["lin"][:, 0:2], dim=1)
    return vel_r + pos_r + height + ball_fwd + vel_fwd
