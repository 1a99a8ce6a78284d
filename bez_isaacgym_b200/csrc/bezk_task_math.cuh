// Per-env math of the BezKick / walk / orient task step (device functions; arithmetic order follows the reference op by op).
// Used by the tile kernel (bezk_task.cu).
#pragma once
#include "bezk_common.cuh"
#include "bezk_internal.h"
#include <math.h>

namespace bezk {

constexpr int DOF_ROW = 36;          // floats per env in dof_state
// Task variants (tasks/kick_env.py, tasks/walk_env.py, tasks/orient_env.py share one skeleton): BezKick has two actors per env
// (robot + ball -> 26 root floats) and a 54-wide observation; walk / orient have the robot only (13) and 52 columns.
__host__ __device__ constexpr int root_row(int task) { return task == BEZK_TASK_KICK ? 26 : 13; }
__host__ __device__ constexpr int obs_row(int task) { return task == BEZK_TASK_KICK ? 54 : 52; }

// ------------------------------------------------------------------------------------------------
// per-env math (device functions; arithmetic order follows the reference op by op)
// ------------------------------------------------------------------------------------------------

// compute_imu, kick_env.py:918-930, with quaternion_to_matrix (:857-885) applied to the xyzw
// quaternion as if it were real-first: (r,i,j,k) = (x,y,z,w).
template <bool F>
__device__ __forceinline__ void imu_term(const float (&q)[4], const float (&v)[3], const float (&w)[3],
                                         const float (&prev)[3], const BezkTaskCfg& c, float (&out)[6], Mth<F>& m) {
    float a[3];
    a[0] = m.div(v[0] - prev[0], c.dt) - 0.0f;
    a[1] = m.div(v[1] - prev[1], c.dt) - 0.0f;
    a[2] = m.div(v[2] - prev[2], c.dt) - (-1.0f);        // gravity_vec = (0,0,-1), :217
    const float r = q[0], i = q[1], j = q[2], k = q[3];
    const float two_s = m.div(2.0f, ((r * r + i * i) + j * j) + k * k);
    const float m00 = 1.0f - two_s * (j * j + k * k), m01 = two_s * (i * j - k * r), m02 = two_s * (i * k + j * r);
    const float m10 = two_s * (i * j + k * r), m11 = 1.0f - two_s * (i * i + k * k), m12 = two_s * (j * k - i * r);
    const float m20 = two_s * (i * k - j * r), m21 = two_s * (j * k + i * r), m22 = 1.0f - two_s * (i * i + j * j);
    const float t0 = (m00 * a[0] + m01 * a[1]) + m02 * a[2];
    const float t1 = (m10 * a[0] + m11 * a[1]) + m12 * a[2];
    const float t2 = (m20 * a[0] + m21 * a[1]) + m22 * a[2];
    out[0] = clamp_nan(t0, -c.imu_max_lin_acc, c.imu_max_lin_acc);
    out[1] = clamp_nan(t1, -c.imu_max_lin_acc, c.imu_max_lin_acc);
    out[2] = clamp_nan(t2, -c.imu_max_lin_acc, c.imu_max_lin_acc);
    out[3] = clamp_nan(w[0], -c.imu_max_ang_vel, c.imu_max_ang_vel);
    out[4] = clamp_nan(w[1], -c.imu_max_ang_vel, c.imu_max_ang_vel);
    out[5] = clamp_nan(w[2], -c.imu_max_ang_vel, c.imu_max_ang_vel);
}

// torch.remainder(x, 2 pi) (python-style, Tensor.__mod__) for x = atan2f_z(..) in [-pi, pi]: |x| < 2 pi, so fmod(x, 2 pi) is x
// itself and the remainder is x (+ 2 pi when x < 0); identical bits to fmodf + sign fix-up, without the fmodf loop.  NaN and
// -0.0 pass through unchanged, as they do there.
__device__ __forceinline__ float wrap_2pi(float x) {
    return (x < 0.0f) ? x + 6.283185307179586f : x;
}

// compute_off_orn, kick_env.py:941-960 (+ yaw of get_euler_xyz)
template <bool F>
__device__ __forceinline__ void off_orn_term(float px, float py, const float (&q)[4], float gx, float gy, float (&out)[2], Mth<F>& m) {
    const float dx = gx - px, dy = gy - py;
    const float nrm = m.sqr(dx * dx + dy * dy);
    const float ux = m.div(dx, nrm), uy = m.div(dy, nrm);
    const float x = q[0], y = q[1], z = q[2], w = q[3];
    const float siny = 2.0f * (w * z + x * y);
    const float cosy = ((w * w + x * x) - y * y) - z * z;
    const float yaw = wrap_2pi(atan2f_z(siny, cosy));
    float hx, hy;
    sincosf(yaw, &hy, &hx);                              // one shared range reduction; same values as sinf / cosf
    const float c = hx * ux + hy * uy;
    const float cz = ux * hy - uy * hx;                  // only non-zero component of the 3-D cross
    out[0] = m.sqr((0.0f + 0.0f) + cz * cz);             // linalg.norm of (0, 0, cz)
    out[1] = -c;
}

// compute_feet_sensors_no_cleats, kick_env.py:987-1038: returns the 4 bits of one foot and filters f.
__device__ __forceinline__ void foot_bits(float (&f)[3], float (&bits)[4]) {
#pragma unroll
    for (int k = 0; k < 3; ++k) f[k] = (fabsf(f[k]) > 0.01f) ? f[k] : 0.0f;     // NaN -> 0 as in torch.where
    const bool x0 = (f[0] == 0.0f), y0 = (f[1] == 0.0f);
    // (x!=0,y!=0)->case 1, (x!=0,y==0)->3, (x==0,y!=0)->9, (x==0,y==0)->11   (SURVEY a9 truth table)
    float b0 = 1.0f, b1 = x0 ? 1.0f : -1.0f, b2 = y0 ? 1.0f : -1.0f, b3 = (x0 && y0) ? 1.0f : -1.0f;
    if (f[2] < 1.0f) { b0 = b1 = b2 = b3 = -1.0f; }
    bits[0] = b0; bits[1] = b1; bits[2] = b2; bits[3] = b3;
}

// yaw of isaacgym.torch_utils.get_euler_xyz (mod 2 pi)
__device__ __forceinline__ float yaw_mod_2pi(const float (&q)[4]) {
    const float x = q[0], y = q[1], z = q[2], w = q[3];
    const float siny = 2.0f * (w * z + x * y);
    const float cosy = ((w * w + x * x) - y * y) - z * z;
    return wrap_2pi(atan2f_z(siny, cosy));
}

// compute_off_angle, orient_env.py:720-733: (cos, sin) of goal_angle - normalize_angle(yaw)
__device__ __forceinline__ float angle_to_goal(const float (&q)[4], float goal_angle) {
    const float yaw = yaw_mod_2pi(q);
    float sy, cy;
    sincosf(yaw, &sy, &cy);
    const float na = atan2f_z(sy, cy);                     // normalize_angle
    return goal_angle - na;
}

// quantities walk_env.py:849-876 / orient_env.py:875-897 share
struct WalkTerms { float up_proj, vel6, vel_lin, vel_ang, pos; };
template <bool F>
__device__ __forceinline__ WalkTerms walk_terms(const float (&q)[4], const float (&v)[3], const float (&w)[3], float pos_sq, Mth<F>& m) {
    WalkTerms t;
    // get_basis_vector(q, (0,0,1))[2] = quat_rotate z component: a + b + c
    const float qx = q[0], qy = q[1], qz = q[2], qw = q[3];
    const float a_z = 1.0f * (2.0f * (qw * qw) - 1.0f);
    const float b_z = ((qx * 0.0f - qy * 0.0f) * qw) * 2.0f;            // cross(q_vec, v).z * q_w * 2
    const float dot = (qx * 0.0f + qy * 0.0f) + qz * 1.0f;              // bmm(q_vec, v)
    const float c_z = (qz * dot) * 2.0f;
    t.up_proj = (a_z + b_z) + c_z;
    float s3 = v[0] * v[0]; s3 += v[1] * v[1]; s3 += v[2] * v[2];
    float a3 = w[0] * w[0]; a3 += w[1] * w[1]; a3 += w[2] * w[2];
    float s6 = s3; s6 += w[0] * w[0]; s6 += w[1] * w[1]; s6 += w[2] * w[2];
    t.vel6 = m.sqr(s6); t.vel_lin = m.sqr(s3); t.vel_ang = m.sqr(a3);
    t.pos = m.sqr(pos_sq);
    return t;
}

// The outcome class (bezk_internal.h) of an env no termination rule fired for.  Written only by the OC instantiations of the reward
// functions below.
constexpr int OUTCOME_NONE = -1;

// shared tail of the two reward functions: fall, win state, (task rule), horizon.  OC: also the outcome class into *oc_out.  TM:
// tm_out holds the caller's 4 shaping terms; they become 0 when a rule fired, and tm_out[4] gets the override (0 otherwise).
template <bool OC = false, bool TM = false>
__device__ __forceinline__ void walk_tail(const WalkTerms& t, bool close, float rew, bool out_rule, float out_value, const BezkTaskCfg& c,
                                          int64_t progress, int64_t reset_cur, float* rew_out, int64_t* reset_out,
                                          int* oc_out = nullptr, float* tm_out = nullptr) {
    int64_t reset = reset_cur;
    int oc = OUTCOME_NONE;
    if (t.up_proj < 0.7f) { reset = 1; rew = -100.0f; if constexpr (OC || TM) oc = WALK_FELL; }       // fall
    float state = close ? 1.0f : 0.0f;
    if (t.pos < 0.15f) state += 1.0f;
    if (t.vel_ang < 0.1f) state += 1.0f;
    if (t.vel_lin < 0.1f) state += 1.0f;
    if (state == 4.0f) {                                                                          // win state
        reset = 1;
        rew = 1.0f * (1000.0f - 1000.0f * ((float)progress / (float)c.max_episode_length));
        if constexpr (OC || TM) oc = WALK_REACHED;
    }
    if (out_rule) { reset = 1; rew = out_value; if constexpr (OC || TM) oc = WALK_OUT; }               // out of bound
    if (progress >= (int64_t)c.max_episode_length) { reset = 1; rew = 0.0f; if constexpr (OC || TM) oc = WALK_TIMEOUT; }   // horizon
    *rew_out = rew;
    *reset_out = reset;
    if constexpr (OC) *oc_out = oc;
    if constexpr (TM) {
        const bool fired = oc != OUTCOME_NONE;
#pragma unroll
        for (int k = 0; k < 4; ++k) tm_out[k] = fired ? 0.0f : tm_out[k];
        tm_out[4] = fired ? rew : 0.0f;
    }
}

// compute_bez_reward of tasks/walk_env.py:827-997 (debug prints and dead terms dropped).  TM: also the WALK_TERMS reward terms
// into tm_out (goal velocity, uprightness, body velocity, posture, termination).
template <bool F, bool OC = false, bool TM = false>
__device__ __forceinline__ void reward_walk(const float (&bez)[3], const float (&q)[4], const float (&v)[3], const float (&w)[3],
                                            float pos_sq, const float (&goal)[2], const BezkTaskCfg& c, int64_t progress,
                                            int64_t reset_cur, float* rew_out, int64_t* reset_out, Mth<F>& m,
                                            int* oc_out = nullptr, float* tm_out = nullptr) {
    const float dx = goal[0] - bez[0], dy = goal[1] - bez[1];
    const float n_goal = m.sqr(dx * dx + dy * dy);
    const float ux = m.div(dx, n_goal), uy = m.div(dy, n_goal);
    const float vel_fwd = ux * v[0] + uy * v[1];
    const WalkTerms t = walk_terms(q, v, w, pos_sq, m);
    const float dist_h = fabsf(1.0f - t.up_proj);
    const float vel_s = t.vel6 * 0.05f, pos_s = t.pos * 0.05f;
    const float height_vel_pos = -((vel_s + pos_s) + dist_h);
    const float vel_height = (vel_fwd * 10.0f - (dist_h + 5.0f * pos_s)) * 1.0f;
    const bool close = n_goal < 0.05f;
    const float rew = close ? height_vel_pos : vel_height;
    // out of bound: angle between (goal - (0,0)) and (goal - bez_xy)   (walk_env.py:966-989; bez_init_state is zeroed in place)
    const float ix = goal[0] - 0.0f, iy = goal[1] - 0.0f;
    const float n_i = m.sqr(ix * ix + iy * iy);
    const float ang_now = atan2f_z(uy, ux);
    const float ang_init = atan2f_z(m.div(iy, n_i), m.div(ix, n_i));
    const bool out = fabsf(ang_init - ang_now) > 1.5708f;
    if constexpr (TM) {
        tm_out[0] = close ? 0.0f : vel_fwd * 10.0f;
        tm_out[1] = -dist_h;
        tm_out[2] = close ? -vel_s : 0.0f;
        tm_out[3] = close ? -pos_s : -(5.0f * pos_s);
    }
    walk_tail<OC, TM>(t, close, rew, out, -100.0f, c, progress, reset_cur, rew_out, reset_out, oc_out, tm_out);
}

// compute_bez_reward of tasks/orient_env.py:845-1014.  TM: also the WALK_TERMS reward terms into tm_out (heading, uprightness,
// body velocity, posture, termination).
template <bool F, bool OC = false, bool TM = false>
__device__ __forceinline__ void reward_orient(const float (&bez)[3], const float (&q)[4], const float (&v)[3], const float (&w)[3],
                                              float pos_sq, float goal_angle, const BezkTaskCfg& c, int64_t progress,
                                              int64_t reset_cur, float* rew_out, int64_t* reset_out, Mth<F>& m,
                                              int* oc_out = nullptr, float* tm_out = nullptr) {
    const float ang = angle_to_goal(q, goal_angle);
    const WalkTerms t = walk_terms(q, v, w, pos_sq, m);
    const float dist_h = fabsf(1.0f - t.up_proj);
    const float vel_s = t.vel6 * 0.05f, pos_s = t.pos * 0.05f;
    const float height_vel_pos = -((vel_s + pos_s) + dist_h);
    const float vel_height = (fabsf(ang) * -0.5f - (dist_h + 0.05f * pos_s)) * 1.0f;
    const bool close = ang < 0.05f;                       // the SIGNED angle, as the reference compares it
    const float rew = close ? height_vel_pos : vel_height;
    const float tx = bez[0] - c.bez_init_xy[0], ty = bez[1] - c.bez_init_xy[1];
    const bool out = m.sqr(tx * tx + ty * ty) > 0.3f;
    if constexpr (TM) {
        tm_out[0] = close ? 0.0f : fabsf(ang) * -0.5f;
        tm_out[1] = -dist_h;
        tm_out[2] = close ? -vel_s : 0.0f;
        tm_out[3] = close ? -pos_s : -(0.05f * pos_s);
    }
    walk_tail<OC, TM>(t, close, rew, out, -5.0f, c, progress, reset_cur, rew_out, reset_out, oc_out, tm_out);
}

struct RewardIn {
    float bez[3];          // torso root position
    float ball_xy[2];
    float ball_vxy[2];
    float goal[2];
    float ball_init[2];
    float v[3], w[3];      // IMU-link linear / angular velocity
    float pos_sq;          // sum_j (default_j - dof_pos_j)^2, sequential
};

// compute_bez_reward, kick_env.py:1224-1395 (SURVEY A.1).  `progress` is the post-increment value.  OC: also the outcome class
// into *oc_out.  TM: also the KICK_TERMS reward terms into tm_out (ball velocity, approach, height, body velocity, posture,
// termination).
template <bool F, bool OC = false, bool TM = false>
__device__ __forceinline__ void reward_term(const RewardIn& s, const BezkTaskCfg& c, int64_t progress,
                                            int64_t reset_cur, float* rew_out, int64_t* reset_out, Mth<F>& m,
                                            int* oc_out = nullptr, float* tm_out = nullptr) {
    const float dbx = s.ball_xy[0] - s.bez[0], dby = s.ball_xy[1] - s.bez[1];
    const float nbb = m.sqr(dbx * dbx + dby * dby);
    const float vel_fwd = m.div(dbx, nbb) * s.v[0] + m.div(dby, nbb) * s.v[1];

    const float dgx = s.goal[0] - s.ball_xy[0], dgy = s.goal[1] - s.ball_xy[1];
    const float n_goal = m.sqr(dgx * dgx + dgy * dgy);
    const float ugx = m.div(dgx, n_goal), ugy = m.div(dgy, n_goal);
    const float ball_fwd = ugx * s.ball_vxy[0] + ugy * s.ball_vxy[1];

    const float dix = s.goal[0] - s.ball_init[0], diy = s.goal[1] - s.ball_init[1];
    const float n_init = m.sqr(dix * dix + diy * diy);
    const float ang_now = atan2f_z(ugy, ugx);
    const float ang_init = atan2f_z(m.div(diy, n_init), m.div(dix, n_init));
    const float angle_diff = fabsf(ang_init - ang_now);

    float vs = s.v[0] * s.v[0];
    vs += s.v[1] * s.v[1]; vs += s.v[2] * s.v[2];
    vs += s.w[0] * s.w[0]; vs += s.w[1] * s.w[1]; vs += s.w[2] * s.w[2];
    const float vel_r = m.sqr(vs) * 0.05f;
    const float pos_r = m.sqr(s.pos_sq) * 0.05f;
    const float height = fabsf(0.325f - s.bez[2]) * 1.0f;
    const float kx = s.ball_xy[0] - s.ball_init[0], ky = s.ball_xy[1] - s.ball_init[1];
    const float kicked = m.sqr(kx * kx + ky * ky);

    const float far_r = ball_fwd * 0.1f - (height + (vel_r + pos_r));
    const float near_r = ball_fwd * 0.1f + (vel_fwd * 0.05f - height);
    float rew = (kicked > 0.3f) ? far_r : near_r;
    int64_t reset = reset_cur;
    int oc = OUTCOME_NONE;

    if (s.bez[2] < 0.275f) { reset = 1; rew = -1.0f; if constexpr (OC || TM) oc = KICK_FELL; }                 // rule 1
    const float tx = s.bez[0] - c.bez_init_xy[0], ty = s.bez[1] - c.bez_init_xy[1];
    if (m.sqr(tx * tx + ty * ty) > 0.5f) { reset = 1; rew = -1.0f; if constexpr (OC || TM) oc = KICK_STRAYED; }   // rule 2
    if (angle_diff > 1.5708f) { reset = 1; rew = -1.0f; if constexpr (OC || TM) oc = KICK_WIDE; }                // rule 3
    if (n_goal < 0.05f) {                                                                                // rule 4
        reset = 1;
        rew = 1.0f * (100.0f - 100.0f * ((float)progress / (float)c.max_episode_length));
        if constexpr (OC || TM) oc = KICK_SCORED;
    }
    if (progress >= (int64_t)c.max_episode_length) { reset = 1; rew = 0.0f; if constexpr (OC || TM) oc = KICK_TIMEOUT; }   // rule 5
    *rew_out = rew;
    *reset_out = reset;
    if constexpr (OC) *oc_out = oc;
    if constexpr (TM) {
        const bool fired = oc != OUTCOME_NONE, far = kicked > 0.3f;
        tm_out[0] = fired ? 0.0f : ball_fwd * 0.1f;
        tm_out[1] = (fired || far) ? 0.0f : vel_fwd * 0.05f;
        tm_out[2] = fired ? 0.0f : -height;
        tm_out[3] = (fired || !far) ? 0.0f : -vel_r;
        tm_out[4] = (fired || !far) ? 0.0f : -pos_r;
        tm_out[5] = fired ? rew : 0.0f;
    }
}

// rl_games play_steps reward path (a2c_common.py play_steps + tr_helpers.DefaultRewardsShaper; cfg/train/bez_kickPPO.yaml:53-56):
//   shaped = (rew + shift) * scale;  shaped += gamma * values * time_outs.float()   (value_bootstrap)
// and the uint8 copy of the reset mask that becomes the experience buffer's `dones` slot of the next step.
__device__ __forceinline__ void rollout_epilogue(const TaskArgs& a, int64_t e, float rew, int64_t reset, int64_t timeout, float value) {
    if (a.shaped_rew) {
        float s = (rew + a.shp_shift) * a.shp_scale;
        if (a.shp_bootstrap) s = s + (a.shp_gamma * value) * (float)timeout;
        a.shaped_rew[e] = s;
    }
    if (a.dones_u8) a.dones_u8[e] = (uint8_t)(reset != 0);
}

// rl_games play_steps episode bookkeeping of one env (a2c_common.py; `rewards` is the unshaped rew_buf, `dones` the reset mask):
//   current_rewards += rewards; current_lengths += 1; ...; current_* = current_* * not_dones
// r / l are what a done env hands to the game_rewards / game_lengths meters; the carried values are written back as MULTIPLIES by
// (1 - done), so a NaN / inf return stays NaN in the accumulator after the env is done, as in rl_games.
__device__ __forceinline__ void episode_step(float ret, float len, float rew, int64_t reset, float& r, float& l, float& ret_out,
                                             float& len_out) {
    r = ret + rew;
    l = len + 1.0f;
    const float not_done = 1.0f - (reset != 0 ? 1.0f : 0.0f);
    ret_out = r * not_done;
    len_out = l * not_done;
}

// reset_idx DOF part, kick_env.py:786-791
__device__ __forceinline__ void reset_dof_row(const float (&u)[36], const BezkTaskCfg& c, float (&row)[36]) {
#pragma unroll
    for (int j = 0; j < 18; ++j) {
        const float off = c.reset_pos_span * u[j] + c.reset_pos_lo;
        row[2 * j] = tensor_clamp(c.default_dof_pos[j] + off, c.dof_lower[j], c.dof_upper[j]);
        row[2 * j + 1] = c.reset_vel_span * u[18 + j] + c.reset_vel_lo;
    }
}


}  // namespace bezk
