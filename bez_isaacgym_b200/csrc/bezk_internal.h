// Internal launcher interface shared by the .cu translation units of libbezk.so (not installed).
#pragma once
#include "../../include/bezk.h"
#include <cuda_runtime.h>
#include <stdint.h>

namespace bezk {
struct TaskArgs {
    float* dof_state;            // (n*18, 2)
    const float* rigid_body;     // (n*NB, 13)
    float* root_states;          // (n*2, 13)
    float* net_contact;          // (n*NB, 3)
    float* prev_lin_vel;         // (n, 3) or nullptr (aliasing mode)
    float* goal;                 // (n, 2); rewritten on reset by the walk / orient tasks
    const float* goal_angle;     // (n,)  orient task only
    const float* goal_uniforms;  // (2,)  per-step goal draw or nullptr (Philox)
    const float* ball_init;      // (n, 2)  BezKick only
    const float* initial_root;   // (n*2, 13)
    const float* uniforms;       // (n, 36) or nullptr (Philox)
    uint64_t seed, step;
    int64_t env_base;            // global id of env 0 of this launch (Philox key) -- non-zero when a step is launched in chunks
    float* dof_state_wb;         // where reset rows are written back (nullptr: dof_state itself)
    float* root_states_wb;       // likewise for the root rows (nullptr: root_states itself)
    const int64_t* reset_in;
    int64_t* reset_out;
    const int64_t* progress_in;
    int64_t* progress_out;
    int64_t* timeout_buf;
    int64_t* randomize_buf;
    float* obs;
    float* obs_clipped;
    float* rew;
    // rl_games play_steps reward path folded into the reward epilogue (bezk_post_physics_rollout); all optional
    const float* values;         // (n,) un-normalised critic values of this step (value bootstrap)
    int values_stride;           // floats between two envs' values (0 = 1; the host pipeline's records carry them in their last float)
    float* shaped_rew;           // (n,) out: (rew + shift) * scale [+ gamma * value * timeout]
    uint8_t* dones_u8;           // (n,) out: reset mask as uint8 (the experience buffer's `dones` slot of the NEXT step)
    float shp_scale, shp_shift, shp_gamma;
    int shp_bootstrap;
    // Layout of the two sparse inputs, in floats.  0 = Isaac Gym's AoS layout derived from BezkTaskCfg (env stride
    // num_bodies * 13 resp. * 3; the IMU-link slice at (imu_body * 13 + 3), the foot rows at body * 3); the host pipeline's
    // compact staging buffers (bezk_stage_sparse_rows) set them explicitly.
    int rb_stride, rb_off;       // rigid_body: floats per env, offset of the 10-float IMU-link slice
    int cf_stride, cf_l_off, cf_r_off;   // net_contact: floats per env, offsets of the left / right foot (first cleat) rows
    int64_t n;
    int use_tma;      // all dense bases 16 B aligned
    int rb_vec2;      // IMU-link slice of every env is 8 B aligned
    int rb_win;       // slice only 4 B aligned, but the 16-byte aligned window around it is readable: 3-4 vector loads
    int cf_vec2;      // both foot force rows of every env are 8 B aligned
    int smart_granule;  // per-lane 64 B / 128 B fill choice for the sparse gathers (env BEZK_SMART_GRANULE=0 disables)
    // set_l2_policy: 1 = the step accesses the carried state (obs rows, reset / progress / timeout, rew, prev_lin_vel, goal,
    // ball_init / goal_angle) with evict_last and the dense tiles and sparse gathers with evict_first (task_tile_l2_kernel)
    int l2_resident;
};
// Episode accumulators of the fused step (bezk_post_physics_rollout_ep; rl_games play_steps' current_rewards / current_lengths and
// the done-env sums its game_rewards / game_lengths meters are fed with).  A separate kernel parameter of task_tile_ep_kernel /
// task_tile_ep_l2_kernel, not TaskArgs fields: a longer TaskArgs would move the BezkTaskCfg parameter of every other kernel.
struct EpArgs {
    float* ret;                  // (n,) carried episode return: ret + rew, times (1 - done)
    float* len;                  // (n,) carried episode length: len + 1, times (1 - done)
    double* partials;            // (3, W), W = ceil(n / 32): per warp of 32 envs [count of done envs, sum of their return, sum of their length]
    int64_t w;                   // W
};
// Eval-mode observation normaliser of the fused step (bezk_post_physics_rollout_ep_norm; rl_games RunningMeanStd.forward with
// frozen statistics, what PpoPlayerContinuous feeds the policy).  A separate kernel parameter of task_tile_obsnorm_kernel /
// task_tile_obsnorm_l2_kernel, for the reason EpArgs is one.
struct NormArgs {
    const double* mean;          // (obs_row,) running_mean, read every launch
    const double* var;           // (obs_row,) running_var
    float* out;                  // (n, obs_row) clamp((x - mean) / sqrt(var + eps), -5, 5), x = the row step() returns
    float eps;
};
// fills l2_resident (bezk_task.cu): after fill_alignment, before the launch; ep: the armed episode accumulators or nullptr
void set_l2_policy(int task, uint32_t cfg_flags, TaskArgs& a, const EpArgs* ep = nullptr);
// demote [ptr, ptr + bytes) to the normal L2 eviction priority (the 128-byte lines entirely inside the range)
cudaError_t launch_l2_release(const void* ptr, uint64_t bytes, cudaStream_t st);
struct PpoArgs {
    const float *actions, *mu, *logstd, *old_mu, *old_sigma, *values, *old_values, *returns, *old_neglogp, *advantages;
    float *grad_mu, *grad_values, *neglogp_out;
    double* partials;
    double* stats;             // (8,) loss terms; with fused_finalize CTA 0 writes them after a grid barrier
    float* grad_logstd;
    int fused_finalize;
    int64_t m;
    int64_t slab_rows, slab_stride;   // rollout-side tensors as slabs of time-major storage (slab_rows == m: contiguous)
    int slabs;
    int use_tma;
};
// the tile kernel for (task, parts): kick takes parts 1..7, walk / orient 2, 3, 4 or 7; ep (the episode accumulators,
// task_tile_ep_kernel / task_tile_ep_l2_kernel) only with parts = 7; nm (the observation normaliser, task_tile_obsnorm_kernel /
// task_tile_obsnorm_l2_kernel) only together with ep.  cudaErrorInvalidValue for any other combination.
cudaError_t launch_task(int task, int parts, const TaskArgs& a, const BezkTaskCfg& cfg, const EpArgs* ep, cudaStream_t st,
                        const NormArgs* nm = nullptr);
// folds `steps` x (3, ceil(n / 32)) partials of launch_task's episode accumulators into the two AverageMeters (bezk_rollout.cu)
cudaError_t launch_episode_meter_update(const double* partials, int steps, int64_t n, int64_t games_to_track, float* mean2,
                                        int64_t* size2, cudaStream_t st);
// folds the same partials into rl_games BasePlayer.run's game tally [games_played, sum_rewards, sum_steps, steps_folded]
// up to games_num games (bezk_rollout.cu)
cudaError_t launch_player_tally_update(const double* partials, int steps, int64_t n, int64_t games_num, double* tally,
                                       double* per_step, cudaStream_t st);
cudaError_t launch_goal_uniforms(uint64_t seed, uint64_t step, float* out2, cudaStream_t st);
void fill_alignment(TaskArgs& a, const BezkTaskCfg& cfg);
cudaError_t stage_feet_gather(const float*, const BezkTaskCfg&, float*, int64_t, int64_t, cudaStream_t);
cudaError_t stage_imu_rows(const float*, const BezkTaskCfg&, float*, int64_t, int64_t, cudaStream_t);
cudaError_t stage_sparse_rows(const float*, const float*, const BezkTaskCfg&, float*, float*, int64_t, int64_t, cudaStream_t);
// layout of the host pipeline's packed per-env record (bezk_host_pack.cu), in floats
struct PackLayout { int stride, l_off, r_off, feet_w, root_off, root_n; };
PackLayout pack_layout(int task, const BezkTaskCfg& cfg);
int host_pack_config(int threads, int spin_us, int pin);
int64_t host_pack_begin(int task, const float*, const float*, const float*, const float*, const float*, const BezkTaskCfg&, float*, int64_t,
                        int64_t);
cudaError_t launch_unpack_root(int task, const float* records, PackLayout L, float* root_states, int64_t n, cudaStream_t st);
int host_pack_wait(int64_t ticket);
cudaError_t launch_pre_physics(const float*, float*, float*, const BezkTaskCfg&, int64_t, cudaStream_t);
cudaError_t launch_reset_idx(const int64_t*, int64_t, const float*, uint64_t, uint64_t, float*, float*, const float*, int64_t*,
                             int64_t*, const BezkTaskCfg&, int64_t, int, float*, const float*, int64_t, cudaStream_t);
cudaError_t launch_philox_uniforms(uint64_t, uint64_t, float*, int64_t, cudaStream_t);
cudaError_t launch_gae(const float*, const float*, const void*, const float*, const void*, int, double, double, float*, float*,
                       int, int64_t, cudaStream_t);
int64_t rms_scratch_doubles(int c);
cudaError_t launch_rms_moments(const float*, const double*, double*, double*, int64_t, int, int64_t, int64_t, cudaStream_t,
                               const double* snap_var = nullptr, const double* snap_count = nullptr);
cudaError_t launch_rms_merge_normalize(const float*, const double*, double*, double*, double*, float, float*, int64_t, int, int64_t,
                                       int64_t, cudaStream_t);
cudaError_t launch_rms_merge(const double*, const double*, double*, double*, double*, int, cudaStream_t);
cudaError_t launch_rms_moments_batched(const float*, const double*, double*, double*, int64_t, int, int64_t, int64_t, int64_t, int,
                                       cudaStream_t);
cudaError_t launch_rms_merge_sequence(const double*, const int32_t*, int, const double*, double*, double*, double*, double*, int,
                                      cudaStream_t);
cudaError_t launch_rms_normalize(const float*, const double*, const double*, float, int, float*, int64_t, int, int64_t, int64_t,
                                 cudaStream_t);
cudaError_t launch_rms_normalize_batched(const float*, const double*, const double*, float, float*, int64_t, int, int64_t, int64_t,
                                         int64_t, int64_t, int, cudaStream_t);
cudaError_t launch_adv_moments(const float*, const float*, double*, double*, int64_t, cudaStream_t);
cudaError_t launch_adv_normalize(const float*, const float*, const double*, float*, int, int64_t, cudaStream_t);
cudaError_t launch_swap_flatten(const void*, void*, int, int64_t, int64_t, int64_t, int, cudaStream_t);
cudaError_t launch_policy_head(const float*, const float*, const float*, const double*, const double*, float, const float*, uint64_t,
                               uint64_t, float*, float*, float*, float*, float*, const BezkTaskCfg*, float*, float*, int64_t, int64_t,
                               cudaStream_t);
cudaError_t launch_normal_noise(uint64_t, uint64_t, float*, int64_t, int64_t, cudaStream_t);
cudaError_t launch_dr_noise(const float*, const float*, const float*, uint64_t, uint64_t, const BezkNoiseCfg&, float*, float*, float,
                            int64_t, cudaStream_t);
cudaError_t launch_dr_fill(uint64_t, uint64_t, int, float*, int64_t, cudaStream_t);
cudaError_t launch_selftest_fastmath(uint64_t, uint64_t, unsigned long long*, cudaStream_t);
int64_t ppo_scratch_doubles();
cudaError_t launch_ppo_loss(const PpoArgs&, const BezkPpoCfg&, double*, float*, cudaStream_t);
cudaError_t launch_quat_rotate(const float*, const float*, float*, int, int64_t, cudaStream_t);
cudaError_t launch_scale_transform(const float*, const float*, const float*, float*, int, int64_t, int, cudaStream_t);
bool fused_stats_eligible(int64_t m, int c);
cudaError_t launch_rms_train_forward(const float*, double*, double*, double*, float, float*, double*, int64_t, int, int64_t, int64_t,
                                     cudaStream_t);
cudaError_t launch_adv_fused(const float*, const float*, float*, double*, int, int64_t, cudaStream_t);
}  // namespace bezk
