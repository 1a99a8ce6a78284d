/*
 * bezk.h -- C ABI of libbezk.so, the B200 (sm_100a) BezKick hot path.
 *
 * Drop-in boundary for the per-step tensor path of utra-robosoccer/Bez_IsaacGym's BezKick task and
 * the rl_games rollout math it feeds.  Every entry point takes caller-owned DEVICE pointers
 * (Isaac-Gym-layout state tensors are borrowed, never reallocated), sizes and a CUDA stream
 * (passed as void* so this header needs no CUDA include); nothing allocates, nothing synchronises,
 * everything is stream-ordered.  Return value: 0 on success, otherwise a cudaError_t value or one
 * of the BEZK_E_* codes below; bezk_last_error() gives the message.  There is no CPU fallback.
 *
 * "ref:" cites the reference interface each entry replaces, relative to
 * /root/reference/bez_isaacgym/ (rl_games is third-party, un-vendored: cited by upstream file).
 */
#ifndef BEZK_H_
#define BEZK_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define BEZK_VERSION 130          /* 0.1.3: host packer, packed / staged entries with the reward epilogue, planned RunningMeanStd updates */
#define BEZK_NUM_DOF 18
#define BEZK_NUM_OBS 54

#define BEZK_E_BADARG   10001     /* null pointer / negative size / bad enum */
#define BEZK_E_ALIGN    10002     /* pointer not aligned as documented */
#define BEZK_E_CONFIG   10003     /* BezkTaskCfg inconsistent (body index >= num_bodies ...) */

/* flags for BezkTaskCfg.flags */
#define BEZK_F_CLEATS              1u  /* 8 cleat bodies instead of 2 foot bodies (tasks/kick_env.py:188-196) */
#define BEZK_F_WRITE_CONTACT_FILTER 2u /* write the |f|<=0.01 -> 0 noise filter back into net_contact
                                          (the reference does, tasks/kick_env.py:987-990) */
#define BEZK_F_RESET_ROOT_STATES   4u  /* masked reset also copies initial_root_states rows into
                                          root_states (what the simulator's indexed setters do,
                                          tasks/kick_env.py:831-837); off when a real simulator owns that */
#define BEZK_F_OBS_STREAMED        8u  /* obs / obs_clipped point at a different buffer every step (e.g. the next slot of a
                                          rollout buffer): their rows are not kept resident in L2 (bezk_l2_release) */

/* Constants of one BezKick instance.  Passed BY VALUE into the kernels (constant bank).
 * ref: tasks/kick_env.py:46-238 (constructor), cfg/task/bez_kick.yaml. */
typedef struct BezkTaskCfg {
    int32_t num_bodies;          /* rigid bodies per env incl. the ball: 22 (30 with cleats) */
    int32_t imu_body;            /* 1   tasks/kick_env.py:175-177 */
    int32_t left_foot_body;      /* 12  (:193)   with cleats: first of 4 cleat bodies, 13 (:188) */
    int32_t right_foot_body;     /* 20  (:195)   with cleats: first of 4 cleat bodies, 25 (:190) */
    int32_t max_episode_length;  /* 900 = int(15 / 0.01667 + 0.5)  (:126-127) */
    uint32_t flags;              /* BEZK_F_* */
    float dt;                    /* 0.01667 */
    float imu_max_lin_acc;       /* 19.62   (:100) */
    float imu_max_ang_vel;       /* 8.7266  (:99)  */
    float clip_obs;              /* +inf by default (tasks/base/vec_task.py:97) */
    float clip_actions;          /* 3.9 (cfg/task/bez_kick.yaml:11) */
    float bez_init_xy[2];        /* (:160) */
    /* torch_rand_float(lo, hi) = (hi - lo) * U + lo with (hi - lo) formed in double on the host:
     * positions U(-0.15, 0.15) (:786) -> lo = -0.15f, span = (float)0.3; velocities U(-0.1, 0.1) (:787). */
    float reset_pos_lo, reset_pos_span;
    float reset_vel_lo, reset_vel_span;
    float default_dof_pos[BEZK_NUM_DOF];   /* readyJointAngles in DOF order (:204-209) */
    float dof_lower[BEZK_NUM_DOF];         /* (:393-406) */
    float dof_upper[BEZK_NUM_DOF];
} BezkTaskCfg;

int  bezk_version(void);
const char* bezk_last_error(void);
/* Device-wide hint (cudaLimitMaxL2FetchGranularity: 32, 64 or 128 bytes) for the current device.  The task
 * kernels gather 12..40-byte slices out of 264..1144-byte Isaac Gym rows, so a 32-byte L2 fetch
 * granularity avoids dragging unused neighbouring sectors out of HBM.  Returns the value in effect
 * through *effective (may be NULL). */
int bezk_set_l2_fetch_granularity(int32_t bytes, int32_t* effective);

/* ---------------------------------------------------------------- task side ------------------ */

/* K0.  ref: tasks/base/vec_task.py:317 + tasks/kick_env.py:410-419 (KickEnv.pre_physics_step).
 * actions (n,18) f32 -> targets (n,18) f32 = clamp(zero_head(clip(actions)) + default, lower, upper).
 * actions_out (n,18) receives the stored `self.actions` (clipped, head zeroed); may be NULL. */
int bezk_pre_physics(const float* actions, float* actions_out, float* targets,
                     const BezkTaskCfg* cfg, int64_t n, void* stream);

/* K1 (function level).  ref: KickEnv.compute_observations tasks/kick_env.py:749-777 and the jit
 * functions :857-1069,1398-1417.  Reads dof_state (n*18,2), rigid_body (n*NB,13), root_states
 * (n*2,13), net_contact (n*NB,3; filtered in place when BEZK_F_WRITE_CONTACT_FILTER), goal (n,2),
 * ball_init (n,2).  prev_lin_vel (n,3) f32 is read then overwritten with the current IMU-link
 * linear velocity; NULL selects the reference's steady-state aliasing (prev == current velocity,
 * tasks/kick_env.py:930).  obs (n,54).  obs_clipped (n,54) or NULL (written only if non-NULL). */
int bezk_compute_observations(const float* dof_state, const float* rigid_body, const float* root_states,
                              float* net_contact, float* prev_lin_vel, const float* goal,
                              const float* ball_init, const BezkTaskCfg* cfg, float* obs,
                              float* obs_clipped, int64_t n, void* stream);

/* K2 (function level).  ref: compute_bez_reward tasks/kick_env.py:1198-1395 (+ wrapper :724-747).
 * reset_in / progress (n,) i64 are the function's reset_buf / progress_buf arguments;
 * rew (n,) f32 and reset_out (n,) i64 its two results (reset_out may alias reset_in). */
int bezk_compute_reward(const float* dof_state, const float* rigid_body, const float* root_states,
                        const float* goal, const float* ball_init, const int64_t* reset_in,
                        const int64_t* progress, const BezkTaskCfg* cfg, float* rew,
                        int64_t* reset_out, int64_t n, void* stream);

/* K3 (function level).  ref: KickEnv.reset_idx tasks/kick_env.py:779-850 for an explicit,
 * ascending id list env_ids (k,) i64.  uniforms (k,36) f32 in [0,1): cols 0:18 feed the position
 * draw, 18:36 the velocity draw (the two torch_rand_float calls, :786-787); NULL -> Philox4x32-10
 * keyed (seed, step, env id).  Writes dof_state rows, root_states rows (flag), progress=0, reset=0. */
int bezk_reset_idx(const int64_t* env_ids, int64_t k, const float* uniforms, uint64_t seed,
                   uint64_t step, float* dof_state, float* root_states,
                   const float* initial_root_states, int64_t* progress, int64_t* reset,
                   const BezkTaskCfg* cfg, int64_t n, void* stream);

/* Fused post-physics step = everything VecTask.step does after gym.simulate, in ONE launch.
 * ref: tasks/base/vec_task.py:331-332 (timeout from pre-increment progress) +
 * KickEnv.post_physics_step tasks/kick_env.py:426-438 (progress++, reset of envs whose reset_buf
 * was set by the previous step, observations, reward/termination).
 *   reset_buf    (n,) i64 in: previous step's mask; out: this step's mask
 *   progress_buf (n,) i64 in/out;  timeout_buf (n,) i64 out;  randomize_buf (n,) i64 in/out or NULL
 *   uniforms     (n,36) f32 per-ENV reset draws or NULL -> Philox keyed (seed, step, env id)
 *   parts        bitmask: 1 = bookkeeping+masked reset, 2 = observations, 4 = reward/termination.
 *                7 = whole step.  3 and 4 give the north-star's two kernels (obs kernel, reward kernel). */
#define BEZK_PART_BOOKKEEP 1
#define BEZK_PART_OBS      2
#define BEZK_PART_REWARD   4
int bezk_post_physics(float* dof_state, const float* rigid_body, float* root_states,
                      float* net_contact, float* prev_lin_vel, const float* goal,
                      const float* ball_init, const float* initial_root_states,
                      const float* uniforms, uint64_t seed, uint64_t step,
                      int64_t* reset_buf, int64_t* progress_buf, int64_t* timeout_buf,
                      int64_t* randomize_buf, const BezkTaskCfg* cfg, float* obs, float* obs_clipped,
                      float* rew, int parts, int64_t n, void* stream);

/* One CHUNK of a step: the same kernel over envs [env_base, env_base + n) of a larger task, every pointer already offset to
 * the chunk's first env.  env_base keeps the Philox reset noise keyed by the GLOBAL env id, so a step launched in chunks
 * (the host pipeline overlaps the DMA of chunk c+1 with the kernel of chunk c) gives the results of one launch.
 * dof_state_wb / root_states_wb: where the rows of the envs that reset are written back (NULL: dof_state / root_states
 * themselves) -- with a staged copy of the dense tensors on the device, the reset rows still go to the simulator's own
 * (pinned host) tensors. */
int bezk_post_physics_chunk(float* dof_state, const float* rigid_body, float* root_states,
                            float* net_contact, float* prev_lin_vel, const float* goal,
                            const float* ball_init, const float* initial_root_states,
                            const float* uniforms, uint64_t seed, uint64_t step,
                            int64_t* reset_buf, int64_t* progress_buf, int64_t* timeout_buf,
                            int64_t* randomize_buf, const BezkTaskCfg* cfg, float* obs, float* obs_clipped,
                            float* rew, int parts, int64_t n, int64_t env_base, float* dof_state_wb,
                            float* root_states_wb, void* stream);

/* Parameters of the reward epilogue (documented at bezk_post_physics_rollout below). */
typedef struct BezkRolloutCfg {
    float scale_value;        /* 0.01 */
    float shift_value;        /* 0    */
    float gamma;              /* (float)0.99 -- torch multiplies the fp32 tensor by the Python double cast to fp32 */
    int32_t value_bootstrap;  /* 1 */
} BezkRolloutCfg;

/* Host pipeline (sim_device=cpu / use_gpu_pipeline: False; ref: tasks/base/vec_task.py:51-98 device selection): the simulator
 * tensors live in PINNED HOST memory.  bezk_stage_sparse_rows pulls the few bytes per env the step needs out of the two sparse
 * AoS tensors with strided copy-engine transfers (cudaMemcpy2DAsync) into compact DEVICE staging, for envs [env0, env0 + n):
 *   imu_stage  (N,10) f32  <- rigid_body row (env, imu_body), floats 3..12 (quaternion, linear and angular velocity)
 *   feet_stage (N,8)  f32  <- [left foot xyz, pad, right foot xyz, pad]        (cleats: (N,24) = [4 left cleat rows, 4 right])
 * (pointers are the tensor BASES; env0 selects the chunk).  bezk_post_physics_staged is bezk_post_physics_chunk reading those
 * staging buffers in place of rigid_body / net_contact, for any task (arguments as bezk_post_physics_task); everything else
 * (dense dof_state / root_states staging copies, the write-back pointers into the simulator's own host tensors, env_base) as
 * documented there.  BEZK_F_WRITE_CONTACT_FILTER must be
 * clear (the filtered forces would land in the staging buffer, not in the simulator's tensor). */
int bezk_stage_sparse_rows(const float* rigid_body_host, const float* net_contact_host, const BezkTaskCfg* cfg,
                           float* imu_stage, float* feet_stage, int64_t env0, int64_t n, void* stream);
/* As bezk_stage_sparse_rows, but only the IMU slices go through the copy engine (on copy_stream); the foot rows are fetched by a
 * small gather kernel on gather_stream that reads the pinned host tensor directly, concurrently with the engine's transfers. */
int bezk_stage_sparse_rows_split(const float* rigid_body_host, const float* net_contact_host, const BezkTaskCfg* cfg,
                                 float* imu_stage, float* feet_stage, int64_t env0, int64_t n, void* copy_stream,
                                 void* gather_stream);
/* The same gather done by HOST worker threads instead of the copy engine, into ONE compact record per env in PINNED host memory.
 * A job covers envs [env0, env0 + n) of the simulator tensors (passed as tensor BASES) and writes to dst, the job's OWN
 * destination (16-byte aligned): n records of bezk_host_pack_record_floats floats each,
 *   [ IMU-link q, v, w (10) | left foot row (3; cleats 12) | right foot row | root subset | zero pad to a multiple of 4 floats ]
 * root subset = the only floats of root_states the step reads: robot position xyz, and for BezKick the ball's xy position and xy
 * velocity (7 floats of 26; walk / orient: 3 of 13).  BezKick: 24 floats = 96 B per env instead of 1512 B of AoS rows.
 * With dof_state_host != NULL the job ALSO copies the chunk's dense dof_state rows: dst = [ n x 36 dof floats | n records ], so
 * that ONE cudaMemcpyAsync moves everything the chunk's kernel reads (every additional H2D call costs the link ~40 us under
 * bidirectional load, profiles/r02_host_pack.md).
 * The copy engine serving the H2D direction is row-rate-bound on strided pulls (1.4 ns per row); the simulator's host cores, idle
 * between simulate() calls, gather the rows of chunk c + 1 while the engine streams chunk c (ref: tasks/base/vec_task.py:51-98,
 * the sim_device=cpu pipeline).
 * bezk_host_pack_begin is asynchronous: it returns a ticket > 0 (0 for n == 0, -BEZK_E_* on a bad argument);
 * bezk_host_pack_wait(ticket) returns once the job's output is written (the caller's thread packs too while it waits).
 * Jobs are served in issue order; any thread may issue and wait (the pool is process-wide).  bezk_host_pack_config sizes the pool (threads = 0:
 * hardware threads - 1, at most 16; the pool only grows), sets how long an idle worker polls for the next job before it blocks
 * (spin_us, default 100; < 0 keeps the current value: between steps the workers sleep and leave the cores to the simulator -- raise
 * it to the step period on hosts where a futex wake is expensive) and whether workers are pinned one per CPU (pin, honoured before the first worker starts; < 0 keeps it); it
 * returns the worker count (-BEZK_E_BADARG on a bad thread count).  No CUDA call is made by these four.
 * bezk_post_physics_packed is bezk_post_physics_chunk for a chunk whose records are on the DEVICE (pointer already offset to the
 * chunk's first record, like every other argument): it scatters the root subset into the chunk's rows of root_states (a device
 * image of the simulator tensor; its other columns are never read) and runs the step reading the IMU slice and the foot rows
 * straight out of the records.  BEZK_F_WRITE_CONTACT_FILTER must be clear.
 * Both bezk_post_physics_staged and bezk_post_physics_packed take the reward-epilogue arguments of bezk_post_physics_rollout
 * (rollout, values, shaped_rewards, dones_u8: DEVICE pointers offset to the chunk; all NULL = off; parts must be 7).  With the
 * packed records the critic values can travel in the record's last (pad) float instead: pass values_host (N,) to
 * bezk_host_pack_begin and values = NULL to bezk_post_physics_packed. */
int bezk_host_pack_config(int32_t threads, int32_t spin_us, int32_t pin);
int bezk_host_pack_record_floats(int task, const BezkTaskCfg* cfg);
int64_t bezk_host_pack_begin(int task, const float* rigid_body_host, const float* net_contact_host,
                             const float* root_states_host, const float* dof_state_host, const float* values_host,
                             const BezkTaskCfg* cfg, float* dst, int64_t env0, int64_t n);
int bezk_host_pack_wait(int64_t ticket);
int bezk_post_physics_packed(int task, float* dof_state, const float* records, float* root_states, float* prev_lin_vel,
                             float* goal, const float* goal_angle, const float* ball_init,
                             const float* initial_root_states, const float* uniforms, const float* goal_uniforms,
                             uint64_t seed, uint64_t step, int64_t* reset_buf, int64_t* progress_buf,
                             int64_t* timeout_buf, int64_t* randomize_buf, const BezkTaskCfg* cfg, float* obs,
                             float* obs_clipped, float* rew, int parts, int64_t n, int64_t env_base,
                             float* dof_state_wb, float* root_states_wb, const BezkRolloutCfg* rollout,
                             const float* values, float* shaped_rewards, uint8_t* dones_u8, void* stream);
int bezk_post_physics_staged(int task, float* dof_state, const float* imu_stage, float* root_states, float* feet_stage,
                             float* prev_lin_vel, float* goal, const float* goal_angle, const float* ball_init,
                             const float* initial_root_states, const float* uniforms, const float* goal_uniforms,
                             uint64_t seed, uint64_t step, int64_t* reset_buf, int64_t* progress_buf,
                             int64_t* timeout_buf, int64_t* randomize_buf, const BezkTaskCfg* cfg, float* obs,
                             float* obs_clipped, float* rew, int parts, int64_t n, int64_t env_base,
                             float* dof_state_wb, float* root_states_wb, const BezkRolloutCfg* rollout,
                             const float* values, float* shaped_rewards, uint8_t* dones_u8, void* stream);

/* The dense (n,36) uniforms the Philox path of bezk_post_physics / bezk_reset_idx consumes for
 * (seed, step): lets a checker feed the identical draws to the reference's reset_idx. */
int bezk_philox_uniforms(uint64_t seed, uint64_t step, float* out, int64_t n, void* stream);

/* ---------------------------------------------------------------- rollout / learner math ----- */

/* K6.  ref: rl_games/common/a2c_common.py A2CBase.discount_values (+ mb_returns = advs + values).
 * rewards, values (T,n) f32; dones (T,n): dones_kind 0 = uint8, 1 = float32; last_values (n,) f32;
 * last_dones (n,) same kind.  Out: advs, returns (T,n) f32.  time-major, env fastest.
 * gamma, tau are the Python doubles of the config; the kernel uses (float)gamma and (float)(gamma*tau)
 * exactly as torch's scalar promotion does. */
int bezk_gae(const float* rewards, const float* values, const void* dones, const float* last_values,
             const void* last_dones, int dones_kind, double gamma, double tau, float* advs,
             float* returns, int32_t horizon, int64_t n, void* stream);

/* K4a.  Pivoted batch moments for RunningMeanStd (ref: rl_games/algos_torch/running_mean_std.py
 * forward, training branch).  x (m,c) f32 row-major.  pivot = running_mean (c,) f64 (may be NULL -> 0).
 * acc (1+2c,) f64 is OVERWRITTEN with [m, sum_j(x-p), sum_j(x-p)^2]: additive across ranks, so a
 * single SUM all-reduce of acc merges shards exactly.  partials: scratch f64, >= bezk_rms_scratch_doubles(c). */
int64_t bezk_rms_scratch_doubles(int32_t c);
int bezk_rms_moments(const float* x, const double* pivot, double* acc, double* partials,
                     int64_t m, int32_t c, void* stream);
/* K4b.  Merge acc (from bezk_rms_moments, possibly all-reduced) into running_mean/var (c,) f64 and
 * count () f64 with the reference's parallel-variance update (unbiased batch variance). */
int bezk_rms_merge(const double* acc, const double* pivot, double* running_mean, double* running_var,
                   double* count, int32_t c, void* stream);
/* bezk_rms_moments_slabs for n_batches equally spaced minibatches in one pair of launches: batch b is the slab view based at
 * x + b * batch_stride * c (batch_stride in rows), acc (n_batches, 1+2c) receives one row per batch; same pivot, same scratch. */
int bezk_rms_moments_slabs_batched(const float* x, int64_t slab_rows, int64_t slab_stride, int64_t batch_stride,
                                   const double* pivot, double* acc, double* partials, int64_t m, int32_t c,
                                   int32_t n_batches, void* stream);
/* K4c.  A SEQUENCE of those merges in one launch: acc (n_batches, 1+2c) holds the moments of n_batches distinct batches (all taken
 * with the same pivot, possibly all-reduced over ranks in ONE collective); update u = 0 .. n_updates-1 merges batch order[u]
 * (device int32, values in [0, n_batches)) exactly as bezk_rms_merge would; seq (n_updates, 2, c) f64 receives [mean, var] AFTER
 * update u -- the statistics the u-th train-mode forward normalises with (pass seq + u*2*c and seq + (u*2+1)*c to
 * bezk_rms_normalize[_slabs]) -- and running_mean / running_var / count the final state.  rl_games updates the obs normaliser with
 * the SAME minibatches in every mini-epoch (calc_gradients: `obs = self.running_mean_std(obs)` in train mode) and the moments do
 * not depend on the policy: n_batches moment passes per epoch instead of mini_epochs * n_batches, same statistics. */
int bezk_rms_merge_sequence(const double* acc, int32_t n_batches, const int32_t* order, int32_t n_updates,
                            const double* pivot, double* running_mean, double* running_var, double* count, double* seq,
                            int32_t c, void* stream);
/* K5.  y = clamp((x - mean.float()) / sqrt(var.float() + eps), -5, 5)   (unnorm = 0)
 *      y = sqrt(var.float() + eps) * clamp(x, -5, 5) + mean.float()      (unnorm = 1)
 * x, y (m,c) f32 (y may alias x). */
int bezk_rms_normalize(const float* x, const double* running_mean, const double* running_var,
                       float eps, int unnorm, float* y, int64_t m, int32_t c, void* stream);

/* K4 + K5 in ONE call: the train-mode forward of RunningMeanStd (update the running statistics with the batch, then normalise
 * the batch with the UPDATED statistics), what rl_games runs on every minibatch of every mini-epoch (SURVEY a19).  x may be a
 * slab view (slab_rows / slab_stride as in bezk_rms_moments_slabs; slab_rows <= 0: contiguous); y (m,c) contiguous.
 * Three launches (moments with pivot = running_mean read in place; fold + snapshot of the old statistics; merge + normalise in
 * one kernel), against five for the separate entries; c == 1 (value normaliser) runs as ONE cooperative kernel.
 * Single-GPU form; env-sharded ranks use the two halves below with one SUM all-reduce of acc_ext[0 : 1 + 2c] in between.
 * partials: scratch f64, >= bezk_rms_scratch_doubles(c). */
int bezk_rms_train_forward(const float* x, int64_t slab_rows, int64_t slab_stride, double* running_mean,
                           double* running_var, double* count, float eps, float* y, double* partials,
                           int64_t m, int32_t c, void* stream);
/* acc_ext (2 + 4c,) f64 = [m, sum_j(x - mean), sum_j(x - mean)^2, old mean(c), old var(c), old count]: the pivoted batch moments
 * (pivot = running_mean, identical on every rank) followed by a snapshot of the running statistics. */
int bezk_rms_moments_ext(const float* x, int64_t slab_rows, int64_t slab_stride, const double* running_mean,
                         const double* running_var, const double* count, double* acc_ext, double* partials,
                         int64_t m, int32_t c, void* stream);
/* Merge acc_ext (its first 1 + 2c entries possibly all-reduced) into running_mean / running_var / count and write
 * y = clamp((x - mean') / sqrt(var' + eps), -5, 5) with the updated statistics, one launch. */
int bezk_rms_merge_normalize(const float* x, int64_t slab_rows, int64_t slab_stride, const double* acc_ext,
                             double* running_mean, double* running_var, double* count, float eps, float* y,
                             int64_t m, int32_t c, void* stream);

/* K7 in ONE call (single GPU): adv_out = returns - values, normalised to zero mean / unit (unbiased) std when normalize != 0.
 * One cooperative kernel up to ~6 M samples, the bezk_adv_moments / bezk_adv_normalize chain beyond.
 * partials: scratch f64, >= bezk_rms_scratch_doubles(1). */
int bezk_adv_normalize_fused(const float* returns, const float* values, float* adv_out, double* partials,
                             int normalize, int64_t m, void* stream);

/* K7.  ref: a2c_common.py prepare_dataset: adv = returns - values, then (adv - mean)/(std + 1e-8)
 * with the unbiased std.  Step 1 accumulates acc (3,) f64 = [m, sum adv, sum adv^2] (additive across
 * ranks); step 2 normalises.  returns, values (m,) f32; adv_out (m,) f32. */
int bezk_adv_moments(const float* returns, const float* values, double* acc, double* partials,
                     int64_t m, void* stream);
int bezk_adv_normalize(const float* returns, const float* values, const double* acc, float* adv_out,
                       int normalize, int64_t m, void* stream);

/* K8.  ref: rl_games/algos_torch/a2c_continuous.py calc_gradients loss block +
 * common_losses.actor_loss/critic_loss + bound_loss + torch_ext.policy_kl + models neglogp.
 * Forward AND backward of
 *   loss = mean(a) + 0.5*critic_coef*mean(c) - entropy_coef*mean(ent) + bounds_loss_coef*mean(b)
 * in one pass.  Inputs (m = minibatch): actions, mu, old_mu, old_sigma (m,18); logstd (18,)
 * (fixed_sigma); values, old_values, returns, old_neglogp, advantages (m,).
 * Outputs: stats (8,) f64 = [loss, a_loss, c_loss, entropy, b_loss, kl, clip_frac, 0] (means);
 * grad_mu (m,18), grad_values (m,), grad_logstd (18,) f32 = d loss / d(.)  (any may be NULL to
 * skip); neglogp_out (m,) or NULL.  partials: scratch f64 >= bezk_ppo_scratch_doubles(). */
typedef struct BezkPpoCfg {
    float e_clip;            /* 0.2 */
    float critic_coef;       /* 2   */
    float entropy_coef;      /* 0   */
    float bounds_loss_coef;  /* 0.001 */
    float soft_bound;        /* 1.1 */
    int32_t clip_value;      /* 1 */
    int32_t bound_form;      /* 0 = rl_games 1.1.3 as recalled, 1 = later "outside" form */
} BezkPpoCfg;
int64_t bezk_ppo_scratch_doubles(void);
int bezk_ppo_loss(const float* actions, const float* mu, const float* logstd, const float* old_mu,
                  const float* old_sigma, const float* values, const float* old_values,
                  const float* returns, const float* old_neglogp, const float* advantages,
                  const BezkPpoCfg* cfg, double* stats, float* grad_mu, float* grad_values,
                  float* grad_logstd, float* neglogp_out, double* partials, int64_t m, void* stream);

/* ---------------------------------------------------------------- sibling tasks (SURVEY 8f row 3) ----- */

/* WalkEnv / OrientEnv (ref: tasks/walk_env.py, tasks/orient_env.py) share BezKick's skeleton: same K0, same IMU / feet /
 * bookkeeping / masked reset; they differ in
 *   - layout: ONE actor per env (root_states (n,13)), 21 bodies (29 with cleats), observation (n,52) =
 *     [dof_pos 18, dof_vel 18, imu 6, heading 2, feet 8]   (walk_env.py:1032-1050)
 *   - heading: walk = compute_off_orn vs goal (n,2) (walk_env.py:379-386); orient = compute_off_angle =
 *     (cos, sin)(goal_angle - normalize_angle(yaw)) with goal_angle (n,) (orient_env.py:719-733)
 *   - reward / termination: walk_env.py:827-997, orient_env.py:845-1014 (up-vector projection, win state, out of bound)
 *   - reset: additionally goal[env] = (U(-2,2), U(-2,2)); the reference assigns the FIRST draw of the reset batch to every
 *     env resetting in that step (walk_env.py:570-574 `self.goal[env_ids, 0] = goal_x[0]`), so the draw is per STEP:
 *     goal_uniforms (2,) f32 in [0,1) or NULL -> Philox keyed (seed, step) alone.
 * goal (n,2) is read AND written.  goal_angle is read by BEZK_TASK_ORIENT only.  Everything else as bezk_post_physics
 * (task = BEZK_TASK_KICK forwards to it; ball_init is then required and goal is not written). */
#define BEZK_TASK_KICK   0
#define BEZK_TASK_WALK   1
#define BEZK_TASK_ORIENT 2
int bezk_post_physics_task(int task, float* dof_state, const float* rigid_body, float* root_states,
                           float* net_contact, float* prev_lin_vel, float* goal, const float* goal_angle,
                           const float* ball_init, const float* initial_root_states,
                           const float* uniforms, const float* goal_uniforms, uint64_t seed, uint64_t step,
                           int64_t* reset_buf, int64_t* progress_buf, int64_t* timeout_buf,
                           int64_t* randomize_buf, const BezkTaskCfg* cfg, float* obs, float* obs_clipped,
                           float* rew, int parts, int64_t n, void* stream);
/* The fused step with rl_games' per-step reward path in its epilogue (SURVEY 8 a16).
 * ref: rl_games/common/a2c_common.py play_steps -- `shaped_rewards = self.rewards_shaper(rewards)`;
 * `shaped_rewards += self.gamma * res_dict['values'] * self.cast_obs(infos['time_outs']).unsqueeze(1).float()` (value_bootstrap);
 * `self.dones = dones.byte()` -- with rl_games/common/tr_helpers.py DefaultRewardsShaper ((r + shift_value) * scale_value),
 * configured by cfg/train/bez_kickPPO.yaml:53-56 (value_bootstrap: True, reward_shaper.scale_value: 0.01).
 *   values         (n,) f32 in : un-normalised critic values of this step (what bezk_policy_head wrote); needed when
 *                                value_bootstrap != 0
 *   shaped_rewards (n,) f32 out: (rew + shift) * scale + (gamma * value) * (float)timeout   -> experience slot mb_rewards[t]
 *   dones_u8       (n,) u8  out: reset_buf != 0                                             -> experience slot dones[t+1]
 * Each of shaped_rewards / dones_u8 may be NULL.  rew / reset_buf / timeout_buf are written as by bezk_post_physics_task.
 * Always the whole step (parts = 7).  env_base: global id of env 0 of this launch (Philox key of the reset noise; 0 for an
 * un-sharded task) -- env-sharded ranks pass their shard offset so that the noise does not depend on the sharding. */
int bezk_post_physics_rollout(int task, float* dof_state, const float* rigid_body, float* root_states,
                              float* net_contact, float* prev_lin_vel, float* goal, const float* goal_angle,
                              const float* ball_init, const float* initial_root_states,
                              const float* uniforms, const float* goal_uniforms, uint64_t seed, uint64_t step,
                              int64_t* reset_buf, int64_t* progress_buf, int64_t* timeout_buf,
                              int64_t* randomize_buf, const BezkTaskCfg* cfg, float* obs, float* obs_clipped,
                              float* rew, const BezkRolloutCfg* rollout, const float* values,
                              float* shaped_rewards, uint8_t* dones_u8, int64_t env_base, int64_t n, void* stream);
/* bezk_post_physics_rollout with rl_games' episode bookkeeping in the same epilogue (a2c_common.py play_steps:
 * `current_rewards += rewards; current_lengths += 1; ...; current_rewards = current_rewards * not_dones`, likewise the lengths;
 * `rewards` is the unshaped rew, `dones` the reset mask this step writes).  ep_return, ep_length, ep_partials: all NULL (then this
 * is bezk_post_physics_rollout) or all non-NULL, DEVICE memory:
 *   ep_return, ep_length (n,) f32 in/out: the episode return / length so far; every env adds this step's rew / 1 and writes the
 *                                         sum back multiplied by (1 - done) -- a NaN return stays NaN, as in rl_games
 *   ep_partials (3, W) f64 out, W = ceil(n / 32): per group of 32 envs (env / 32) the count of envs done in this step, the sum of
 *                                         their returns and the sum of their lengths (this step's rew / 1 included).  Every slot is
 *                                         written each step; the sums have a fixed order (the same bits every run).
 * Accumulators armed: obs, rew, reset, progress, time-outs, reset rows, shaped rewards and dones_u8 are the same bytes as without
 * them. */
int bezk_post_physics_rollout_ep(int task, float* dof_state, const float* rigid_body, float* root_states,
                                 float* net_contact, float* prev_lin_vel, float* goal, const float* goal_angle,
                                 const float* ball_init, const float* initial_root_states,
                                 const float* uniforms, const float* goal_uniforms, uint64_t seed, uint64_t step,
                                 int64_t* reset_buf, int64_t* progress_buf, int64_t* timeout_buf,
                                 int64_t* randomize_buf, const BezkTaskCfg* cfg, float* obs, float* obs_clipped,
                                 float* rew, const BezkRolloutCfg* rollout, const float* values,
                                 float* shaped_rewards, uint8_t* dones_u8, int64_t env_base, int64_t n,
                                 float* ep_return, float* ep_length, double* ep_partials, void* stream);
/* rl_games' game_rewards / game_lengths meters (torch_ext.AverageMeter(1, games_to_track)) updated from `steps` consecutive
 * ep_partials of bezk_post_physics_rollout_ep over n envs (partials: (steps, 3, ceil(n / 32)) f64), step by step in order:
 *   new_mean = sum / count (fp64, rounded to fp32); size = min(count, games_to_track);
 *   old_size = min(games_to_track - size, current_size); current_size = old_size + size;
 *   mean = (mean * old_size + new_mean * size) / current_size          (fp32; a step with count 0 changes nothing)
 * mean2 (2,) f32 and size2 (2,) i64, DEVICE memory, in/out: [returns meter, lengths meter].  No host synchronisation (graph
 * capturable); steps == 0 or n == 0 is a no-op. */
int bezk_episode_meter_update(const double* partials, int steps, int64_t n, int64_t games_to_track, float* mean2,
                              int64_t* size2, void* stream);
/* bezk_post_physics_rollout_ep that also writes the observation row through rl_games' RunningMeanStd.forward in eval mode (what
 * the player feeds its policy), from the tile the step already holds:
 *   obs_norm (n, obs_width) f32 out = clamp((x - (float)obs_mean) / sqrtf((float)obs_var + obs_eps), -5, 5)
 * x = the row the step returns (obs_clipped when given, obs otherwise); IEEE division and square root, NaN propagating -- the same
 * bits as bezk_rms_normalize(x, obs_mean, obs_var, obs_eps, 0, ...).  obs_mean / obs_var (obs_width,) f64, DEVICE memory, are
 * read by every launch.  obs_mean, obs_var, obs_norm: all NULL (then this is bezk_post_physics_rollout_ep) or all non-NULL; armed,
 * the episode accumulators must be armed too (BEZK_E_BADARG otherwise), obs_norm 16-byte and obs_mean / obs_var 8-byte aligned
 * (BEZK_E_ALIGN).  Every other output is the same bytes as without obs_norm. */
int bezk_post_physics_rollout_ep_norm(int task, float* dof_state, const float* rigid_body, float* root_states,
                                      float* net_contact, float* prev_lin_vel, float* goal, const float* goal_angle,
                                      const float* ball_init, const float* initial_root_states,
                                      const float* uniforms, const float* goal_uniforms, uint64_t seed, uint64_t step,
                                      int64_t* reset_buf, int64_t* progress_buf, int64_t* timeout_buf,
                                      int64_t* randomize_buf, const BezkTaskCfg* cfg, float* obs, float* obs_clipped,
                                      float* rew, const BezkRolloutCfg* rollout, const float* values,
                                      float* shaped_rewards, uint8_t* dones_u8, int64_t env_base, int64_t n,
                                      float* ep_return, float* ep_length, double* ep_partials,
                                      const double* obs_mean, const double* obs_var, float obs_eps, float* obs_norm, void* stream);
/* rl_games BasePlayer.run's game tally fed by `steps` consecutive ep_partials over n envs (partials: (steps, 3, ceil(n / 32)) f64),
 * step by step in order: games_played += count; sum_rewards += return sum; sum_steps += length sum, where a step that starts with
 * games_played >= games_num adds nothing (the step that reaches games_num is added whole).  Each step's sums over its slots have
 * a fixed order, so the result does not depend on how the steps are split over calls.
 *   tally (4,) f64 in/out, DEVICE memory: [games_played, sum_rewards, sum_steps, steps_folded]
 *   per_step (steps, 3) f64 out or NULL: each folded step's [count, return sum, length sum], zeros for the steps not folded.
 * No host synchronisation (graph capturable); steps == 0 or n == 0 is a no-op; games_num <= 0 is BEZK_E_BADARG. */
int bezk_player_tally_update(const double* partials, int steps, int64_t n, int64_t games_num, double* tally, double* per_step,
                             void* stream);
/* bezk_reset_idx for any task: root rows are 13 floats for walk / orient, and their goal (n,2) rows are redrawn.
 * env_base: global id of local env 0 (Philox key = env_base + env id), as in bezk_post_physics_rollout. */
int bezk_reset_idx_task(int task, const int64_t* env_ids, int64_t k, const float* uniforms, const float* goal_uniforms,
                        uint64_t seed, uint64_t step, float* dof_state, float* root_states,
                        const float* initial_root_states, float* goal, int64_t* progress, int64_t* reset,
                        const BezkTaskCfg* cfg, int64_t env_base, int64_t n, void* stream);
/* The (2,) uniforms the Philox path uses for the goal draw of (seed, step). */
int bezk_goal_uniforms(uint64_t seed, uint64_t step, float* out2, void* stream);
/* The device-memory post-physics entries (bezk_post_physics, _task, _rollout, bezk_compute_*) access the state an env carries
 * from step to step -- obs (and obs_clipped) rows, reset / progress / time-out flags, rew, prev_lin_vel, goal, ball_init /
 * goal_angle -- with the L2 eviction priority evict_last when that state of all n envs fits 75 % of the device's L2 and one
 * step streams more than L2 holds (per-instruction cache hints; no set-aside, no access-policy window, no device limit).  Lines so marked keep that priority while
 * they stay in L2, also after the buffers are freed: an owner that drops those buffers calls bezk_l2_release on each of them
 * first (stream-ordered; the 128-byte lines entirely inside [ptr, ptr + bytes) go back to the normal priority).  Env
 * BEZK_L2_RESIDENT=0 (read once per process) turns the hints off. */
int bezk_l2_release(const void* ptr, uint64_t bytes, void* stream);

/* ---------------------------------------------------------------- rollout storage (SURVEY 8f rows 1-2) ----- */

/* Slab addressing.  rl_games keeps the rollout time-major -- ExperienceBuffer tensors are (T, N, ...) -- and builds its
 * dataset with swap_and_flatten01 (a full read + write of every tensor) before slicing minibatches of consecutive
 * env-major rows (rl_games/common/a2c_common.py play_steps / prepare_dataset, rl_games/common/datasets.py PPODataset).
 * Minibatch i of E = minibatch_size / T envs is the sample set {(t, e): e0 <= e < e0 + E}.  The *_slabs entries read that
 * set IN PLACE: the m = T * E batch rows are T slabs of `slab_rows` (= E) consecutive source rows, slab s starting at row
 * s * slab_stride (= N) of the base pointer (= tensor + e0 * row width).  Batch row r = t * E + (e - e0): the same samples
 * as rl_games' minibatch, ordered time-major inside the batch (a permutation that no mean / moment / gradient depends on).
 * slab_rows == m (or <= 0) means "contiguous", which makes every *_slabs entry equal to its plain counterpart. */
int bezk_rms_moments_slabs(const float* x, int64_t slab_rows, int64_t slab_stride, const double* pivot, double* acc,
                           double* partials, int64_t m, int32_t c, void* stream);
/* y (m,c) is written contiguously in batch-row order (the network input). */
int bezk_rms_normalize_slabs(const float* x, int64_t slab_rows, int64_t slab_stride, const double* running_mean,
                             const double* running_var, float eps, int unnorm, float* y, int64_t m, int32_t c,
                             void* stream);
/* n_batches minibatches in ONE launch, each with its own statistics (the planned updates of bezk_rms_merge_sequence: the
 * minibatches of one mini-epoch): batch b is the slab view based at x + b * batch_stride * c (batch_stride in rows: E for the
 * consecutive env blocks of time-major storage), normalised with mean + b * stat_stride / var + b * stat_stride (doubles; 2c for
 * consecutive updates of a seq buffer) into y + b * m * c. */
int bezk_rms_normalize_slabs_batched(const float* x, int64_t slab_rows, int64_t slab_stride, int64_t batch_stride,
                                     const double* mean, const double* var, int64_t stat_stride, float eps, float* y,
                                     int64_t m, int32_t c, int32_t n_batches, void* stream);
/* bezk_ppo_loss with the ROLLOUT-side tensors (actions, old_mu, old_sigma (.,18); old_values, returns, old_neglogp,
 * advantages (.,)) read as slabs; mu, values (network outputs) and all outputs are contiguous batch rows. */
int bezk_ppo_loss_slabs(const float* actions, const float* mu, const float* logstd, const float* old_mu,
                        const float* old_sigma, const float* values, const float* old_values,
                        const float* returns, const float* old_neglogp, const float* advantages,
                        int64_t slab_rows, int64_t slab_stride,
                        const BezkPpoCfg* cfg, double* stats, float* grad_mu, float* grad_values,
                        float* grad_logstd, float* neglogp_out, double* partials, int64_t m, void* stream);

/* ref: rl_games/common/a2c_common.py swap_and_flatten01 (+ the minibatch slice of PPODataset):
 *   dst[(e - env0) * horizon + t][:] = src[t * num_envs + e][:]   for env0 <= e < env0 + envs, 0 <= t < horizon
 * rows of row_bytes bytes (any dtype; 216 for observations, 72 for actions, 4 for scalars, 1 for uint8 dones).
 * One tiled shared-memory transposition; src and dst must not overlap. */
int bezk_swap_and_flatten01(const void* src, void* dst, int32_t horizon, int64_t num_envs, int64_t env0, int64_t envs,
                            int32_t row_bytes, void* stream);

/* Policy-head epilogue: what rl_games does between the MLP and env.step in play_steps, in one kernel.
 * ref: rl_games/algos_torch/models.py ModelA2CContinuousLogStd.forward (is_train=False: sigma = exp(logstd),
 * Normal(mu, sigma).sample(), neglogp), a2c_common.py get_action_values (values = value_mean_std(values, unnorm=True)),
 * play_steps (experience_buffer.update_data of actions / neglogpacs / values / mus / sigmas), preprocess_actions
 * (clamp(-1,1) + rescale_actions; cf. the in-tree fork utils/players.py:11-15,63-64) and KickEnv.pre_physics_step.
 *   mu (n,18), logstd (18,), value_norm (n,) [NULL: no values]; value_mean/value_var: () f64 running stats [NULL: copy]
 *   noise (n,18) N(0,1) draws, or NULL -> Philox4x32-10 keyed (seed, step, env_base + row) + Box-Muller; env_base = global id of
 *   row 0 (the rank's shard offset under env-sharded multi-GPU training, 0 otherwise), so that ranks sharing one seed
 *   draw DIFFERENT noise and the union over ranks equals the un-sharded draw
 *   outputs (each may be NULL): actions (n,18), neglogp (n,), values (n,), mus (n,18), sigmas (n,18),
 *   env_actions (n,18) = clamp(actions,-1,1); targets (n,18) = K0(env_actions) when task_cfg != NULL. */
int bezk_policy_head(const float* mu, const float* logstd, const float* value_norm, const double* value_mean,
                     const double* value_var, float value_eps, const float* noise, uint64_t seed, uint64_t step,
                     float* actions, float* neglogp, float* values, float* mus, float* sigmas,
                     const BezkTaskCfg* task_cfg, float* env_actions, float* targets, int64_t env_base, int64_t n,
                     void* stream);
/* The (n,18) normals the Philox path of bezk_policy_head uses for (seed, step) and rows env_base .. env_base + n - 1: lets a
 * checker feed identical noise to the reference's Normal.sample() replacement. */
int bezk_normal_noise(uint64_t seed, uint64_t step, float* out, int64_t env_base, int64_t n, void* stream);

/* ---------------------------------------------------------------- domain-randomisation noise (SURVEY 8f row 4) ----- */

/* The observation / action noise lambdas VecTask.apply_randomizations builds (ref: tasks/base/vec_task.py:562-618; applied
 * to the actions at :314-315 and to obs_buf at :338-339; parameters cfg/task/bez_kick.yaml:153-162):
 *     y = op(x, (corr * a_corr + b_corr) + w * a + b)
 * gaussian: a = var, b = mu, a_corr = var_corr, b_corr = mu_corr, w ~ N(0,1)
 * uniform:  a = hi - lo, b = lo, a_corr = hi_corr - lo_corr, b_corr = lo_corr, w ~ U[0,1)   (corr stays N(0,1), as upstream)
 * (schedule scaling is applied by the host when it fills the struct, as the reference does when it builds the lambda).
 * x, y (total,) f32 (y may alias x); corr (total,) f32 persistent N(0,1) draw or NULL (= zeros); white (total,) f32 draws or
 * NULL -> Philox4x32-10 keyed (seed, step, element / 4). */
typedef struct BezkNoiseCfg {
    int32_t distribution;   /* 0 = gaussian, 1 = uniform */
    int32_t operation;      /* 0 = additive, 1 = scaling */
    float a, b, a_corr, b_corr;
} BezkNoiseCfg;
int bezk_dr_noise(const float* x, const float* corr, const float* white, uint64_t seed, uint64_t step,
                  const BezkNoiseCfg* cfg, float* y, int64_t total, void* stream);
/* bezk_dr_noise that ALSO writes y_clipped = clamp(y, -clip, clip): VecTask.step clamps the observations after the noise lambda
 * (ref: tasks/base/vec_task.py:338-343), so with a finite clip_obs the clipped copy is refreshed in the same pass. */
int bezk_dr_noise_clip(const float* x, const float* corr, const float* white, uint64_t seed, uint64_t step,
                       const BezkNoiseCfg* cfg, float* y, float* y_clipped, float clip, int64_t total, void* stream);
/* The draws the Philox path of bezk_dr_noise uses for (seed, step): distribution 0 -> N(0,1), 1 -> U[0,1).  Also the way
 * the host creates `corr`. */
int bezk_dr_fill(uint64_t seed, uint64_t step, int32_t distribution, float* out, int64_t total, void* stream);

/* ---------------------------------------------------------------- generic jit helpers (north_star: quat_rotate_inverse, projected gravity, scaling) ----- */

/* ref: isaacgym.torch_utils quat_rotate / quat_rotate_inverse (star-imported by utils/torch_jit_utils.py:31, used by
 * compute_rot :52-63; projected gravity = quat_rotate_inverse(q, gravity_vec)).  q (n,4) xyzw, v (n,3) -> out (n,3).
 * The reference's KickEnv does not call them (its calls are commented out, tasks/kick_env.py:905-908). */
int bezk_quat_rotate(const float* q, const float* v, float* out, int inverse, int64_t n, void* stream);
/* ref: utils/torch_jit_utils.py scale_transform :78-96 (mode 0), unscale_transform :99-117 (mode 1), saturate :119-134 (mode 2).
 * x, y (n,dims) f32 (y may alias x); lower, upper (dims,). */
int bezk_scale_transform(const float* x, const float* lower, const float* upper, float* y, int mode, int64_t n,
                         int32_t dims, void* stream);

/* Diagnostic: the task kernels evaluate IEEE division and square root through branch-free fast sequences with a sticky
 * validity flag and a once-per-env precise recomputation (bezk_common.cuh: Mth).  This checks the fast sequences against the
 * built-in operators over ALL 2^32 radicands and `pairs` random + special quotients.  counts (4,) u64 DEVICE memory:
 * [0] sqrt mismatches, [1] div mismatches (both must be 0), [2] / [3] how many inputs the fast paths accepted. */
int bezk_selftest_fastmath(uint64_t pairs, uint64_t seed, uint64_t* counts, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* BEZK_H_ */
