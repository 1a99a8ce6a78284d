// extern "C" surface of libbezk.so (declared in include/bezk.h): argument validation + launches.
// Plain pointers and sizes only; no torch types; no allocation; no synchronisation.
#include "bezk_internal.h"
#include <stdio.h>
#include <string.h>



static thread_local char g_err[256] = "";

static int fail(int code, const char* what) {
    snprintf(g_err, sizeof(g_err), "%s", what);
    return code;
}
static int cuda_rc(cudaError_t e, const char* where) {
    if (e == cudaSuccess) return 0;
    snprintf(g_err, sizeof(g_err), "%s: %s", where, cudaGetErrorString(e));
    return (int)e;
}
static int check_cfg(const BezkTaskCfg* c) {
    if (!c) return fail(BEZK_E_BADARG, "cfg is NULL");
    const int span = (c->flags & BEZK_F_CLEATS) ? 4 : 1;
    if (c->num_bodies <= 0 || c->imu_body < 0 || c->imu_body >= c->num_bodies || c->left_foot_body < 0 ||
        c->right_foot_body < 0 || c->left_foot_body + span > c->num_bodies || c->right_foot_body + span > c->num_bodies)
        return fail(BEZK_E_CONFIG, "body index outside num_bodies");
    if (!(c->dt > 0.0f) || c->max_episode_length <= 0) return fail(BEZK_E_CONFIG, "dt / max_episode_length must be positive");
    return 0;
}
#define REQUIRE(cond, msg) do { if (!(cond)) return fail(BEZK_E_BADARG, msg); } while (0)
#define ALIGNED(p, a) ((reinterpret_cast<uintptr_t>(p) & ((a) - 1)) == 0)

extern "C" {

int bezk_version(void) { return BEZK_VERSION; }
const char* bezk_last_error(void) { return g_err; }

int bezk_set_l2_fetch_granularity(int32_t bytes, int32_t* effective) {
    REQUIRE(bytes == 32 || bytes == 64 || bytes == 128, "granularity must be 32, 64 or 128");
    cudaError_t e = cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)bytes);
    if (e != cudaSuccess) return cuda_rc(e, "cudaDeviceSetLimit(MaxL2FetchGranularity)");
    size_t got = 0;
    e = cudaDeviceGetLimit(&got, cudaLimitMaxL2FetchGranularity);
    if (effective) *effective = (int32_t)got;
    return cuda_rc(e, "cudaDeviceGetLimit(MaxL2FetchGranularity)");
}

int bezk_pre_physics(const float* actions, float* actions_out, float* targets, const BezkTaskCfg* cfg, int64_t n, void* stream) {
    if (int rc = check_cfg(cfg)) return rc;
    REQUIRE(n >= 0, "n < 0");
    if (n == 0) return 0;
    REQUIRE(actions && targets, "actions/targets NULL");
    return cuda_rc(bezk::launch_pre_physics(actions, actions_out, targets, *cfg, n, (cudaStream_t)stream), "bezk_pre_physics");
}

// rl_games play_steps reward path in the fused step's epilogue (bezk_post_physics_rollout and the host-pipeline entries)
static void set_rollout(bezk::TaskArgs& a, const BezkRolloutCfg* rollout, const float* values, float* shaped_rewards, uint8_t* dones_u8) {
    a.shaped_rew = shaped_rewards; a.dones_u8 = dones_u8;
    if (shaped_rewards) {
        a.shp_scale = rollout->scale_value; a.shp_shift = rollout->shift_value; a.shp_gamma = rollout->gamma;
        a.shp_bootstrap = rollout->value_bootstrap != 0;
        a.values = a.shp_bootstrap ? values : nullptr;
    }
}

// The step's tensors as one TaskArgs: reset_buf / progress_buf are read and written in place, what an entry does not take is
// NULL / 0 (fill_alignment derives the defaults)
static bezk::TaskArgs step_args(float* dof_state, const float* rigid_body, float* root_states, float* net_contact, float* prev_lin_vel,
                                float* goal, const float* goal_angle, const float* ball_init, const float* initial_root_states,
                                const float* uniforms, const float* goal_uniforms, uint64_t seed, uint64_t step, int64_t* reset_buf,
                                int64_t* progress_buf, int64_t* timeout_buf, int64_t* randomize_buf, float* obs, float* obs_clipped,
                                float* rew, int64_t n, int64_t env_base, float* dof_state_wb, float* root_states_wb) {
    bezk::TaskArgs a;
    memset(&a, 0, sizeof(a));
    a.dof_state = dof_state; a.rigid_body = rigid_body; a.root_states = root_states; a.net_contact = net_contact;
    a.prev_lin_vel = prev_lin_vel; a.goal = goal; a.goal_angle = goal_angle; a.goal_uniforms = goal_uniforms; a.ball_init = ball_init;
    a.initial_root = initial_root_states; a.uniforms = uniforms; a.seed = seed; a.step = step; a.env_base = env_base;
    a.dof_state_wb = dof_state_wb; a.root_states_wb = root_states_wb;
    a.reset_in = reset_buf; a.reset_out = reset_buf; a.progress_in = progress_buf; a.progress_out = progress_buf;
    a.timeout_buf = timeout_buf; a.randomize_buf = randomize_buf;
    a.obs = obs; a.obs_clipped = obs_clipped; a.rew = rew; a.n = n;
    return a;
}

static int run_task(int parts, bezk::TaskArgs& a, const BezkTaskCfg* cfg, void* stream, const char* where, int task = BEZK_TASK_KICK,
                    bezk::EpArgs* ep = nullptr, const bezk::NormArgs* nm = nullptr, bezk::OutArgs* oa = nullptr,
                    bezk::TermArgs* ta = nullptr) {
    if (int rc = check_cfg(cfg)) return rc;
    REQUIRE(a.n >= 0, "n < 0");
    if (a.n == 0) return 0;
    REQUIRE(a.dof_state && a.rigid_body && a.root_states, "state tensor NULL");
    if (task == BEZK_TASK_KICK) {
        REQUIRE(a.goal && a.ball_init, "goal / ball_init NULL");
        if (!ALIGNED(a.goal, 8) || !ALIGNED(a.ball_init, 8)) return fail(BEZK_E_ALIGN, "goal / ball_init must be 8-byte aligned");
    } else {
        REQUIRE(parts == 2 || parts == 3 || parts == 4 || parts == 7, "walk / orient: parts must be 2, 3, 4 or 7");
        REQUIRE(a.goal, "goal NULL");
        if (!ALIGNED(a.goal, 8)) return fail(BEZK_E_ALIGN, "goal must be 8-byte aligned");
        if (task == BEZK_TASK_ORIENT) REQUIRE(a.goal_angle, "goal_angle NULL");
    }
    if (parts & BEZK_PART_OBS) REQUIRE(a.net_contact && a.obs, "net_contact/obs NULL");
    if (parts & BEZK_PART_REWARD) REQUIRE(a.rew && a.reset_in && a.reset_out && a.progress_in, "reward buffers NULL");
    if (parts & BEZK_PART_BOOKKEEP) {
        REQUIRE(a.reset_in && a.reset_out && a.progress_in && a.progress_out && a.timeout_buf, "bookkeeping buffers NULL");
        if (cfg->flags & BEZK_F_RESET_ROOT_STATES) REQUIRE(a.initial_root, "initial_root_states NULL");
    }
    bezk::fill_alignment(a, *cfg);
    bezk::set_l2_policy(task, cfg->flags, a, ep);
    if (ep) ep->w = (a.n + 31) / 32;
    if (oa) oa->w = (a.n + 31) / 32;
    if (ta) ta->w = (a.n + 31) / 32;
    return cuda_rc(bezk::launch_task(task, parts, a, *cfg, ep, (cudaStream_t)stream, nm, oa, ta), where);
}

int bezk_compute_observations(const float* dof_state, const float* rigid_body, const float* root_states, float* net_contact,
                              float* prev_lin_vel, const float* goal, const float* ball_init, const BezkTaskCfg* cfg,
                              float* obs, float* obs_clipped, int64_t n, void* stream) {
    bezk::TaskArgs a = step_args(const_cast<float*>(dof_state), rigid_body, const_cast<float*>(root_states), net_contact, prev_lin_vel,
                                 const_cast<float*>(goal), nullptr, ball_init, nullptr, nullptr, nullptr, 0, 0, nullptr, nullptr, nullptr,
                                 nullptr, obs, obs_clipped, nullptr, n, 0, nullptr, nullptr);
    return run_task(BEZK_PART_OBS, a, cfg, stream, "bezk_compute_observations");
}

int bezk_compute_reward(const float* dof_state, const float* rigid_body, const float* root_states, const float* goal,
                        const float* ball_init, const int64_t* reset_in, const int64_t* progress, const BezkTaskCfg* cfg,
                        float* rew, int64_t* reset_out, int64_t n, void* stream) {
    bezk::TaskArgs a = step_args(const_cast<float*>(dof_state), rigid_body, const_cast<float*>(root_states), nullptr, nullptr,
                                 const_cast<float*>(goal), nullptr, ball_init, nullptr, nullptr, nullptr, 0, 0, nullptr, nullptr, nullptr,
                                 nullptr, nullptr, nullptr, rew, n, 0, nullptr, nullptr);
    a.reset_in = reset_in; a.reset_out = reset_out; a.progress_in = progress;     // the reset mask goes to its own buffer; progress is only read
    return run_task(BEZK_PART_REWARD, a, cfg, stream, "bezk_compute_reward");
}

int bezk_reset_idx(const int64_t* env_ids, int64_t k, const float* uniforms, uint64_t seed, uint64_t step, float* dof_state,
                   float* root_states, const float* initial_root_states, int64_t* progress, int64_t* reset,
                   const BezkTaskCfg* cfg, int64_t n, void* stream) {
    if (int rc = check_cfg(cfg)) return rc;
    REQUIRE(k >= 0 && n >= 0, "k/n < 0");
    if (k == 0) return 0;
    REQUIRE(env_ids && dof_state && progress && reset, "reset_idx buffers NULL");
    if (cfg->flags & BEZK_F_RESET_ROOT_STATES) REQUIRE(root_states && initial_root_states, "root state buffers NULL");
    return cuda_rc(bezk::launch_reset_idx(env_ids, k, uniforms, seed, step, dof_state, root_states, initial_root_states, progress,
                                          reset, *cfg, n, BEZK_TASK_KICK, nullptr, nullptr, 0, (cudaStream_t)stream), "bezk_reset_idx");
}

int bezk_reset_idx_task(int task, const int64_t* env_ids, int64_t k, const float* uniforms, const float* goal_uniforms, uint64_t seed,
                        uint64_t step, float* dof_state, float* root_states, const float* initial_root_states, float* goal,
                        int64_t* progress, int64_t* reset, const BezkTaskCfg* cfg, int64_t env_base, int64_t n, void* stream) {
    REQUIRE(task == BEZK_TASK_KICK || task == BEZK_TASK_WALK || task == BEZK_TASK_ORIENT, "unknown task");
    if (int rc = check_cfg(cfg)) return rc;
    REQUIRE(k >= 0 && n >= 0 && env_base >= 0, "k / n / env_base < 0");
    if (k == 0) return 0;
    REQUIRE(env_ids && dof_state && progress && reset, "reset_idx buffers NULL");
    if (task != BEZK_TASK_KICK) REQUIRE(goal, "goal NULL");
    if (cfg->flags & BEZK_F_RESET_ROOT_STATES) REQUIRE(root_states && initial_root_states, "root state buffers NULL");
    return cuda_rc(bezk::launch_reset_idx(env_ids, k, uniforms, seed, step, dof_state, root_states, initial_root_states, progress,
                                          reset, *cfg, n, task, goal, goal_uniforms, env_base, (cudaStream_t)stream), "bezk_reset_idx_task");
}

int bezk_post_physics(float* dof_state, const float* rigid_body, float* root_states, float* net_contact, float* prev_lin_vel,
                      const float* goal, const float* ball_init, const float* initial_root_states, const float* uniforms,
                      uint64_t seed, uint64_t step, int64_t* reset_buf, int64_t* progress_buf, int64_t* timeout_buf,
                      int64_t* randomize_buf, const BezkTaskCfg* cfg, float* obs, float* obs_clipped, float* rew, int parts,
                      int64_t n, void* stream) {
    REQUIRE(parts >= 1 && parts <= 7, "parts must be a non-empty subset of {1,2,4}");
    bezk::TaskArgs a = step_args(dof_state, rigid_body, root_states, net_contact, prev_lin_vel, const_cast<float*>(goal), nullptr, ball_init,
                                 initial_root_states, uniforms, nullptr, seed, step, reset_buf, progress_buf, timeout_buf, randomize_buf,
                                 obs, obs_clipped, rew, n, 0, nullptr, nullptr);
    return run_task(parts, a, cfg, stream, "bezk_post_physics");
}

int bezk_post_physics_chunk(float* dof_state, const float* rigid_body, float* root_states, float* net_contact, float* prev_lin_vel,
                            const float* goal, const float* ball_init, const float* initial_root_states, const float* uniforms,
                            uint64_t seed, uint64_t step, int64_t* reset_buf, int64_t* progress_buf, int64_t* timeout_buf,
                            int64_t* randomize_buf, const BezkTaskCfg* cfg, float* obs, float* obs_clipped, float* rew, int parts,
                            int64_t n, int64_t env_base, float* dof_state_wb, float* root_states_wb, void* stream) {
    REQUIRE(parts >= 1 && parts <= 7, "parts must be a non-empty subset of {1,2,4}");
    REQUIRE(env_base >= 0, "env_base < 0");
    bezk::TaskArgs a = step_args(dof_state, rigid_body, root_states, net_contact, prev_lin_vel, const_cast<float*>(goal), nullptr, ball_init,
                                 initial_root_states, uniforms, nullptr, seed, step, reset_buf, progress_buf, timeout_buf, randomize_buf,
                                 obs, obs_clipped, rew, n, env_base, dof_state_wb, root_states_wb);
    return run_task(parts, a, cfg, stream, "bezk_post_physics_chunk");
}

int bezk_stage_sparse_rows(const float* rigid_body_host, const float* net_contact_host, const BezkTaskCfg* cfg, float* imu_stage,
                           float* feet_stage, int64_t env0, int64_t n, void* stream) {
    if (int rc = check_cfg(cfg)) return rc;
    REQUIRE(env0 >= 0 && n >= 0, "env0 / n < 0");
    if (n == 0) return 0;
    REQUIRE(rigid_body_host && net_contact_host && imu_stage && feet_stage, "staging buffers NULL");
    return cuda_rc(bezk::stage_sparse_rows(rigid_body_host, net_contact_host, *cfg, imu_stage, feet_stage, env0, n,
                                           (cudaStream_t)stream), "bezk_stage_sparse_rows");
}

int bezk_stage_sparse_rows_split(const float* rigid_body_host, const float* net_contact_host, const BezkTaskCfg* cfg, float* imu_stage,
                                 float* feet_stage, int64_t env0, int64_t n, void* copy_stream, void* gather_stream) {
    if (int rc = check_cfg(cfg)) return rc;
    REQUIRE(env0 >= 0 && n >= 0, "env0 / n < 0");
    if (n == 0) return 0;
    REQUIRE(rigid_body_host && net_contact_host && imu_stage && feet_stage, "staging buffers NULL");
    cudaError_t e = bezk::stage_imu_rows(rigid_body_host, *cfg, imu_stage, env0, n, (cudaStream_t)copy_stream);
    if (e == cudaSuccess) e = bezk::stage_feet_gather(net_contact_host, *cfg, feet_stage, env0, n, (cudaStream_t)gather_stream);
    return cuda_rc(e, "bezk_stage_sparse_rows_split");
}

int bezk_host_pack_config(int32_t threads, int32_t spin_us, int32_t pin) {
    if (threads < 0 || threads > 64) { fail(BEZK_E_BADARG, "threads must be 0 (default) .. 64"); return -BEZK_E_BADARG; }
    return bezk::host_pack_config(threads, spin_us, pin);
}

int bezk_host_pack_record_floats(int task, const BezkTaskCfg* cfg) {
    if (!(task == BEZK_TASK_KICK || task == BEZK_TASK_WALK || task == BEZK_TASK_ORIENT)) { fail(BEZK_E_BADARG, "unknown task"); return -BEZK_E_BADARG; }
    if (int rc = check_cfg(cfg)) return -rc;
    return bezk::pack_layout(task, *cfg).stride;
}

int64_t bezk_host_pack_begin(int task, const float* rigid_body_host, const float* net_contact_host, const float* root_states_host,
                             const float* dof_state_host, const float* values_host, const BezkTaskCfg* cfg, float* dst, int64_t env0,
                             int64_t n) {
    if (!(task == BEZK_TASK_KICK || task == BEZK_TASK_WALK || task == BEZK_TASK_ORIENT)) return -(int64_t)fail(BEZK_E_BADARG, "unknown task");
    if (int rc = check_cfg(cfg)) return -(int64_t)rc;
    if (env0 < 0 || n < 0) return -(int64_t)fail(BEZK_E_BADARG, "env0 / n < 0");
    if (n == 0) return 0;
    if (!(rigid_body_host && net_contact_host && root_states_host && dst)) return -(int64_t)fail(BEZK_E_BADARG, "pack buffers NULL");
    if (!ALIGNED(dst, 16)) return -(int64_t)fail(BEZK_E_ALIGN, "dst must be 16-byte aligned");
    return bezk::host_pack_begin(task, rigid_body_host, net_contact_host, root_states_host, dof_state_host, values_host, *cfg, dst, env0, n);
}

int bezk_host_pack_wait(int64_t ticket) {
    if (bezk::host_pack_wait(ticket) != 0) return fail(BEZK_E_BADARG, "bezk_host_pack_wait: unknown ticket");
    return 0;
}

int bezk_post_physics_staged(int task, float* dof_state, const float* imu_stage, float* root_states, float* feet_stage,
                             float* prev_lin_vel, float* goal, const float* goal_angle, const float* ball_init,
                             const float* initial_root_states, const float* uniforms, const float* goal_uniforms, uint64_t seed,
                             uint64_t step, int64_t* reset_buf, int64_t* progress_buf, int64_t* timeout_buf, int64_t* randomize_buf,
                             const BezkTaskCfg* cfg, float* obs, float* obs_clipped, float* rew, int parts, int64_t n,
                             int64_t env_base, float* dof_state_wb, float* root_states_wb, const BezkRolloutCfg* rollout,
                             const float* values, float* shaped_rewards, uint8_t* dones_u8, void* stream) {
    REQUIRE(task == BEZK_TASK_KICK || task == BEZK_TASK_WALK || task == BEZK_TASK_ORIENT, "unknown task");
    REQUIRE(parts >= 1 && parts <= 7, "parts must be a non-empty subset of {1,2,4}");
    REQUIRE(env_base >= 0, "env_base < 0");
    REQUIRE(cfg, "cfg is NULL");
    REQUIRE(!(cfg->flags & BEZK_F_WRITE_CONTACT_FILTER), "the contact-filter write-back would land in the staging buffer: clear BEZK_F_WRITE_CONTACT_FILTER");
    REQUIRE(!(shaped_rewards || dones_u8) || parts == 7, "the reward epilogue rides in the fused step (parts = 7)");
    REQUIRE(!shaped_rewards || rollout, "shaped_rewards requested without a BezkRolloutCfg");
    REQUIRE(!(shaped_rewards && rollout && rollout->value_bootstrap) || values, "value_bootstrap needs values");
    bezk::TaskArgs a = step_args(dof_state, imu_stage, root_states, feet_stage, prev_lin_vel, goal, goal_angle, ball_init, initial_root_states,
                                 uniforms, goal_uniforms, seed, step, reset_buf, progress_buf, timeout_buf, randomize_buf, obs, obs_clipped,
                                 rew, n, env_base, dof_state_wb, root_states_wb);
    const bool cleats = (cfg->flags & BEZK_F_CLEATS) != 0;
    a.rb_stride = 10; a.rb_off = 0;
    a.cf_stride = cleats ? 24 : 8; a.cf_l_off = 0; a.cf_r_off = cleats ? 12 : 4;
    set_rollout(a, rollout, values, shaped_rewards, dones_u8);
    return run_task(parts, a, cfg, stream, "bezk_post_physics_staged", task);
}

int bezk_post_physics_packed(int task, float* dof_state, const float* records, float* root_states, float* prev_lin_vel, float* goal,
                             const float* goal_angle, const float* ball_init, const float* initial_root_states, const float* uniforms,
                             const float* goal_uniforms, uint64_t seed, uint64_t step, int64_t* reset_buf, int64_t* progress_buf,
                             int64_t* timeout_buf, int64_t* randomize_buf, const BezkTaskCfg* cfg, float* obs, float* obs_clipped,
                             float* rew, int parts, int64_t n, int64_t env_base, float* dof_state_wb, float* root_states_wb,
                             const BezkRolloutCfg* rollout, const float* values, float* shaped_rewards, uint8_t* dones_u8,
                             void* stream) {
    REQUIRE(task == BEZK_TASK_KICK || task == BEZK_TASK_WALK || task == BEZK_TASK_ORIENT, "unknown task");
    REQUIRE(parts >= 1 && parts <= 7, "parts must be a non-empty subset of {1,2,4}");
    REQUIRE(env_base >= 0 && n >= 0, "env_base / n < 0");
    REQUIRE(!(shaped_rewards || dones_u8) || parts == 7, "the reward epilogue rides in the fused step (parts = 7)");
    REQUIRE(!shaped_rewards || rollout, "shaped_rewards requested without a BezkRolloutCfg");
    if (int rc = check_cfg(cfg)) return rc;
    if (n == 0) return 0;
    REQUIRE(records && root_states, "records / root_states NULL");
    REQUIRE(!(cfg->flags & BEZK_F_WRITE_CONTACT_FILTER), "the contact-filter write-back would land in the records: clear BEZK_F_WRITE_CONTACT_FILTER");
    const bezk::PackLayout L = bezk::pack_layout(task, *cfg);
    if (int rc = cuda_rc(bezk::launch_unpack_root(task, records, L, root_states, n, (cudaStream_t)stream), "bezk_post_physics_packed (unpack)"))
        return rc;
    bezk::TaskArgs a = step_args(dof_state, records, root_states, const_cast<float*>(records), prev_lin_vel, goal, goal_angle, ball_init,
                                 initial_root_states, uniforms, goal_uniforms, seed, step, reset_buf, progress_buf, timeout_buf, randomize_buf,
                                 obs, obs_clipped, rew, n, env_base, dof_state_wb, root_states_wb);
    a.rb_stride = L.stride; a.rb_off = 0;
    a.cf_stride = L.stride; a.cf_l_off = L.l_off; a.cf_r_off = L.r_off;
    // values == NULL with value_bootstrap: the critic values ride in the records' last float (bezk_host_pack_begin's values_host)
    const bool in_records = shaped_rewards && rollout->value_bootstrap && values == nullptr;
    set_rollout(a, rollout, in_records ? records + (L.stride - 1) : values, shaped_rewards, dones_u8);
    if (in_records) a.values_stride = L.stride;
    return run_task(parts, a, cfg, stream, "bezk_post_physics_packed", task);
}

int bezk_post_physics_task(int task, float* dof_state, const float* rigid_body, float* root_states, float* net_contact,
                           float* prev_lin_vel, float* goal, const float* goal_angle, const float* ball_init,
                           const float* initial_root_states, const float* uniforms, const float* goal_uniforms, uint64_t seed,
                           uint64_t step, int64_t* reset_buf, int64_t* progress_buf, int64_t* timeout_buf, int64_t* randomize_buf,
                           const BezkTaskCfg* cfg, float* obs, float* obs_clipped, float* rew, int parts, int64_t n, void* stream) {
    REQUIRE(task == BEZK_TASK_KICK || task == BEZK_TASK_WALK || task == BEZK_TASK_ORIENT, "unknown task");
    REQUIRE(parts >= 1 && parts <= 7, "parts must be a non-empty subset of {1,2,4}");
    bezk::TaskArgs a = step_args(dof_state, rigid_body, root_states, net_contact, prev_lin_vel, goal, goal_angle, ball_init, initial_root_states,
                                 uniforms, goal_uniforms, seed, step, reset_buf, progress_buf, timeout_buf, randomize_buf, obs, obs_clipped,
                                 rew, n, 0, nullptr, nullptr);
    return run_task(parts, a, cfg, stream, "bezk_post_physics_task", task);
}

}  // extern "C"

// the whole step with the optional episode accumulators, observation normaliser, outcome counts and reward terms: the body of
// bezk_post_physics_rollout_ep_norm (outcome_partials and term_partials NULL), bezk_post_physics_rollout_ep_outcome (term_partials
// NULL) and bezk_post_physics_rollout_ep_terms
static int rollout_step(int task, float* dof_state, const float* rigid_body, float* root_states, float* net_contact, float* prev_lin_vel,
                        float* goal, const float* goal_angle, const float* ball_init, const float* initial_root_states,
                        const float* uniforms, const float* goal_uniforms, uint64_t seed, uint64_t step, int64_t* reset_buf,
                        int64_t* progress_buf, int64_t* timeout_buf, int64_t* randomize_buf, const BezkTaskCfg* cfg, float* obs,
                        float* obs_clipped, float* rew, const BezkRolloutCfg* rollout, const float* values, float* shaped_rewards,
                        uint8_t* dones_u8, int64_t env_base, int64_t n, float* ep_return, float* ep_length, double* ep_partials,
                        const double* obs_mean, const double* obs_var, float obs_eps, float* obs_norm, int32_t* outcome_partials,
                        double* term_partials, void* stream) {
    REQUIRE(task == BEZK_TASK_KICK || task == BEZK_TASK_WALK || task == BEZK_TASK_ORIENT, "unknown task");
    REQUIRE(env_base >= 0, "env_base < 0");
    REQUIRE(!shaped_rewards || rollout, "shaped_rewards requested without a BezkRolloutCfg");
    REQUIRE(!(shaped_rewards && rollout && rollout->value_bootstrap) || values, "value_bootstrap needs values");
    const int armed = (ep_return != nullptr) + (ep_length != nullptr) + (ep_partials != nullptr);
    REQUIRE(armed == 0 || armed == 3, "ep_return, ep_length and ep_partials must be all NULL or all non-NULL");
    if (armed && !(ALIGNED(ep_return, 4) && ALIGNED(ep_length, 4) && ALIGNED(ep_partials, 8)))
        return fail(BEZK_E_ALIGN, "ep_return / ep_length must be 4-byte and ep_partials 8-byte aligned");
    const int norm = (obs_mean != nullptr) + (obs_var != nullptr) + (obs_norm != nullptr);
    REQUIRE(norm == 0 || norm == 3, "obs_mean, obs_var and obs_norm must be all NULL or all non-NULL");
    if (norm) {
        REQUIRE(armed == 3, "obs_norm needs the episode accumulators: ep_return, ep_length and ep_partials are NULL");
        REQUIRE(obs_eps >= 0.0f, "obs_eps must be >= 0");
        if (!ALIGNED(obs_norm, 16)) return fail(BEZK_E_ALIGN, "obs_norm must be 16-byte aligned");
        if (!(ALIGNED(obs_mean, 8) && ALIGNED(obs_var, 8))) return fail(BEZK_E_ALIGN, "obs_mean / obs_var must be 8-byte aligned");
    }
    bezk::TaskArgs a = step_args(dof_state, rigid_body, root_states, net_contact, prev_lin_vel, goal, goal_angle, ball_init, initial_root_states,
                                 uniforms, goal_uniforms, seed, step, reset_buf, progress_buf, timeout_buf, randomize_buf, obs, obs_clipped,
                                 rew, n, env_base, nullptr, nullptr);
    set_rollout(a, rollout, values, shaped_rewards, dones_u8);
    bezk::EpArgs ep = {ep_return, ep_length, ep_partials, 0};
    const bezk::NormArgs nm = {obs_mean, obs_var, obs_norm, obs_eps};
    bezk::OutArgs oa = {outcome_partials, 0};
    bezk::TermArgs ta = {term_partials, 0};
    return run_task(BEZK_PART_BOOKKEEP | BEZK_PART_OBS | BEZK_PART_REWARD, a, cfg, stream,
                    term_partials ? "bezk_post_physics_rollout_ep_terms"
                                  : (outcome_partials ? "bezk_post_physics_rollout_ep_outcome"
                                                      : (norm ? "bezk_post_physics_rollout_ep_norm"
                                                              : (armed ? "bezk_post_physics_rollout_ep" : "bezk_post_physics_rollout"))),
                    task, armed ? &ep : nullptr, norm ? &nm : nullptr, outcome_partials ? &oa : nullptr, term_partials ? &ta : nullptr);
}

extern "C" {

int bezk_post_physics_rollout_ep_norm(int task, float* dof_state, const float* rigid_body, float* root_states, float* net_contact,
                                      float* prev_lin_vel, float* goal, const float* goal_angle, const float* ball_init,
                                      const float* initial_root_states, const float* uniforms, const float* goal_uniforms, uint64_t seed,
                                      uint64_t step, int64_t* reset_buf, int64_t* progress_buf, int64_t* timeout_buf,
                                      int64_t* randomize_buf, const BezkTaskCfg* cfg, float* obs, float* obs_clipped, float* rew,
                                      const BezkRolloutCfg* rollout, const float* values, float* shaped_rewards, uint8_t* dones_u8,
                                      int64_t env_base, int64_t n, float* ep_return, float* ep_length, double* ep_partials,
                                      const double* obs_mean, const double* obs_var, float obs_eps, float* obs_norm, void* stream) {
    return rollout_step(task, dof_state, rigid_body, root_states, net_contact, prev_lin_vel, goal, goal_angle, ball_init,
                        initial_root_states, uniforms, goal_uniforms, seed, step, reset_buf, progress_buf, timeout_buf, randomize_buf, cfg,
                        obs, obs_clipped, rew, rollout, values, shaped_rewards, dones_u8, env_base, n, ep_return, ep_length, ep_partials,
                        obs_mean, obs_var, obs_eps, obs_norm, nullptr, nullptr, stream);
}

int bezk_post_physics_rollout_ep_outcome(int task, float* dof_state, const float* rigid_body, float* root_states, float* net_contact,
                                         float* prev_lin_vel, float* goal, const float* goal_angle, const float* ball_init,
                                         const float* initial_root_states, const float* uniforms, const float* goal_uniforms,
                                         uint64_t seed, uint64_t step, int64_t* reset_buf, int64_t* progress_buf, int64_t* timeout_buf,
                                         int64_t* randomize_buf, const BezkTaskCfg* cfg, float* obs, float* obs_clipped, float* rew,
                                         const BezkRolloutCfg* rollout, const float* values, float* shaped_rewards, uint8_t* dones_u8,
                                         int64_t env_base, int64_t n, float* ep_return, float* ep_length, double* ep_partials,
                                         const double* obs_mean, const double* obs_var, float obs_eps, float* obs_norm,
                                         int32_t* outcome_partials, void* stream) {
    REQUIRE(task == BEZK_TASK_KICK || task == BEZK_TASK_WALK || task == BEZK_TASK_ORIENT, "unknown task");
    REQUIRE(outcome_partials, "outcome_partials NULL");
    REQUIRE(ep_return && ep_length && ep_partials, "the outcome counts need the episode accumulators: ep_return, ep_length and ep_partials must be non-NULL");
    if (!ALIGNED(outcome_partials, 4)) return fail(BEZK_E_ALIGN, "outcome_partials must be 4-byte aligned");
    return rollout_step(task, dof_state, rigid_body, root_states, net_contact, prev_lin_vel, goal, goal_angle, ball_init,
                        initial_root_states, uniforms, goal_uniforms, seed, step, reset_buf, progress_buf, timeout_buf, randomize_buf, cfg,
                        obs, obs_clipped, rew, rollout, values, shaped_rewards, dones_u8, env_base, n, ep_return, ep_length, ep_partials,
                        obs_mean, obs_var, obs_eps, obs_norm, outcome_partials, nullptr, stream);
}

int bezk_post_physics_rollout_ep_terms(int task, float* dof_state, const float* rigid_body, float* root_states, float* net_contact,
                                       float* prev_lin_vel, float* goal, const float* goal_angle, const float* ball_init,
                                       const float* initial_root_states, const float* uniforms, const float* goal_uniforms,
                                       uint64_t seed, uint64_t step, int64_t* reset_buf, int64_t* progress_buf, int64_t* timeout_buf,
                                       int64_t* randomize_buf, const BezkTaskCfg* cfg, float* obs, float* obs_clipped, float* rew,
                                       const BezkRolloutCfg* rollout, const float* values, float* shaped_rewards, uint8_t* dones_u8,
                                       int64_t env_base, int64_t n, float* ep_return, float* ep_length, double* ep_partials,
                                       const double* obs_mean, const double* obs_var, float obs_eps, float* obs_norm,
                                       int32_t* outcome_partials, double* term_partials, void* stream) {
    REQUIRE(task == BEZK_TASK_KICK || task == BEZK_TASK_WALK || task == BEZK_TASK_ORIENT, "unknown task");
    REQUIRE(term_partials, "term_partials NULL");
    REQUIRE(ep_return && ep_length && ep_partials, "the reward terms need the episode accumulators: ep_return, ep_length and ep_partials must be non-NULL");
    REQUIRE(!obs_mean && !obs_var && !obs_norm, "the reward terms do not ride with the observation normaliser: obs_mean, obs_var and obs_norm must be NULL");
    if (!ALIGNED(term_partials, 8)) return fail(BEZK_E_ALIGN, "term_partials must be 8-byte aligned");
    if (!ALIGNED(outcome_partials, 4)) return fail(BEZK_E_ALIGN, "outcome_partials must be 4-byte aligned");
    return rollout_step(task, dof_state, rigid_body, root_states, net_contact, prev_lin_vel, goal, goal_angle, ball_init,
                        initial_root_states, uniforms, goal_uniforms, seed, step, reset_buf, progress_buf, timeout_buf, randomize_buf, cfg,
                        obs, obs_clipped, rew, rollout, values, shaped_rewards, dones_u8, env_base, n, ep_return, ep_length, ep_partials,
                        obs_mean, obs_var, obs_eps, obs_norm, outcome_partials, term_partials, stream);
}

int bezk_post_physics_rollout_ep(int task, float* dof_state, const float* rigid_body, float* root_states, float* net_contact,
                                 float* prev_lin_vel, float* goal, const float* goal_angle, const float* ball_init,
                                 const float* initial_root_states, const float* uniforms, const float* goal_uniforms, uint64_t seed,
                                 uint64_t step, int64_t* reset_buf, int64_t* progress_buf, int64_t* timeout_buf, int64_t* randomize_buf,
                                 const BezkTaskCfg* cfg, float* obs, float* obs_clipped, float* rew, const BezkRolloutCfg* rollout,
                                 const float* values, float* shaped_rewards, uint8_t* dones_u8, int64_t env_base, int64_t n,
                                 float* ep_return, float* ep_length, double* ep_partials, void* stream) {
    return bezk_post_physics_rollout_ep_norm(task, dof_state, rigid_body, root_states, net_contact, prev_lin_vel, goal, goal_angle,
                                             ball_init, initial_root_states, uniforms, goal_uniforms, seed, step, reset_buf, progress_buf,
                                             timeout_buf, randomize_buf, cfg, obs, obs_clipped, rew, rollout, values, shaped_rewards,
                                             dones_u8, env_base, n, ep_return, ep_length, ep_partials, nullptr, nullptr, 0.0f, nullptr,
                                             stream);
}

int bezk_post_physics_rollout(int task, float* dof_state, const float* rigid_body, float* root_states, float* net_contact,
                              float* prev_lin_vel, float* goal, const float* goal_angle, const float* ball_init,
                              const float* initial_root_states, const float* uniforms, const float* goal_uniforms, uint64_t seed,
                              uint64_t step, int64_t* reset_buf, int64_t* progress_buf, int64_t* timeout_buf, int64_t* randomize_buf,
                              const BezkTaskCfg* cfg, float* obs, float* obs_clipped, float* rew, const BezkRolloutCfg* rollout,
                              const float* values, float* shaped_rewards, uint8_t* dones_u8, int64_t env_base, int64_t n,
                              void* stream) {
    return bezk_post_physics_rollout_ep(task, dof_state, rigid_body, root_states, net_contact, prev_lin_vel, goal, goal_angle, ball_init,
                                        initial_root_states, uniforms, goal_uniforms, seed, step, reset_buf, progress_buf, timeout_buf,
                                        randomize_buf, cfg, obs, obs_clipped, rew, rollout, values, shaped_rewards, dones_u8, env_base, n,
                                        nullptr, nullptr, nullptr, stream);
}

int bezk_episode_meter_update(const double* partials, int steps, int64_t n, int64_t games_to_track, float* mean2, int64_t* size2,
                              void* stream) {
    REQUIRE(steps >= 0 && n >= 0, "steps / n < 0");
    REQUIRE(games_to_track > 0, "games_to_track must be positive");
    if (steps == 0 || n == 0) return 0;
    REQUIRE(partials && mean2 && size2, "partials / mean2 / size2 NULL");
    if (!ALIGNED(partials, 8) || !ALIGNED(mean2, 4) || !ALIGNED(size2, 8))
        return fail(BEZK_E_ALIGN, "partials / size2 must be 8-byte and mean2 4-byte aligned");
    return cuda_rc(bezk::launch_episode_meter_update(partials, steps, n, games_to_track, mean2, size2, (cudaStream_t)stream),
                   "bezk_episode_meter_update");
}

int bezk_player_tally_update(const double* partials, int steps, int64_t n, int64_t games_num, double* tally, double* per_step,
                             void* stream) {
    REQUIRE(steps >= 0 && n >= 0, "steps / n < 0");
    REQUIRE(games_num > 0, "games_num must be positive");
    if (steps == 0 || n == 0) return 0;
    REQUIRE(partials && tally, "partials / tally NULL");
    if (!ALIGNED(partials, 8) || !ALIGNED(tally, 8) || !ALIGNED(per_step, 8))
        return fail(BEZK_E_ALIGN, "partials / tally / per_step must be 8-byte aligned");
    return cuda_rc(bezk::launch_player_tally_update(partials, steps, n, games_num, tally, per_step, (cudaStream_t)stream),
                   "bezk_player_tally_update");
}

int bezk_outcome_classes(int task) {
    REQUIRE(task == BEZK_TASK_KICK || task == BEZK_TASK_WALK || task == BEZK_TASK_ORIENT, "unknown task");
    return bezk::outcome_classes(task);
}

int bezk_outcome_meter_update(const int32_t* partials, int steps, int64_t n, int task, int64_t games_to_track, float* mean_k,
                              int64_t* size, void* stream) {
    REQUIRE(task == BEZK_TASK_KICK || task == BEZK_TASK_WALK || task == BEZK_TASK_ORIENT, "unknown task");
    REQUIRE(steps >= 0 && n >= 0, "steps / n < 0");
    REQUIRE(games_to_track > 0, "games_to_track must be positive");
    if (steps == 0 || n == 0) return 0;
    REQUIRE(partials && mean_k && size, "partials / mean_k / size NULL");
    if (!ALIGNED(partials, 4) || !ALIGNED(mean_k, 4) || !ALIGNED(size, 8))
        return fail(BEZK_E_ALIGN, "partials / mean_k must be 4-byte and size 8-byte aligned");
    return cuda_rc(bezk::launch_outcome_meter_update(partials, steps, n, bezk::outcome_classes(task), games_to_track, mean_k, size,
                                                     (cudaStream_t)stream), "bezk_outcome_meter_update");
}

int bezk_player_outcome_update(const int32_t* partials, int steps, int64_t n, int task, int64_t games_num, double* counts,
                               double* per_step, void* stream) {
    REQUIRE(task == BEZK_TASK_KICK || task == BEZK_TASK_WALK || task == BEZK_TASK_ORIENT, "unknown task");
    REQUIRE(steps >= 0 && n >= 0, "steps / n < 0");
    REQUIRE(games_num > 0, "games_num must be positive");
    if (steps == 0 || n == 0) return 0;
    REQUIRE(partials && counts, "partials / counts NULL");
    if (!ALIGNED(partials, 4) || !ALIGNED(counts, 8) || !ALIGNED(per_step, 8))
        return fail(BEZK_E_ALIGN, "partials must be 4-byte and counts / per_step 8-byte aligned");
    return cuda_rc(bezk::launch_player_outcome_update(partials, steps, n, bezk::outcome_classes(task), games_num, counts, per_step,
                                                      (cudaStream_t)stream), "bezk_player_outcome_update");
}

int bezk_reward_terms(int task) {
    REQUIRE(task == BEZK_TASK_KICK || task == BEZK_TASK_WALK || task == BEZK_TASK_ORIENT, "unknown task");
    return bezk::reward_terms(task);
}

int bezk_reward_terms_update(const double* partials, int steps, int64_t n, int task, double* mean_k, void* stream) {
    REQUIRE(task == BEZK_TASK_KICK || task == BEZK_TASK_WALK || task == BEZK_TASK_ORIENT, "unknown task");
    REQUIRE(steps >= 0 && n >= 0, "steps / n < 0");
    if (steps == 0 || n == 0) return 0;
    REQUIRE(partials && mean_k, "partials / mean_k NULL");
    if (!ALIGNED(partials, 8) || !ALIGNED(mean_k, 8)) return fail(BEZK_E_ALIGN, "partials / mean_k must be 8-byte aligned");
    return cuda_rc(bezk::launch_reward_terms_update(partials, steps, n, bezk::reward_terms(task), mean_k, (cudaStream_t)stream),
                   "bezk_reward_terms_update");
}

int bezk_goal_uniforms(uint64_t seed, uint64_t step, float* out2, void* stream) {
    REQUIRE(out2, "out2 NULL");
    return cuda_rc(bezk::launch_goal_uniforms(seed, step, out2, (cudaStream_t)stream), "bezk_goal_uniforms");
}

int bezk_l2_release(const void* ptr, uint64_t bytes, void* stream) {
    if (bytes == 0) return 0;
    REQUIRE(ptr, "ptr NULL");
    return cuda_rc(bezk::launch_l2_release(ptr, bytes, (cudaStream_t)stream), "bezk_l2_release");
}

int bezk_philox_uniforms(uint64_t seed, uint64_t step, float* out, int64_t n, void* stream) {
    REQUIRE(n >= 0, "n < 0");
    if (n == 0) return 0;
    REQUIRE(out, "out NULL");
    return cuda_rc(bezk::launch_philox_uniforms(seed, step, out, n, (cudaStream_t)stream), "bezk_philox_uniforms");
}

int bezk_gae(const float* rewards, const float* values, const void* dones, const float* last_values, const void* last_dones,
             int dones_kind, double gamma, double tau, float* advs, float* returns, int32_t horizon, int64_t n, void* stream) {
    REQUIRE(horizon >= 0 && n >= 0, "horizon/n < 0");
    REQUIRE(dones_kind == 0 || dones_kind == 1, "dones_kind must be 0 (uint8) or 1 (float32)");
    if (horizon == 0 || n == 0) return 0;
    REQUIRE(rewards && values && dones && last_values && last_dones && advs && returns, "gae buffers NULL");
    return cuda_rc(bezk::launch_gae(rewards, values, dones, last_values, last_dones, dones_kind, gamma, tau, advs, returns,
                                    horizon, n, (cudaStream_t)stream), "bezk_gae");
}

int64_t bezk_rms_scratch_doubles(int32_t c) { return bezk::rms_scratch_doubles(c); }

int bezk_rms_moments(const float* x, const double* pivot, double* acc, double* partials, int64_t m, int32_t c, void* stream) {
    REQUIRE(m > 0 && c > 0, "m/c must be positive");
    REQUIRE(x && acc && partials, "rms buffers NULL");
    return cuda_rc(bezk::launch_rms_moments(x, pivot, acc, partials, m, c, m, m, (cudaStream_t)stream), "bezk_rms_moments");
}

static int check_slabs(int64_t& slab_rows, int64_t& slab_stride, int64_t m) {
    if (slab_rows <= 0 || slab_rows >= m) { slab_rows = m; slab_stride = m; return 0; }
    REQUIRE(m % slab_rows == 0, "m must be a multiple of slab_rows");
    REQUIRE(slab_stride >= slab_rows, "slab_stride < slab_rows (slabs would overlap)");
    return 0;
}

int bezk_rms_moments_slabs(const float* x, int64_t slab_rows, int64_t slab_stride, const double* pivot, double* acc,
                           double* partials, int64_t m, int32_t c, void* stream) {
    REQUIRE(m > 0 && c > 0, "m/c must be positive");
    REQUIRE(x && acc && partials, "rms buffers NULL");
    if (int rc = check_slabs(slab_rows, slab_stride, m)) return rc;
    return cuda_rc(bezk::launch_rms_moments(x, pivot, acc, partials, m, c, slab_rows, slab_stride, (cudaStream_t)stream),
                   "bezk_rms_moments_slabs");
}

int bezk_rms_moments_slabs_batched(const float* x, int64_t slab_rows, int64_t slab_stride, int64_t batch_stride, const double* pivot,
                                   double* acc, double* partials, int64_t m, int32_t c, int32_t n_batches, void* stream) {
    REQUIRE(m > 0 && c > 0 && n_batches >= 0 && n_batches <= 65535 && batch_stride >= 0, "bad m / c / n_batches / batch_stride");
    if (n_batches == 0) return 0;
    REQUIRE(x && acc && partials, "rms buffers NULL");
    if (slab_rows <= 0 || slab_rows > m) { slab_rows = m; slab_stride = m; }
    if (int rc = check_slabs(slab_rows, slab_stride, m)) return rc;
    return cuda_rc(bezk::launch_rms_moments_batched(x, pivot, acc, partials, m, c, slab_rows, slab_stride, batch_stride, n_batches,
                                                    (cudaStream_t)stream), "bezk_rms_moments_slabs_batched");
}

int bezk_rms_merge(const double* acc, const double* pivot, double* running_mean, double* running_var, double* count, int32_t c,
                   void* stream) {
    REQUIRE(c > 0, "c must be positive");
    REQUIRE(acc && running_mean && running_var && count, "rms buffers NULL");
    return cuda_rc(bezk::launch_rms_merge(acc, pivot, running_mean, running_var, count, c, (cudaStream_t)stream), "bezk_rms_merge");
}

int bezk_rms_merge_sequence(const double* acc, int32_t n_batches, const int32_t* order, int32_t n_updates, const double* pivot,
                            double* running_mean, double* running_var, double* count, double* seq, int32_t c, void* stream) {
    REQUIRE(c > 0 && c <= 1024, "c must be 1 .. 1024");
    REQUIRE(n_batches > 0 && n_updates >= 0, "n_batches must be positive, n_updates non-negative");
    if (n_updates == 0) return 0;
    REQUIRE(acc && order && running_mean && running_var && count && seq, "rms buffers NULL");
    return cuda_rc(bezk::launch_rms_merge_sequence(acc, order, n_updates, pivot, running_mean, running_var, count, seq, c,
                                                   (cudaStream_t)stream), "bezk_rms_merge_sequence");
}

int bezk_rms_normalize(const float* x, const double* running_mean, const double* running_var, float eps, int unnorm, float* y,
                       int64_t m, int32_t c, void* stream) {
    REQUIRE(m >= 0 && c > 0 && c <= 4096, "bad m/c");
    if (m == 0) return 0;
    REQUIRE(x && y && running_mean && running_var, "rms buffers NULL");
    return cuda_rc(bezk::launch_rms_normalize(x, running_mean, running_var, eps, unnorm, y, m, c, m, m, (cudaStream_t)stream),
                   "bezk_rms_normalize");
}

int bezk_rms_normalize_slabs(const float* x, int64_t slab_rows, int64_t slab_stride, const double* running_mean,
                             const double* running_var, float eps, int unnorm, float* y, int64_t m, int32_t c, void* stream) {
    REQUIRE(m >= 0 && c > 0 && c <= 4096, "bad m/c");
    if (m == 0) return 0;
    REQUIRE(x && y && running_mean && running_var, "rms buffers NULL");
    if (int rc = check_slabs(slab_rows, slab_stride, m)) return rc;
    REQUIRE(m / slab_rows <= 65535, "more than 65535 slabs");
    return cuda_rc(bezk::launch_rms_normalize(x, running_mean, running_var, eps, unnorm, y, m, c, slab_rows, slab_stride,
                                              (cudaStream_t)stream), "bezk_rms_normalize_slabs");
}

int bezk_rms_normalize_slabs_batched(const float* x, int64_t slab_rows, int64_t slab_stride, int64_t batch_stride,
                                     const double* mean, const double* var, int64_t stat_stride, float eps, float* y, int64_t m,
                                     int32_t c, int32_t n_batches, void* stream) {
    REQUIRE(m >= 0 && c > 0 && c <= 4096 && n_batches >= 0 && n_batches <= 65535, "bad m / c / n_batches");
    if (m == 0 || n_batches == 0) return 0;
    REQUIRE(x && y && mean && var, "rms buffers NULL");
    REQUIRE(batch_stride >= 0 && stat_stride >= 0, "negative stride");
    if (slab_rows <= 0 || slab_rows > m) { slab_rows = m; slab_stride = m; }
    if (int rc = check_slabs(slab_rows, slab_stride, m)) return rc;
    REQUIRE(m / slab_rows <= 65535, "more than 65535 slabs");
    return cuda_rc(bezk::launch_rms_normalize_batched(x, mean, var, eps, y, m, c, slab_rows, slab_stride, batch_stride, stat_stride,
                                                      n_batches, (cudaStream_t)stream), "bezk_rms_normalize_slabs_batched");
}

int bezk_rms_train_forward(const float* x, int64_t slab_rows, int64_t slab_stride, double* running_mean, double* running_var,
                           double* count, float eps, float* y, double* partials, int64_t m, int32_t c, void* stream) {
    REQUIRE(m > 0 && c > 0 && c <= 4096, "bad m/c");
    REQUIRE(x && y && running_mean && running_var && count && partials, "rms buffers NULL");
    if (int rc = check_slabs(slab_rows, slab_stride, m)) return rc;
    cudaStream_t st = (cudaStream_t)stream;
    // the cooperative single-kernel form wins only where the whole pass is latency (c == 1: 8.3 us vs 12.6 us for the chain at
    // 131 072 values); for the 54-wide minibatch its three serial phases lose to the chain's wide kernels (27 us vs 12.6 us,
    // profiles/r02_learner_kernels.md)
    if (c == 1 && bezk::fused_stats_eligible(m, c))
        return cuda_rc(bezk::launch_rms_train_forward(x, running_mean, running_var, count, eps, y, partials, m, c, slab_rows, slab_stride,
                                                      st), "bezk_rms_train_forward");
    // three launches: moments (pivot = the running mean itself, no copy) -> finalize (+ snapshot of the old statistics) ->
    // merge + normalise.  The extended accumulator lives at the tail of `partials`.
    REQUIRE(m / slab_rows <= 65535, "more than 65535 slabs");
    double* acc = partials + bezk::rms_scratch_doubles(c) - (2 + 4 * (int64_t)c);
    cudaError_t e = bezk::launch_rms_moments(x, running_mean, acc, partials, m, c, slab_rows, slab_stride, st, running_var, count);
    if (e == cudaSuccess) e = bezk::launch_rms_merge_normalize(x, acc, running_mean, running_var, count, eps, y, m, c, slab_rows, slab_stride, st);
    return cuda_rc(e, "bezk_rms_train_forward");
}

int bezk_rms_moments_ext(const float* x, int64_t slab_rows, int64_t slab_stride, const double* running_mean, const double* running_var,
                         const double* count, double* acc_ext, double* partials, int64_t m, int32_t c, void* stream) {
    REQUIRE(m > 0 && c > 0 && c <= 4096, "bad m/c");
    REQUIRE(x && running_mean && running_var && count && acc_ext && partials, "rms buffers NULL");
    if (int rc = check_slabs(slab_rows, slab_stride, m)) return rc;
    return cuda_rc(bezk::launch_rms_moments(x, running_mean, acc_ext, partials, m, c, slab_rows, slab_stride, (cudaStream_t)stream,
                                            running_var, count), "bezk_rms_moments_ext");
}

int bezk_rms_merge_normalize(const float* x, int64_t slab_rows, int64_t slab_stride, const double* acc_ext, double* running_mean,
                             double* running_var, double* count, float eps, float* y, int64_t m, int32_t c, void* stream) {
    REQUIRE(m > 0 && c > 0 && c <= 4096, "bad m/c");
    REQUIRE(x && y && acc_ext && running_mean && running_var && count, "rms buffers NULL");
    if (int rc = check_slabs(slab_rows, slab_stride, m)) return rc;
    REQUIRE(m / slab_rows <= 65535, "more than 65535 slabs");
    return cuda_rc(bezk::launch_rms_merge_normalize(x, acc_ext, running_mean, running_var, count, eps, y, m, c, slab_rows, slab_stride,
                                                    (cudaStream_t)stream), "bezk_rms_merge_normalize");
}

int bezk_adv_normalize_fused(const float* returns, const float* values, float* adv_out, double* partials, int normalize, int64_t m,
                             void* stream) {
    REQUIRE(m > 0, "m must be positive");
    REQUIRE(returns && values && adv_out && partials, "adv buffers NULL");
    cudaStream_t st = (cudaStream_t)stream;
    if (bezk::fused_stats_eligible(m, 1))
        return cuda_rc(bezk::launch_adv_fused(returns, values, adv_out, partials, normalize, m, st), "bezk_adv_normalize_fused");
    double* acc = partials + bezk::rms_scratch_doubles(1) - 4;
    cudaError_t e = cudaSuccess;
    if (normalize) e = bezk::launch_adv_moments(returns, values, acc, partials, m, st);
    if (e == cudaSuccess) e = bezk::launch_adv_normalize(returns, values, acc, adv_out, normalize, m, st);
    return cuda_rc(e, "bezk_adv_normalize_fused");
}

int bezk_adv_moments(const float* returns, const float* values, double* acc, double* partials, int64_t m, void* stream) {
    REQUIRE(m > 0, "m must be positive");
    REQUIRE(returns && values && acc && partials, "adv buffers NULL");
    return cuda_rc(bezk::launch_adv_moments(returns, values, acc, partials, m, (cudaStream_t)stream), "bezk_adv_moments");
}

int bezk_adv_normalize(const float* returns, const float* values, const double* acc, float* adv_out, int normalize, int64_t m,
                       void* stream) {
    REQUIRE(m >= 0, "m < 0");
    if (m == 0) return 0;
    REQUIRE(returns && values && adv_out && (acc || !normalize), "adv buffers NULL");
    return cuda_rc(bezk::launch_adv_normalize(returns, values, acc, adv_out, normalize, m, (cudaStream_t)stream), "bezk_adv_normalize");
}

int64_t bezk_ppo_scratch_doubles(void) { return bezk::ppo_scratch_doubles(); }

static int ppo_impl(const float* actions, const float* mu, const float* logstd, const float* old_mu, const float* old_sigma,
                    const float* values, const float* old_values, const float* returns, const float* old_neglogp,
                    const float* advantages, int64_t slab_rows, int64_t slab_stride, const BezkPpoCfg* cfg, double* stats,
                    float* grad_mu, float* grad_values, float* grad_logstd, float* neglogp_out, double* partials, int64_t m,
                    void* stream) {
    REQUIRE(cfg, "cfg NULL");
    REQUIRE(m > 0, "m must be positive");
    REQUIRE(actions && mu && logstd && old_mu && old_sigma && values && old_values && returns && old_neglogp && advantages &&
            stats && partials, "ppo buffers NULL");
    REQUIRE(cfg->bound_form == 0 || cfg->bound_form == 1, "bound_form must be 0 or 1");
    REQUIRE(ALIGNED(actions, 8) && ALIGNED(mu, 8) && ALIGNED(old_mu, 8) && ALIGNED(old_sigma, 8), "row arrays must be 8-byte aligned");
    bezk::PpoArgs a;
    a.actions = actions; a.mu = mu; a.logstd = logstd; a.old_mu = old_mu; a.old_sigma = old_sigma; a.values = values;
    a.old_values = old_values; a.returns = returns; a.old_neglogp = old_neglogp; a.advantages = advantages;
    a.grad_mu = grad_mu; a.grad_values = grad_values; a.neglogp_out = neglogp_out; a.partials = partials; a.m = m; a.use_tma = 0;
    if (int rc = check_slabs(slab_rows, slab_stride, m)) return rc;
    a.slab_rows = slab_rows; a.slab_stride = slab_stride; a.slabs = 0;
    return cuda_rc(bezk::launch_ppo_loss(a, *cfg, stats, grad_logstd, (cudaStream_t)stream), "bezk_ppo_loss");
}

int bezk_ppo_loss(const float* actions, const float* mu, const float* logstd, const float* old_mu, const float* old_sigma,
                  const float* values, const float* old_values, const float* returns, const float* old_neglogp,
                  const float* advantages, const BezkPpoCfg* cfg, double* stats, float* grad_mu, float* grad_values,
                  float* grad_logstd, float* neglogp_out, double* partials, int64_t m, void* stream) {
    return ppo_impl(actions, mu, logstd, old_mu, old_sigma, values, old_values, returns, old_neglogp, advantages, m, m, cfg, stats,
                    grad_mu, grad_values, grad_logstd, neglogp_out, partials, m, stream);
}

int bezk_ppo_loss_slabs(const float* actions, const float* mu, const float* logstd, const float* old_mu, const float* old_sigma,
                        const float* values, const float* old_values, const float* returns, const float* old_neglogp,
                        const float* advantages, int64_t slab_rows, int64_t slab_stride, const BezkPpoCfg* cfg, double* stats,
                        float* grad_mu, float* grad_values, float* grad_logstd, float* neglogp_out, double* partials, int64_t m,
                        void* stream) {
    return ppo_impl(actions, mu, logstd, old_mu, old_sigma, values, old_values, returns, old_neglogp, advantages, slab_rows,
                    slab_stride, cfg, stats, grad_mu, grad_values, grad_logstd, neglogp_out, partials, m, stream);
}

int bezk_swap_and_flatten01(const void* src, void* dst, int32_t horizon, int64_t num_envs, int64_t env0, int64_t envs,
                            int32_t row_bytes, void* stream) {
    REQUIRE(horizon >= 0 && num_envs >= 0 && env0 >= 0 && envs >= 0 && row_bytes >= 0, "negative size");
    REQUIRE(env0 + envs <= num_envs, "env range outside num_envs");
    if (horizon == 0 || envs == 0 || row_bytes == 0) return 0;
    REQUIRE(src && dst, "src/dst NULL");
    return cuda_rc(bezk::launch_swap_flatten(src, dst, horizon, num_envs, env0, envs, row_bytes, (cudaStream_t)stream),
                   "bezk_swap_and_flatten01");
}

int bezk_policy_head(const float* mu, const float* logstd, const float* value_norm, const double* value_mean,
                     const double* value_var, float value_eps, const float* noise, uint64_t seed, uint64_t step, float* actions,
                     float* neglogp, float* values, float* mus, float* sigmas, const BezkTaskCfg* task_cfg, float* env_actions,
                     float* targets, int64_t env_base, int64_t n, void* stream) {
    REQUIRE(n >= 0 && env_base >= 0, "n / env_base < 0");
    if (n == 0) return 0;
    REQUIRE(mu && logstd, "mu/logstd NULL");
    REQUIRE(!values || value_norm, "values requested without value_norm");
    REQUIRE((value_mean == nullptr) == (value_var == nullptr), "value_mean and value_var go together");
    REQUIRE(!targets || task_cfg, "targets requested without task_cfg");
    if (task_cfg) { if (int rc = check_cfg(task_cfg)) return rc; }
    REQUIRE(ALIGNED(mu, 8) && (!noise || ALIGNED(noise, 8)), "mu / noise must be 8-byte aligned");
    return cuda_rc(bezk::launch_policy_head(mu, logstd, value_norm, value_mean, value_var, value_eps, noise, seed, step, actions,
                                            neglogp, values, mus, sigmas, task_cfg, env_actions, targets, env_base, n, (cudaStream_t)stream),
                   "bezk_policy_head");
}

int bezk_dr_noise(const float* x, const float* corr, const float* white, uint64_t seed, uint64_t step, const BezkNoiseCfg* cfg,
                  float* y, int64_t total, void* stream) {
    REQUIRE(cfg, "cfg NULL");
    REQUIRE(total >= 0, "total < 0");
    REQUIRE((cfg->distribution == 0 || cfg->distribution == 1) && (cfg->operation == 0 || cfg->operation == 1), "bad distribution / operation");
    if (total == 0) return 0;
    REQUIRE(x && y, "x / y NULL");
    return cuda_rc(bezk::launch_dr_noise(x, corr, white, seed, step, *cfg, y, nullptr, 0.0f, total, (cudaStream_t)stream), "bezk_dr_noise");
}

int bezk_dr_noise_clip(const float* x, const float* corr, const float* white, uint64_t seed, uint64_t step, const BezkNoiseCfg* cfg,
                       float* y, float* y_clipped, float clip, int64_t total, void* stream) {
    REQUIRE(cfg, "cfg NULL");
    REQUIRE(total >= 0, "total < 0");
    REQUIRE((cfg->distribution == 0 || cfg->distribution == 1) && (cfg->operation == 0 || cfg->operation == 1), "bad distribution / operation");
    if (total == 0) return 0;
    REQUIRE(x && y && y_clipped, "x / y / y_clipped NULL");
    return cuda_rc(bezk::launch_dr_noise(x, corr, white, seed, step, *cfg, y, y_clipped, clip, total, (cudaStream_t)stream),
                   "bezk_dr_noise_clip");
}

int bezk_dr_fill(uint64_t seed, uint64_t step, int32_t distribution, float* out, int64_t total, void* stream) {
    REQUIRE(total >= 0 && (distribution == 0 || distribution == 1), "bad total / distribution");
    if (total == 0) return 0;
    REQUIRE(out, "out NULL");
    return cuda_rc(bezk::launch_dr_fill(seed, step, distribution, out, total, (cudaStream_t)stream), "bezk_dr_fill");
}

int bezk_quat_rotate(const float* q, const float* v, float* out, int inverse, int64_t n, void* stream) {
    REQUIRE(n >= 0, "n < 0");
    if (n == 0) return 0;
    REQUIRE(q && v && out, "q / v / out NULL");
    return cuda_rc(bezk::launch_quat_rotate(q, v, out, inverse != 0, n, (cudaStream_t)stream), "bezk_quat_rotate");
}

int bezk_scale_transform(const float* x, const float* lower, const float* upper, float* y, int mode, int64_t n, int32_t dims,
                         void* stream) {
    REQUIRE(n >= 0 && dims >= 0, "n / dims < 0");
    REQUIRE(mode >= 0 && mode <= 2, "mode must be 0 (scale), 1 (unscale) or 2 (saturate)");
    if (n == 0 || dims == 0) return 0;
    REQUIRE(x && lower && upper && y, "x / lower / upper / y NULL");
    return cuda_rc(bezk::launch_scale_transform(x, lower, upper, y, mode, n, dims, (cudaStream_t)stream), "bezk_scale_transform");
}

int bezk_selftest_fastmath(uint64_t pairs, uint64_t seed, uint64_t* counts, void* stream) {
    REQUIRE(counts, "counts NULL");
    return cuda_rc(bezk::launch_selftest_fastmath(pairs, seed, reinterpret_cast<unsigned long long*>(counts), (cudaStream_t)stream),
                   "bezk_selftest_fastmath");
}

int bezk_normal_noise(uint64_t seed, uint64_t step, float* out, int64_t env_base, int64_t n, void* stream) {
    REQUIRE(n >= 0 && env_base >= 0, "n / env_base < 0");
    if (n == 0) return 0;
    REQUIRE(out, "out NULL");
    return cuda_rc(bezk::launch_normal_noise(seed, step, out, n, env_base, (cudaStream_t)stream), "bezk_normal_noise");
}

}  // extern "C"
