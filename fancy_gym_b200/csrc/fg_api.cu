// C ABI of fancy_gym_b200 (include/fancy_gym_b200.h): handle management and kernel dispatch.
#include <cuda_runtime.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <atomic>
#include <new>
#include <vector>

#include "fancy_gym_b200.h"
#include "fg_device.cuh"
#include "fg_dispatch.h"
#include "fg_env_step.h"
#include "fg_reset.cuh"

namespace {
thread_local char g_err[512] = "";

fg_status fail(fg_status st, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
  return st;
}

#define FG_CUDA(call)                                                                         \
  do {                                                                                        \
    cudaError_t e_ = (call);                                                                  \
    if (e_ != cudaSuccess) return fail(FG_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_)); \
  } while (0)
}  // namespace

struct fg_handle {
  fg_config cfg;
  fg::DevCfg dev;
  int device;
  float* d_tab_a;
  float* d_tab_b;
  float* d_quad_rec;
  // work queues of persistent rollout grids: kQueues pairs of device words (next env, finished blocks), zero between
  // launches (the kernel resets its pair); concurrent launches on different streams take different pairs
  unsigned* d_queue;
  mutable std::atomic<unsigned> next_queue;
  int max_smem_optin;
  int sm_count;
};
static constexpr unsigned kQueues = 64;

extern "C" {

const char* fg_last_error(void) { return g_err; }
int32_t fg_abi_version(void) { return FG_ABI_VERSION; }

fg_status fg_destroy(fg_handle* h);

fg_status fg_create(const fg_config* cfg, int32_t device, fg_handle** out) {
  if (!cfg || !out) return fail(FG_ERR_INVALID, "fg_create: null argument");
  if (cfg->struct_size != sizeof(fg_config))
    return fail(FG_ERR_INVALID, "fg_create: struct_size %u != %zu (ABI mismatch)", cfg->struct_size, sizeof(fg_config));
  if (cfg->n_dof < 1 || cfg->n_dof > FG_MAX_DOF) return fail(FG_ERR_INVALID, "n_dof %d out of range 1..%d", cfg->n_dof, FG_MAX_DOF);
  if (cfg->n_steps < 2) return fail(FG_ERR_INVALID, "n_steps %d < 2", cfg->n_steps);
  if (cfg->env_kind < 0 || cfg->env_kind > FG_ENV_TOY) return fail(FG_ERR_INVALID, "unknown env_kind %d", cfg->env_kind);
  if (cfg->mp_kind < 0 || cfg->mp_kind > FG_MP_TRAJ) return fail(FG_ERR_INVALID, "unknown mp_kind %d", cfg->mp_kind);
  if (cfg->ctrl_kind < 0 || cfg->ctrl_kind > FG_CTRL_MOTOR) return fail(FG_ERR_INVALID, "unknown ctrl_kind %d", cfg->ctrl_kind);
  if (cfg->mp_kind != FG_MP_TRAJ && (cfg->n_basis < 1 || !cfg->tab_a || !cfg->tab_b))
    return fail(FG_ERR_INVALID, "n_basis >= 1 and both tables are required for mp_kind %d", cfg->mp_kind);
  if (cfg->n_obs_out < 0 || cfg->n_obs_out > FG_MAX_OBS) return fail(FG_ERR_INVALID, "n_obs_out %d out of range", cfg->n_obs_out);
  if (cfg->env_kind == FG_ENV_HOLE_REACHER && (cfg->rew_fct < 0 || cfg->rew_fct > 2))
    return fail(FG_ERR_INVALID, "hole reacher rew_fct %d unknown (0 simple, 1 vel_acc, 2 unbounded)", cfg->rew_fct);

  fg_handle* h = new (std::nothrow) fg_handle();
  if (!h) return fail(FG_ERR_NOMEM, "out of host memory");
  h->cfg = *cfg;
  h->device = device;
  h->d_tab_a = h->d_tab_b = h->d_quad_rec = nullptr;
  h->d_queue = nullptr;
  h->next_queue = 0;
  // (any failure from here on frees what has been allocated and restores the caller's current device)
#define FG_CUDA_H(call)                                                                   \
  do {                                                                                    \
    cudaError_t e_ = (call);                                                              \
    if (e_ != cudaSuccess) {                                                              \
      cudaSetDevice(prev);                                                                \
      fg_destroy(h);                                                                      \
      return fail(FG_ERR_CUDA, "%s: %s", #call, cudaGetErrorString(e_));                  \
    }                                                                                     \
  } while (0)
  int prev = 0;
  FG_CUDA_H(cudaGetDevice(&prev));
  FG_CUDA_H(cudaSetDevice(device));
  FG_CUDA_H(cudaDeviceGetAttribute(&h->max_smem_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device));
  FG_CUDA_H(cudaDeviceGetAttribute(&h->sm_count, cudaDevAttrMultiProcessorCount, device));

  fg::DevCfg& d = h->dev;
  memset(&d, 0, sizeof(d));
  const int T = cfg->n_steps, K = cfg->n_basis, N = cfg->n_dof;
  d.n_dof = N; d.T = T; d.K = K;
  d.env.dt = cfg->dt; d.env.dt_f = (float)cfg->dt; d.env.max_steps = cfg->max_episode_steps;
  d.env.allow_self = cfg->allow_self_collision; d.env.allow_wall = cfg->allow_wall_collision;
  d.env.rew_fct = cfg->rew_fct; d.env.wall_mode = cfg->wall_mode; d.env.penalty = cfg->collision_penalty;
  const bool torque = cfg->env_kind == FG_ENV_SIMPLE_REACHER;
  // Box(low=-bound, high=bound) with the default float32 dtype (base_reacher_direct.py:16-18, _torque.py:16-18;
  // ToyEnv: +-1, test_black_box.py:29)
  d.act_lim = torque ? 1000.0f : (cfg->env_kind == FG_ENV_TOY ? 1.0f : (float)(2.0 * fg::kPi));
  for (int i = 0; i < FG_MAX_DOF; ++i) { d.p[i] = cfg->p_gains[i]; d.d[i] = cfg->d_gains[i]; }
  d.tau = cfg->tau; d.alpha = cfg->dmp_alpha; d.beta = cfg->dmp_alpha / 4.0f;
  d.wscale = cfg->weights_scale; d.gscale = cfg->goal_scale; d.rel_goal = cfg->relative_goal;
  d.time_aware = cfg->time_aware; d.ctrl = cfg->ctrl_kind;
  d.n_obs_out = cfg->n_obs_out;
  d.n_obs_full = fg::obs_dim(cfg->env_kind, N) + (cfg->time_aware ? 1 : 0);
  for (int j = 0; j < cfg->n_obs_out; ++j) {
    if (cfg->obs_index[j] < 0 || cfg->obs_index[j] >= d.n_obs_full) {
      cudaSetDevice(prev);
      fg_destroy(h);
      return fail(FG_ERR_INVALID, "obs_index[%d]=%d outside the %d-wide step observation", j, cfg->obs_index[j], d.n_obs_full);
    }
    d.obs_index[j] = cfg->obs_index[j];
  }
  size_t na = 0, nb = 0;
  switch (cfg->mp_kind) {
    case FG_MP_PROMP: d.cols_a = K; d.rows_b = T - 1; d.cols_b = 1; break;
    case FG_MP_DMP: d.cols_a = K; d.rows_b = T - 1; d.cols_b = 1; break;
    case FG_MP_PRODMP: d.cols_a = K + 3; d.rows_b = T; d.cols_b = K + 3; break;
    default: d.cols_a = 0; d.rows_b = 0; d.cols_b = 0; break;
  }
  na = (size_t)T * d.cols_a; nb = (size_t)d.rows_b * d.cols_b;
  if (na) {
    FG_CUDA_H(cudaMalloc(&h->d_tab_a, na * sizeof(float)));
    FG_CUDA_H(cudaMemcpy(h->d_tab_a, cfg->tab_a, na * sizeof(float), cudaMemcpyHostToDevice));
    FG_CUDA_H(cudaMalloc(&h->d_tab_b, nb * sizeof(float)));
    FG_CUDA_H(cudaMemcpy(h->d_tab_b, cfg->tab_b, nb * sizeof(float), cudaMemcpyHostToDevice));
  }
  d.tab_a = h->d_tab_a; d.tab_b = h->d_tab_b;
  if (cfg->mp_kind == FG_MP_PROMP || cfg->mp_kind == FG_MP_PRODMP) {
    // quad records for fg_trajgen (layout: fg_device.cuh); 1/dt is the correctly rounded float32 reciprocal, like __frcp_rn
    const int kw = d.cols_a, r4 = fg::traj_r4(kw), rec4 = fg::traj_rec4(cfg->mp_kind, kw), nq = (T + 3) / 4;
    const int rowf = r4 * 4, recf = rec4 * 4;
    std::vector<float> rec((size_t)nq * recf, 0.f);
    for (int q = 0; q < nq; ++q) {
      float* o = rec.data() + (size_t)q * recf;
      const int rows = (cfg->mp_kind == FG_MP_PROMP) ? 5 : 4;
      for (int r = 0; r < rows; ++r) {
        const int t = (4 * q + r < T - 1) ? 4 * q + r : T - 1;
        for (int col = 0; col < kw; ++col) {
          o[r * rowf + col] = cfg->tab_a[(size_t)t * kw + col];
          if (cfg->mp_kind == FG_MP_PRODMP) o[(4 + r) * rowf + col] = cfg->tab_b[(size_t)t * kw + col];
        }
      }
      if (cfg->mp_kind == FG_MP_PROMP) {
        for (int j = 0; j < 4; ++j) {
          const int tb = (4 * q + j < d.rows_b - 1) ? 4 * q + j : d.rows_b - 1;
          o[5 * rowf + j] = cfg->tab_b[tb];
          o[5 * rowf + 4 + j] = 1.0f / cfg->tab_b[tb];
        }
      }
    }
    FG_CUDA_H(cudaMalloc(&h->d_quad_rec, rec.size() * sizeof(float)));
    FG_CUDA_H(cudaMemcpy(h->d_quad_rec, rec.data(), rec.size() * sizeof(float), cudaMemcpyHostToDevice));
    d.quad_rec = reinterpret_cast<const float4*>(h->d_quad_rec);
    d.quad_rec4 = rec4;
  }
  FG_CUDA_H(cudaMalloc(&h->d_queue, 2 * kQueues * sizeof(unsigned)));
  FG_CUDA_H(cudaMemset(h->d_queue, 0, 2 * kQueues * sizeof(unsigned)));
  h->cfg.tab_a = h->cfg.tab_b = nullptr;   // host pointers are not retained
  FG_CUDA_H(cudaSetDevice(prev));
  *out = h;
  return FG_OK;
#undef FG_CUDA_H
}

fg_status fg_destroy(fg_handle* h) {
  if (!h) return FG_OK;
  if (h->d_tab_a) cudaFree(h->d_tab_a);
  if (h->d_tab_b) cudaFree(h->d_tab_b);
  if (h->d_quad_rec) cudaFree(h->d_quad_rec);
  if (h->d_queue) cudaFree(h->d_queue);
  delete h;
  return FG_OK;
}

int32_t fg_num_params(const fg_handle* h) {
  if (!h) return -1;
  const int kp = (h->cfg.mp_kind == FG_MP_PROMP) ? h->cfg.n_basis : h->cfg.n_basis + 1;
  return h->cfg.mp_kind == FG_MP_TRAJ ? 0 : h->cfg.n_dof * kp;
}

int32_t fg_obs_full_dim(const fg_handle* h) { return h ? h->dev.n_obs_full : -1; }

fg_status fg_rollout(const fg_handle* h, const fg_rollout_io* io, int64_t B, int32_t seg_steps, void* stream) {
  if (!h || !io) return fail(FG_ERR_INVALID, "fg_rollout: null argument");
  if (io->struct_size != sizeof(fg_rollout_io)) return fail(FG_ERR_INVALID, "fg_rollout: io struct_size mismatch");
  if (B < 0) return fail(FG_ERR_INVALID, "fg_rollout: negative batch");
  if (B == 0) return FG_OK;
  if (seg_steps < 1 || seg_steps > h->cfg.n_steps)
    return fail(FG_ERR_INVALID, "fg_rollout: seg_steps %d outside 1..%d", seg_steps, h->cfg.n_steps);
  if (io->n_peers < 0 || (io->n_peers > 0 && (!io->peer_bufs || io->peer_offset < 0 || io->n_plans > 1)))
    return fail(FG_ERR_INVALID, "fg_rollout: peer gather needs peer_bufs, a non-negative offset and one plan per launch");
  if (io->n_plans > 1) {       // plans looped inside the launch: the handle's tables hold every plan's rows
    if (io->n_plans > FG_MAX_PLANS) return fail(FG_ERR_INVALID, "fg_rollout: n_plans %d > FG_MAX_PLANS", io->n_plans);
    if (h->cfg.mp_kind == FG_MP_TRAJ || io->seg_steps_env || io->dbg_actions || io->dbg_obs || io->dbg_rewards || io->dbg_state)
      return fail(FG_ERR_UNSUPPORTED, "fg_rollout: n_plans > 1 needs a table-driven MP and no per-step / per-env-length buffers");
    if (io->plan_T < 2) return fail(FG_ERR_INVALID, "fg_rollout: plan_T %d < 2", io->plan_T);
    for (int j = 0; j < io->n_plans; ++j) {
      const int look = (h->cfg.mp_kind == FG_MP_PROMP && io->plan_seg[j] < io->plan_T) ? 1 : 0;   // ProMP reads row t + 1
      if (io->plan_seg[j] < 1 || io->plan_seg[j] > io->plan_T || io->plan_row0[j] < 0 ||
          io->plan_row0[j] + io->plan_seg[j] + look > h->cfg.n_steps)
        return fail(FG_ERR_INVALID, "fg_rollout: plan %d (rows %d + %d steps) does not fit the handle's %d table rows", j,
                    io->plan_row0[j], io->plan_seg[j], h->cfg.n_steps);
    }
  }
  const bool need_state = h->cfg.env_kind != FG_ENV_TOY;
  if ((need_state && (!io->q || !io->v || !io->ctx)) || !io->steps || !io->done || !io->ret || !io->length ||
      !io->flags || !io->obs || !io->info)
    return fail(FG_ERR_INVALID, "fg_rollout: a required buffer is NULL");
  if (h->cfg.mp_kind == FG_MP_TRAJ ? (!io->traj_pos || !io->traj_vel) : !io->params)
    return fail(FG_ERR_INVALID, "fg_rollout: trajectory source buffer is NULL");
  if ((io->use_cond || io->write_cond) && (!io->cond_pos || !io->cond_vel))
    return fail(FG_ERR_INVALID, "fg_rollout: cond buffers required by use_cond/write_cond");
  int prev = 0;
  FG_CUDA(cudaGetDevice(&prev));
  if (prev != h->device) FG_CUDA(cudaSetDevice(h->device));
  const char* why = nullptr;
  unsigned* queue = h->d_queue + 2 * (h->next_queue.fetch_add(1u) % kQueues);
  fg::PhaseConst pcv;
  const fg::PhaseConst* pc = nullptr;
  if (io->phase) {            // per-env tau / delay evaluated inside the rollout
    const fg_phase_basis* pb = io->phase;
    if (pb->struct_size != sizeof(fg_phase_basis)) { if (prev != h->device) cudaSetDevice(prev); return fail(FG_ERR_INVALID, "fg_rollout: phase struct_size mismatch (ABI)"); }
    if (!io->phase_tau || !io->phase_delay || !io->phase_times || pb->n_basis_total < 1 || pb->n_basis_total > fg::kMaxRbfFused ||
        (pb->n_steps_env != nullptr) != (pb->times_table != nullptr) || (pb->n_steps_env && pb->times_stride < h->cfg.n_steps) ||
        !pb->eval_f64) {
      if (prev != h->device) cudaSetDevice(prev);
      return fail(FG_ERR_UNSUPPORTED, "fg_rollout: per-env phase needs tau / delay / times, 1..%d RBFs and the float64 basis", fg::kMaxRbfFused);
    }
    memset(&pcv, 0, sizeof(pcv));
    pcv.n_total = pb->n_basis_total; pcv.first = pb->first_learnable; pcv.phase_kind = pb->phase_kind;
    pcv.exp_right_clip = pb->exp_right_clip; pcv.alpha_phase = pb->alpha_phase; pcv.basis_scale = pb->basis_scale;
    for (int k = 0; k < fg::kMaxRbfFused; ++k) { pcv.cen[k] = pb->centers[k]; pcv.bw[k] = pb->bandwidth[k]; }
    pcv.tau = io->phase_tau; pcv.delay = io->phase_delay; pcv.times = io->phase_times;
    pcv.n_steps_env = pb->n_steps_env; pcv.times_table = pb->times_table; pcv.times_stride = pb->times_stride;
    const bool no_rec = getenv("FG_PHASE_NO_RECURRENCE") != nullptr;             // (A/B runs and tests: evaluate every RBF directly)
    if (!no_rec) fg::rbf_recurrence(pcv.rec, pcv.cen, pcv.bw, pcv.n_total, pcv.phase_kind);
    pc = &pcv;
  }
  cudaError_t e = fg::launch_rollout(h->dev, h->cfg.env_kind, h->cfg.mp_kind, *io, B, seg_steps,
                                     (cudaStream_t)stream, h->max_smem_optin, &why, queue, h->sm_count, pc);
  if (prev != h->device) cudaSetDevice(prev);
  if (why) return fail(FG_ERR_UNSUPPORTED, "fg_rollout: %s", why);
  if (e != cudaSuccess) return fail(FG_ERR_CUDA, "fg_rollout launch: %s", cudaGetErrorString(e));
  return FG_OK;
}

fg_status fg_trajgen(const fg_handle* h, const float* params, const float* bc_pos, const float* bc_vel,
                     float* pos_out, float* vel_out, int64_t B, void* stream) {
  if (!h || !params || !pos_out || !vel_out) return fail(FG_ERR_INVALID, "fg_trajgen: null argument");
  if (h->cfg.mp_kind == FG_MP_TRAJ) return fail(FG_ERR_INVALID, "fg_trajgen: handle has no trajectory generator");
  if (h->cfg.mp_kind != FG_MP_PROMP && (!bc_pos || !bc_vel))
    return fail(FG_ERR_INVALID, "fg_trajgen: DMP / ProDMP need boundary conditions");
  if (B <= 0) return B == 0 ? FG_OK : fail(FG_ERR_INVALID, "fg_trajgen: negative batch");
  int prev = 0;
  FG_CUDA(cudaGetDevice(&prev));
  if (prev != h->device) FG_CUDA(cudaSetDevice(h->device));
  const char* why = nullptr;
  cudaError_t e = fg::launch_trajgen(h->dev, h->cfg.mp_kind, params, bc_pos, bc_vel, pos_out, vel_out, B,
                                     (cudaStream_t)stream, h->max_smem_optin, h->sm_count, &why);
  if (prev != h->device) cudaSetDevice(prev);
  if (why) return fail(FG_ERR_UNSUPPORTED, "fg_trajgen: %s", why);
  if (e != cudaSuccess) return fail(FG_ERR_CUDA, "fg_trajgen launch: %s", cudaGetErrorString(e));
  return FG_OK;
}

fg_status fg_trajgen_phase(const fg_handle* h, const fg_phase_basis* pb, const float* times, const float* tau,
                           const float* delay, const float* params, const float* bc_pos, const float* bc_vel,
                           float* pos_out, float* vel_out, int64_t B, void* stream) {
  if (!h || !pb || !times || !tau || !delay || !params || !pos_out || !vel_out)
    return fail(FG_ERR_INVALID, "fg_trajgen_phase: null argument");
  if (pb->struct_size != sizeof(fg_phase_basis)) return fail(FG_ERR_INVALID, "fg_trajgen_phase: struct_size mismatch (ABI)");
  if (h->cfg.mp_kind == FG_MP_TRAJ) return fail(FG_ERR_INVALID, "fg_trajgen_phase: handle has no trajectory generator");
  if (h->cfg.mp_kind != FG_MP_PROMP && (!bc_pos || !bc_vel))
    return fail(FG_ERR_INVALID, "fg_trajgen_phase: DMP / ProDMP need boundary conditions");
  if (h->cfg.mp_kind == FG_MP_PRODMP && (!pb->pc_pos || !pb->pc_vel || !pb->pc_y || pb->n_pc < 2 || !(pb->scaled_dt > 0.f)))
    return fail(FG_ERR_INVALID, "fg_trajgen_phase: ProDMP needs the pre-integrated basis tables");
  if (h->cfg.n_basis + 1 > 17) return fail(FG_ERR_UNSUPPORTED, "fg_trajgen_phase: at most 16 basis functions");
  if (h->cfg.mp_kind != FG_MP_PRODMP &&
      (pb->n_basis_total < 1 || pb->n_basis_total > 16 || pb->first_learnable < 0 ||
       pb->first_learnable + h->cfg.n_basis > pb->n_basis_total))
    return fail(FG_ERR_INVALID, "fg_trajgen_phase: basis counts inconsistent (total %d, first %d, weighted %d)",
                pb->n_basis_total, pb->first_learnable, h->cfg.n_basis);
  if (B < 0) return fail(FG_ERR_INVALID, "fg_trajgen_phase: negative batch");
  if (B == 0) return FG_OK;
  fg::PhaseArgs a;
  memset(&a, 0, sizeof(a));
  a.mp_kind = h->cfg.mp_kind; a.N = h->cfg.n_dof; a.T = h->cfg.n_steps; a.K = h->cfg.n_basis;
  a.phase_kind = pb->phase_kind; a.n_total = pb->n_basis_total; a.first = pb->first_learnable; a.alpha_phase = pb->alpha_phase;
  a.exp_right_clip = pb->exp_right_clip; a.basis_scale = pb->basis_scale; a.eval_f64 = pb->eval_f64;
  for (int k = 0; k < 16; ++k) { a.cen32[k] = (float)pb->centers[k]; a.bw32[k] = (float)pb->bandwidth[k]; }
  for (int k = 0; k < 16; ++k) { a.cen[k] = pb->centers[k]; a.bw[k] = pb->bandwidth[k]; }
  if (a.mp_kind == FG_MP_PROMP && a.eval_f64 && !getenv("FG_PHASE_NO_RECURRENCE"))
    fg::rbf_recurrence(a.rec, a.cen, a.bw, a.n_total, a.phase_kind);
  a.wscale = h->cfg.weights_scale; a.gscale = h->cfg.goal_scale; a.alpha = h->cfg.dmp_alpha; a.beta = h->cfg.dmp_alpha / 4.0f;
  a.times = times; a.dts = h->d_tab_b; a.tau = tau; a.delay = delay; a.params = params; a.bc_pos = bc_pos; a.bc_vel = bc_vel;
  a.pos = pos_out; a.vel = vel_out;
  a.pc_pos = pb->pc_pos; a.pc_vel = pb->pc_vel; a.pc_y = pb->pc_y; a.n_pc = pb->n_pc; a.rel_goal = h->cfg.relative_goal;
  a.scaled_dt = pb->scaled_dt; a.init_time = pb->init_time;
  for (int k = 0; k < 17; ++k) a.scale[k] = pb->scale[k];
  if ((pb->n_steps_env != nullptr) != (pb->times_table != nullptr))
    return fail(FG_ERR_INVALID, "fg_trajgen_phase: n_steps_env and times_table go together");
  if (pb->n_steps_env && pb->times_stride < h->cfg.n_steps)
    return fail(FG_ERR_INVALID, "fg_trajgen_phase: times_stride %d is shorter than the longest plan (%d points)",
                pb->times_stride, h->cfg.n_steps);
  a.n_steps_env = pb->n_steps_env; a.times_table = pb->times_table; a.times_stride = pb->times_stride;
  int prev = 0;
  FG_CUDA(cudaGetDevice(&prev));
  if (prev != h->device) FG_CUDA(cudaSetDevice(h->device));
  const char* why = nullptr;
  cudaError_t e = fg::launch_trajgen_phase(a, B, (cudaStream_t)stream, h->max_smem_optin, &why);
  if (prev != h->device) cudaSetDevice(prev);
  if (why) return fail(FG_ERR_UNSUPPORTED, "fg_trajgen_phase: %s", why);
  if (e != cudaSuccess) return fail(FG_ERR_CUDA, "fg_trajgen_phase launch: %s", cudaGetErrorString(e));
  return FG_OK;
}

int64_t fg_traj_cov_work_floats(const fg_handle* h, int64_t B) {
  if (!h || B < 0) return -1;
  return B * (int64_t)h->cfg.n_dof * h->cfg.n_steps + B + 1;
}

fg_status fg_traj_cov(const fg_handle* h, const float* params_L, float reg, int32_t reg_scope, float* cov_out,
                      float* std_out, float* work, int32_t path, int64_t B, void* stream) {
  if (!h || !params_L || !work) return fail(FG_ERR_INVALID, "fg_traj_cov: null argument");
  if (h->cfg.mp_kind != FG_MP_PROMP && h->cfg.mp_kind != FG_MP_PRODMP)
    return fail(FG_ERR_INVALID, "fg_traj_cov: only the probabilistic MPs (ProMP, ProDMP) have a trajectory covariance");
  if (!cov_out && !std_out) return fail(FG_ERR_INVALID, "fg_traj_cov: neither cov_out nor std_out given");
  if (path < 0 || path > 2) return fail(FG_ERR_INVALID, "fg_traj_cov: path %d unknown", path);
  if (B < 0) return fail(FG_ERR_INVALID, "fg_traj_cov: negative batch");
  if (B == 0) return FG_OK;
  fg::CovArgs a;
  memset(&a, 0, sizeof(a));
  a.basis = h->d_tab_a;
  a.ld = h->dev.cols_a;
  a.c0 = (h->cfg.mp_kind == FG_MP_PRODMP) ? 2 : 0;      // ProDMP tables start with the two boundary-condition columns
  a.Kc = h->dev.cols_a - a.c0;
  a.T = h->cfg.n_steps; a.N = h->cfg.n_dof;
  a.L = params_L; a.cov = cov_out; a.stdv = std_out;
  a.diag = work; a.envmax = work + B * (int64_t)a.N * a.T; a.gmax = a.envmax + B;
  a.reg = reg; a.batch_scope = reg_scope ? 1 : 0;
  int prev = 0;
  FG_CUDA(cudaGetDevice(&prev));
  if (prev != h->device) FG_CUDA(cudaSetDevice(h->device));
  const char* why = nullptr;
  cudaError_t e = fg::launch_traj_cov(a, B, path == 0 ? 1 : path, (cudaStream_t)stream, h->max_smem_optin, &why);
  if (prev != h->device) cudaSetDevice(prev);
  if (why) return fail(FG_ERR_UNSUPPORTED, "fg_traj_cov: %s", why);
  if (e != cudaSuccess) return fail(FG_ERR_CUDA, "fg_traj_cov launch: %s", cudaGetErrorString(e));
  return FG_OK;
}

fg_status fg_reset(const fg_reset_cfg* cfg, const fg_reset_io* io, int64_t B, void* stream) {
  if (!cfg || !io) return fail(FG_ERR_INVALID, "fg_reset: null argument");
  if (cfg->struct_size != sizeof(fg_reset_cfg) || io->struct_size != sizeof(fg_reset_io))
    return fail(FG_ERR_INVALID, "fg_reset: struct_size mismatch (ABI)");
  if (cfg->env_kind < FG_ENV_HOLE_REACHER || cfg->env_kind > FG_ENV_SIMPLE_REACHER)
    return fail(FG_ERR_INVALID, "fg_reset: env_kind %d has no reset sampler", cfg->env_kind);
  if (cfg->n_dof < 1 || cfg->n_dof > FG_MAX_DOF) return fail(FG_ERR_INVALID, "fg_reset: n_dof %d out of range", cfg->n_dof);
  if (cfg->n_obs_out < 0 || cfg->n_obs_out > FG_MAX_OBS) return fail(FG_ERR_INVALID, "fg_reset: n_obs_out out of range");
  const int n_full = fg::obs_dim(cfg->env_kind, cfg->n_dof) + (cfg->time_aware ? 1 : 0);
  for (int j = 0; j < cfg->n_obs_out; ++j)
    if (cfg->obs_index[j] < 0 || cfg->obs_index[j] >= n_full)
      return fail(FG_ERR_INVALID, "fg_reset: obs_index[%d]=%d outside the %d-wide observation", j, cfg->obs_index[j], n_full);
  if (B < 0) return fail(FG_ERR_INVALID, "fg_reset: negative batch");
  if (B == 0) return FG_OK;
  if (!io->rng_state || !io->q || !io->v || !io->steps || !io->done || !io->ctx)
    return fail(FG_ERR_INVALID, "fg_reset: a required buffer is NULL");
  if (cfg->n_obs_out > 0 && !io->obs) return fail(FG_ERR_INVALID, "fg_reset: obs buffer is NULL");
  fg::ResetCfg c;
  memset(&c, 0, sizeof(c));
  c.env_kind = cfg->env_kind; c.n_dof = cfg->n_dof; c.random_start = cfg->random_start; c.time_aware = cfg->time_aware;
  for (int i = 0; i < 4; ++i) { c.fixed[i] = cfg->fixed[i]; c.has_fixed[i] = cfg->has_fixed[i]; }
  c.n_obs_out = cfg->n_obs_out;
  for (int j = 0; j < cfg->n_obs_out; ++j) c.obs_index[j] = cfg->obs_index[j];
  int prev = 0;
  FG_CUDA(cudaGetDevice(&prev));
  if (prev != cfg->device) FG_CUDA(cudaSetDevice(cfg->device));
  const unsigned blocks = (unsigned)((B + 127) / 128);
  fg::k_reset<<<blocks, 128, 0, (cudaStream_t)stream>>>(c, *io, B);
  const cudaError_t e = cudaGetLastError();
  if (prev != cfg->device) cudaSetDevice(prev);
  if (e != cudaSuccess) return fail(FG_ERR_CUDA, "fg_reset launch: %s", cudaGetErrorString(e));
  return FG_OK;
}

fg_status fg_env_step(const fg_env_step_cfg* cfg, const fg_env_step_io* io, int64_t B, void* stream) {
  if (!cfg || !io) return fail(FG_ERR_INVALID, "fg_env_step: null argument");
  if (cfg->struct_size != sizeof(fg_env_step_cfg) || io->struct_size != sizeof(fg_env_step_io))
    return fail(FG_ERR_INVALID, "fg_env_step: struct_size mismatch (ABI)");
  if (cfg->env_kind == FG_ENV_TOY) return fail(FG_ERR_UNSUPPORTED, "fg_env_step: the toy env has no step kernel");
  if (cfg->env_kind < FG_ENV_HOLE_REACHER || cfg->env_kind > FG_ENV_SIMPLE_REACHER)
    return fail(FG_ERR_INVALID, "fg_env_step: unknown env_kind %d", cfg->env_kind);
  if (cfg->n_dof < 2 || cfg->n_dof > 7)
    return fail(FG_ERR_UNSUPPORTED, "fg_env_step: n_dof %d outside the instantiated 2..7", cfg->n_dof);
  if (cfg->env_kind == FG_ENV_HOLE_REACHER && (cfg->rew_fct < 0 || cfg->rew_fct > 2))
    return fail(FG_ERR_INVALID, "fg_env_step: hole reacher rew_fct %d unknown (0 simple, 1 vel_acc, 2 unbounded)", cfg->rew_fct);
  if (!(cfg->dt > 0.0)) return fail(FG_ERR_INVALID, "fg_env_step: dt must be positive");
  if (B < 0) return fail(FG_ERR_INVALID, "fg_env_step: negative batch");
  if (!io->action || !io->q || !io->v || !io->steps || !io->done || !io->ctx || !io->obs || !io->reward || !io->flag_bytes ||
      !io->info)
    return fail(FG_ERR_INVALID, "fg_env_step: a required buffer is NULL");
  if (cfg->env_kind == FG_ENV_HOLE_REACHER && cfg->rew_fct == 2 && !io->latch)
    return fail(FG_ERR_INVALID, "fg_env_step: rew_fct \"unbounded\" needs the latch buffer");
  if (B == 0) return FG_OK;
  fg::ReacherCfg c;
  memset(&c, 0, sizeof(c));
  c.dt = cfg->dt; c.dt_f = (float)cfg->dt; c.max_steps = cfg->max_episode_steps;
  c.allow_self = cfg->allow_self_collision; c.allow_wall = cfg->allow_wall_collision; c.rew_fct = cfg->rew_fct;
  c.penalty = cfg->collision_penalty;
  const char* why = nullptr;
  const cudaError_t e = fg::launch_env_step(c, cfg->env_kind, cfg->n_dof, cfg->action_f64 != 0, *io, B, (cudaStream_t)stream, &why);
  if (why) return fail(FG_ERR_UNSUPPORTED, "fg_env_step: %s", why);
  if (e != cudaSuccess) return fail(FG_ERR_CUDA, "fg_env_step launch: %s", cudaGetErrorString(e));
  return FG_OK;
}

}  // extern "C"

// ------------------------------------------------------------------------------------------
// FP32 FFMA probe: 8 independent register chains per thread, fully unrolled inner block.
// ------------------------------------------------------------------------------------------
namespace {
__global__ void __launch_bounds__(256) k_ffma_probe(float* sink, int iters) {
  float a0 = threadIdx.x * 1e-3f, a1 = a0 + 1.f, a2 = a0 + 2.f, a3 = a0 + 3.f;
  float a4 = a0 + 4.f, a5 = a0 + 5.f, a6 = a0 + 6.f, a7 = a0 + 7.f;
  const float m = 0.999f + blockIdx.x * 1e-9f, c = 1e-3f;
  for (int i = 0; i < iters; ++i) {
#pragma unroll
    for (int u = 0; u < 16; ++u) {
      a0 = fmaf(a0, m, c); a1 = fmaf(a1, m, c); a2 = fmaf(a2, m, c); a3 = fmaf(a3, m, c);
      a4 = fmaf(a4, m, c); a5 = fmaf(a5, m, c); a6 = fmaf(a6, m, c); a7 = fmaf(a7, m, c);
    }
  }
  const float r = ((a0 + a1) + (a2 + a3)) + ((a4 + a5) + (a6 + a7));
  if (r == 123.456f) sink[0] = r;   // never true: keeps the chains alive
}
}  // namespace

extern "C" fg_status fg_ffma_probe(int32_t blocks, int32_t iters, float* sink_dev, double* flops, void* stream) {
  if (blocks < 1 || iters < 1 || !sink_dev) return fail(FG_ERR_INVALID, "fg_ffma_probe: bad argument");
  k_ffma_probe<<<blocks, 256, 0, (cudaStream_t)stream>>>(sink_dev, iters);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return fail(FG_ERR_CUDA, "fg_ffma_probe: %s", cudaGetErrorString(e));
  if (flops) *flops = 2.0 * 8.0 * 16.0 * (double)iters * 256.0 * (double)blocks;
  return FG_OK;
}
