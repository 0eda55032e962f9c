// Step-based reachers on the device (K8 of DESIGN.md): k_env_step advances B envs by ONE control step — what
// env.step(action) of the reference's classic_control reachers does (base_reacher_direct.py:20-38 /
// base_reacher_torque.py:20-37 with the reward of the configured env), plus gymnasium's TimeLimit truncation.
//
// One thread owns one env.  Unlike k_rollout (fg_rollout.cuh), nothing stays in registers between steps: every launch reads
// the state and the action from HBM and writes the state, the observation, the reward and the flags back (~325 bytes per
// HoleReacher-5 env-step), so the kernel is memory bound.  The per-env rows (q, v: 8 * dof bytes, the observation:
// 4 * (3 * dof + 4) bytes, ...) are strided per thread; they are staged through shared memory so that every global access
// of a warp is one contiguous run.
//
// The step itself is fg_reacher.cuh, the code k_rollout runs for every step of a fused rollout: replaying the actions of a
// fused rollout through this kernel reproduces its per-step observations and rewards bit for bit (tests/test_gpu_step_env.py).
#include <cuda_runtime.h>

#include "fancy_gym_b200.h"
#include "fg_env_step.h"
#include "fg_reacher.cuh"

namespace fg {

constexpr int kStepThreads = 128;

// a block's rows of a [B, W] array, copied between HBM and shared memory with consecutive threads on consecutive elements
template <typename T>
__device__ __forceinline__ void rows_in(T* __restrict__ s, const T* __restrict__ g, int n) {
  for (int i = threadIdx.x; i < n; i += kStepThreads) s[i] = g[i];
}
template <typename T>
__device__ __forceinline__ void rows_out(T* __restrict__ g, const T* __restrict__ s, int n) {
  for (int i = threadIdx.x; i < n; i += kStepThreads) g[i] = s[i];
}

template <int ENV, int N, bool A64>
__global__ void __launch_bounds__(kStepThreads)
k_env_step(const __grid_constant__ ReacherCfg c, const __grid_constant__ fg_env_step_io io, const long long B) {
  using A = typename std::conditional<A64, double, float>::type;
  constexpr int BD = kStepThreads;
  constexpr int NO = obs_dim(ENV, N);
  constexpr bool VEL = (ENV == FG_ENV_HOLE_REACHER || ENV == FG_ENV_VIAPOINT_REACHER);   // velocity controlled (direct)
  __shared__ float s_m[kLinePoints];
  __shared__ double sq[BD * N], sv[BD * N], sctx[BD * 4], sinfo[BD * 2];
  __shared__ A sa[BD * N];
  __shared__ float sobs[BD * NO];

  const int tid = threadIdx.x;
  const long long b0 = (long long)blockIdx.x * BD;
  const int nh = (int)min((long long)BD, B - b0);
  if constexpr (ENV == FG_ENV_HOLE_REACHER) stage_line_points<BD>(s_m);
  rows_in(sq, io.q + b0 * N, nh * N);
  rows_in(sv, io.v + b0 * N, nh * N);
  rows_in(sa, static_cast<const A*>(io.action) + b0 * N, nh * N);
  rows_in(sctx, io.ctx + b0 * 4, nh * 4);
  __syncthreads();

  if (tid < nh) {
    const long long b = b0 + tid;
    double q[N], v[N], a64[N];
    float a32[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
      q[i] = sq[tid * N + i];
      v[i] = sv[tid * N + i];
      a32[i] = (float)sa[tid * N + i];            // (float32 actions: the action itself)
      a64[i] = A64 ? (double)sa[tid * N + i] : (double)a32[i];
    }
    const int steps = io.steps[b];
    const double cx[4] = {sctx[tid * 4 + 0], sctx[tid * 4 + 1], sctx[tid * 4 + 2], sctx[tid * 4 + 3]};

    // v holds the previous float32 action unless the actions are float64 or the env has just been reset (float64 zeros)
    const double acc_cost = reacher_dynamics<ENV, N, A64>(c, __frcp_rn(c.dt_f), __drcp_rn(c.dt), q, v, a64, a32, A64 || !io.v_is_f32 || steps == 0);
    double th[N];
    th[0] = q[0];
#pragma unroll
    for (int i = 1; i < N; ++i) th[i] = th[i - 1] + q[i];
    double ex, ey;                 // float64 end effector (base_reacher.py:95-103): observation and infos of every step
    end_effector64<N>(th, ex, ey);
    ReacherCfg cfg = c;
    cfg.wall_mode = 0;      // the exact wall test: a constant keeps the A/B modes of wall_collision out of this kernel
    auto latch_get = [&](double& x, double& y) { x = io.latch[b * 2 + 0]; y = io.latch[b * 2 + 1]; };
    auto latch_put = [&](double x, double y) { io.latch[b * 2 + 0] = x; io.latch[b * 2 + 1] = y; };
    const StepReward r = reacher_reward<ENV, N, A64>(cfg, q, th, a64, a32, acc_cost, steps, cx, hole_of(cx), s_m,
                                                     [&](double& x, double& y) { x = ex; y = ey; }, latch_get, latch_put);
    const double reward = r.deferred ? collided_reward<ENV>(c, cx, r.aux, ex, ey, latch_put) : r.reward;
    const int steps1 = steps + 1;
    const bool terminated = VEL && r.collided;                              // hole_reacher.py:76-77, viapoint_reacher.py:38
    const bool truncated = c.max_steps > 0 && steps1 >= c.max_steps;       // gymnasium TimeLimit (App. A.6-Q12)
    reacher_obs<ENV, N>(sobs + tid * NO, q, v, cx, ex, ey, steps1);

#pragma unroll
    for (int i = 0; i < N; ++i) {
      sq[tid * N + i] = q[i];
      sv[tid * N + i] = v[i];
    }
    sinfo[tid * 2 + 0] = ENV == FG_ENV_SIMPLE_REACHER ? r.info0 : ex;
    sinfo[tid * 2 + 1] = ENV == FG_ENV_SIMPLE_REACHER ? r.info1 : ey;
    io.steps[b] = steps1;
    io.done[b] = (terminated || truncated) ? 1 : 0;
    io.reward[b] = reward;
    io.flag_bytes[b] = terminated;
    io.flag_bytes[B + b] = truncated;
    io.flag_bytes[2 * B + b] = r.success;
    io.flag_bytes[3 * B + b] = r.collided;
  }
  __syncthreads();
  rows_out(io.q + b0 * N, sq, nh * N);
  rows_out(io.v + b0 * N, sv, nh * N);
  rows_out(io.obs + b0 * NO, sobs, nh * NO);
  rows_out(io.info + b0 * 2, sinfo, nh * 2);
}

template <int ENV, int N>
static cudaError_t launch_n(const ReacherCfg& c, bool a64, const fg_env_step_io& io, long long B, cudaStream_t s) {
  const unsigned blocks = (unsigned)((B + kStepThreads - 1) / kStepThreads);
  if (a64) k_env_step<ENV, N, true><<<blocks, kStepThreads, 0, s>>>(c, io, B);
  else k_env_step<ENV, N, false><<<blocks, kStepThreads, 0, s>>>(c, io, B);
  return cudaGetLastError();
}

template <int ENV>
static cudaError_t launch_env(const ReacherCfg& c, int n, bool a64, const fg_env_step_io& io, long long B, cudaStream_t s,
                              const char** why) {
  switch (n) {
    case 2: return launch_n<ENV, 2>(c, a64, io, B, s);
    case 3: return launch_n<ENV, 3>(c, a64, io, B, s);
    case 4: return launch_n<ENV, 4>(c, a64, io, B, s);
    case 5: return launch_n<ENV, 5>(c, a64, io, B, s);
    case 6: return launch_n<ENV, 6>(c, a64, io, B, s);
    case 7: return launch_n<ENV, 7>(c, a64, io, B, s);
    default: *why = "n_dof outside the instantiated 2..7"; return cudaSuccess;
  }
}

cudaError_t launch_env_step(const ReacherCfg& c, int env_kind, int n_dof, bool a64, const fg_env_step_io& io, long long B,
                            cudaStream_t stream, const char** why) {
  switch (env_kind) {
    case FG_ENV_HOLE_REACHER: return launch_env<FG_ENV_HOLE_REACHER>(c, n_dof, a64, io, B, stream, why);
    case FG_ENV_VIAPOINT_REACHER: return launch_env<FG_ENV_VIAPOINT_REACHER>(c, n_dof, a64, io, B, stream, why);
    case FG_ENV_SIMPLE_REACHER: return launch_env<FG_ENV_SIMPLE_REACHER>(c, n_dof, a64, io, B, stream, why);
    default: *why = "env_kind has no step kernel"; return cudaSuccess;
  }
}

}  // namespace fg
