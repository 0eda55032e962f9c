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
// The arithmetic is the reference's, dtype for dtype (SURVEY.md App. A.6-Q7), and every expression is the one k_rollout
// evaluates for the same step: replaying the actions of a fused rollout through this kernel reproduces its per-step
// observations and rewards bit for bit (tests/test_gpu_step_env.py).
#include <cuda_runtime.h>

#include "fancy_gym_b200.h"
#include "fg_device.cuh"
#include "fg_env_step.h"

namespace fg {

constexpr int kStepThreads = 128;

__host__ __device__ constexpr int step_obs_dim(int env, int n) {   // hole: width, ee - goal, steps; viapoint: 2 + 2 + 1; simple 2 + 1
  return 3 * n + (env == FG_ENV_HOLE_REACHER ? 4 : env == FG_ENV_VIAPOINT_REACHER ? 5 : 3);
}

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
k_env_step(const __grid_constant__ EnvStepDev c, const __grid_constant__ fg_env_step_io io, const long long B) {
  using A = typename std::conditional<A64, double, float>::type;
  constexpr int BD = kStepThreads;
  constexpr int NO = step_obs_dim(ENV, N);
  constexpr bool VEL = (ENV == FG_ENV_HOLE_REACHER || ENV == FG_ENV_VIAPOINT_REACHER);   // velocity controlled (direct)
  __shared__ float s_m[kLinePoints];
  __shared__ double sq[BD * N], sv[BD * N], sctx[BD * 4], sinfo[BD * 2];
  __shared__ A sa[BD * N];
  __shared__ float sobs[BD * NO];

  const int tid = threadIdx.x;
  const long long b0 = (long long)blockIdx.x * BD;
  const int nh = (int)min((long long)BD, B - b0);
  if constexpr (ENV == FG_ENV_HOLE_REACHER)
    for (int i = tid; i < kLinePoints; i += BD)   // float32(numpy.linspace(0,1,100)), as k_rollout stages it
      s_m[i] = (i == kLinePoints - 1) ? 1.0f : (float)((double)i * (1.0 / 99.0));
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
    const double cx0 = sctx[tid * 4 + 0], cx1 = sctx[tid * 4 + 1], cx2 = sctx[tid * 4 + 2], cx3 = sctx[tid * 4 + 3];

    // ---------------------------------------------------------------- dynamics (no clip: that is the black-box wrapper's)
    double acc_cost = 0.0;    // sum(acc^2) of the velocity-controlled envs, in the reference's dtype
    if constexpr (VEL) {
      // base_reacher_direct.py:25-27.  acc = (a - v) / dt: float64 unless v holds the previous float32 action and the action
      // is float32 (the first step after a reset sees float64 zeros) — k_rollout's `MOTOR || steps == 0`
      if (A64 || !io.v_is_f32 || steps == 0) {
        const double r_dt64 = __drcp_rn(c.dt);
#pragma unroll
        for (int i = 0; i < N; ++i) {
          const double ac = div_by64(a64[i] - v[i], c.dt, r_dt64);
          acc_cost += ac * ac;
        }
      } else {
        const float r_dt = __frcp_rn(c.dt_f);
        float s32 = 0.f;
#pragma unroll
        for (int i = 0; i < N; ++i) {
          const float ac = div_by(__fsub_rn(a32[i], (float)v[i]), c.dt_f, r_dt);
          s32 = __fadd_rn(s32, __fmul_rn(ac, ac));
        }
        acc_cost = (double)s32;
      }
#pragma unroll
      for (int i = 0; i < N; ++i) {
        v[i] = a64[i];
        q[i] += A64 ? __dmul_rn(c.dt, a64[i]) : (double)__fmul_rn(c.dt_f, a32[i]);   // dt * v: float32 for a float32 v
      }
    } else {
      // base_reacher_torque.py:25-26
#pragma unroll
      for (int i = 0; i < N; ++i) {
        v[i] += A64 ? __dmul_rn(c.dt, a64[i]) : (double)__fmul_rn(c.dt_f, a32[i]);
        q[i] += __dmul_rn(c.dt, v[i]);
      }
    }

    // ---------------------------------------------------------------- geometry, collisions, reward
    double th[N];
    th[0] = q[0];
#pragma unroll
    for (int i = 1; i < N; ++i) th[i] = th[i - 1] + q[i];
    double ex, ey;                 // float64 end effector (base_reacher.py:95-103): observation and infos of every step
    end_effector64<N>(th, ex, ey);
    double reward = 0.0, info0 = ex, info1 = ey;
    bool collided = false, success = false;
    if constexpr (ENV == FG_ENV_HOLE_REACHER) {
      float cs[N], sn[N];
#pragma unroll
      for (int i = 0; i < N; ++i) sincos_reduced(th[i], sn[i], cs[i]);
      const Hole hole{(float)(cx0 - cx1 / 2), (float)(cx0 + cx1 / 2), (float)(-cx2)};   // hole_reacher.py:152
      bool selfc = false, wallc = false;
      if (!c.allow_self) selfc = self_collision<N>(q, th, cs, sn);                      // base_reacher.py:105-119
      if (!c.allow_wall) wallc = wall_collision<N>(s_m, cs, sn, hole, 0);               // hole_reacher.py:148-179
      collided = selfc | wallc;
      const double dx = ex - cx0, dy = ey - (-cx2);
      if (c.rew_fct == 0) {
        // hr_simple_reward.py:35-53 (distance and collision terms on the last step of the episode)
        reward = __dmul_rn(acc_cost, -5e-8);
        if (collided) {
          const double dist = sqrt(dx * dx + dy * dy);
          reward = __dadd_rn(__dadd_rn(__dmul_rn(dist * dist, -1.0), reward), __dmul_rn(1.0, -c.penalty));
        } else if (steps == 199) {
          const double dist = sqrt(dx * dx + dy * dy);
          success = dist < 0.005;
          reward = __dadd_rn(__dadd_rn(__dmul_rn(dist * dist, -1.0), reward), __dmul_rn(0.0, -c.penalty));
        }
      } else if (c.rew_fct == 1) {
        // hr_dist_vel_acc_reward.py:20-60: distance / collision terms on step 199 only; factors (-1, -1e-4, -1e-6, -penalty)
        double dist_cost = 0.0, coll_cost = 0.0;
        if (steps == 199) {
          const double dist = sqrt(dx * dx + dy * dy);
          dist_cost = dist * dist;
          coll_cost = collided ? dist * dist : 0.0;
          success = (dist < 0.005) && !collided;
        }
        double vel_cost;
        if constexpr (A64) {
          vel_cost = 0.0;
#pragma unroll
          for (int i = 0; i < N; ++i) vel_cost += a64[i] * a64[i];
        } else {      // np.sum(v ** 2) of a float32 v is a float32 sum
          float s32 = 0.f;
#pragma unroll
          for (int i = 0; i < N; ++i) s32 = __fadd_rn(s32, __fmul_rn(a32[i], a32[i]));
          vel_cost = (double)s32;
        }
        reward = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(dist_cost, -1.0), __dmul_rn(vel_cost, -1e-4)),
                                     __dmul_rn(acc_cost, -1e-6)), __dmul_rn(coll_cost, -c.penalty));
      } else {
        // hr_unbounded_reward.py:17-60: the end effector is latched at step 180 or on a collision; factors (1, -5e-6)
        if (collided) {
          io.latch[b * 2 + 0] = ex;
          io.latch[b * 2 + 1] = ey;
          const double dist = sqrt(dx * dx + dy * dy);
          reward = __dadd_rn(0.25 * exp(-dist), __dmul_rn(acc_cost, -5e-6));
        } else {
          double dist_reward = 0.0;
          if (steps == 180) {
            io.latch[b * 2 + 0] = ex;
            io.latch[b * 2 + 1] = ey;
          } else if (steps == 199) {
            const double lx = io.latch[b * 2 + 0], ly = io.latch[b * 2 + 1];
            const double ldx = lx - cx0, ldy = ly - (-cx2);
            const double dist = sqrt(ldx * ldx + ldy * ldy);
            if (ey > 0) dist_reward = exp(-dist);
            else dist_reward = 1 - ly;
            success = true;
          }
          reward = __dadd_rn(dist_reward, __dmul_rn(acc_cost, -5e-6));
        }
      }
    } else if constexpr (ENV == FG_ENV_VIAPOINT_REACHER) {
      // viapoint_reacher.py:79-107 (App. A.6-Q1/Q2: the reward starts from -inf, `acc` is the action)
      if (!c.allow_self) {
        collided = joint_limits<N>(q);
        if (may_self_intersect<N>(q)) {
          float cs[N], sn[N];
#pragma unroll
          for (int i = 0; i < N; ++i) sincos_reduced(th[i], sn[i], cs[i]);
          collided |= links_intersect<N>(th, cs, sn);
        }
      }
      double act_term;
      if constexpr (A64) {
        double asq = 0.0;
#pragma unroll
        for (int i = 0; i < N; ++i) asq += a64[i] * a64[i];
        act_term = 5e-8 * asq;
      } else {   // np.sum(acc**2) of a float32 action is float32, and 5e-8 * float32 stays float32
        float s32 = 0.f;
#pragma unroll
        for (int i = 0; i < N; ++i) s32 = __fadd_rn(s32, __fmul_rn(a32[i], a32[i]));
        act_term = (double)__fmul_rn(5e-8f, s32);
      }
      if (!collided) {
        double dist = INFINITY;
        reward = -INFINITY;
        if (steps == 100 || steps == 199) {
          const double tx = (steps == 100) ? cx0 : cx2, ty = (steps == 100) ? cx1 : cx3;
          dist = sqrt((ex - tx) * (ex - tx) + (ey - ty) * (ey - ty));
        }
        success = dist < 0.005;
        reward -= dist * dist;
        reward -= act_term;
      } else {
        const double dist = sqrt((ex - cx2) * (ex - cx2) + (ey - cx3) * (ey - cx3));
        reward = -c.penalty;
        reward -= dist * dist;
        reward -= act_term;
      }
    } else {
      // simple_reacher.py:56-70 (the collision flag is computed there but not used)
      double rdist = 0.0;
      if (steps >= 199) rdist = -sqrt((ex - cx0) * (ex - cx0) + (ey - cx1) * (ey - cx1));
      double rctrl;
      if constexpr (A64) {
        rctrl = 0.0;
#pragma unroll
        for (int i = 0; i < N; ++i) rctrl += a64[i] * a64[i];
        reward = rdist - rctrl;
      } else {   // float32 action: reward_ctrl is float32; `0 - float32` stays float32 before step 199
        float s32 = 0.f;
#pragma unroll
        for (int i = 0; i < N; ++i) s32 = __fadd_rn(s32, __fmul_rn(a32[i], a32[i]));
        rctrl = (double)s32;
        reward = (steps >= 199) ? rdist - rctrl : (double)(0.f - s32);
      }
      info0 = rdist;
      info1 = rctrl;
    }
    const int steps1 = steps + 1;
    const bool terminated = VEL && collided;                                // hole_reacher.py:76-77, viapoint_reacher.py:38
    const bool truncated = c.max_steps > 0 && steps1 >= c.max_steps;       // gymnasium TimeLimit (App. A.6-Q12)

    // ---------------------------------------------------------------- observation (_get_obs: float64, cast to float32)
    float* ob = sobs + tid * NO;
#pragma unroll
    for (int i = 0; i < N; ++i) ob[i] = (float)cos(q[i]);
#pragma unroll
    for (int i = 0; i < N; ++i) ob[N + i] = (float)sin(q[i]);
#pragma unroll
    for (int i = 0; i < N; ++i) ob[2 * N + i] = (float)v[i];
    int no = 3 * N;
    if constexpr (ENV == FG_ENV_HOLE_REACHER) {                   // hole_reacher.py:114-124
      ob[no++] = (float)cx1;
      ob[no++] = (float)(ex - cx0);
      ob[no++] = (float)(ey - (-cx2));
    } else if constexpr (ENV == FG_ENV_VIAPOINT_REACHER) {        // viapoint_reacher.py:112-121
      ob[no++] = (float)(ex - cx0);
      ob[no++] = (float)(ey - cx1);
      ob[no++] = (float)(ex - cx2);
      ob[no++] = (float)(ey - cx3);
    } else {                                                      // simple_reacher.py:75-83
      ob[no++] = (float)(ex - cx0);
      ob[no++] = (float)(ey - cx1);
    }
    ob[no++] = (float)steps1;

#pragma unroll
    for (int i = 0; i < N; ++i) {
      sq[tid * N + i] = q[i];
      sv[tid * N + i] = v[i];
    }
    sinfo[tid * 2 + 0] = info0;
    sinfo[tid * 2 + 1] = info1;
    io.steps[b] = steps1;
    io.done[b] = (terminated || truncated) ? 1 : 0;
    io.reward[b] = reward;
    io.flag_bytes[b] = terminated;
    io.flag_bytes[B + b] = truncated;
    io.flag_bytes[2 * B + b] = success;
    io.flag_bytes[3 * B + b] = collided;
  }
  __syncthreads();
  rows_out(io.q + b0 * N, sq, nh * N);
  rows_out(io.v + b0 * N, sv, nh * N);
  rows_out(io.obs + b0 * NO, sobs, nh * NO);
  rows_out(io.info + b0 * 2, sinfo, nh * 2);
}

template <int ENV, int N>
static cudaError_t launch_n(const EnvStepDev& c, bool a64, const fg_env_step_io& io, long long B, cudaStream_t s) {
  const unsigned blocks = (unsigned)((B + kStepThreads - 1) / kStepThreads);
  if (a64) k_env_step<ENV, N, true><<<blocks, kStepThreads, 0, s>>>(c, io, B);
  else k_env_step<ENV, N, false><<<blocks, kStepThreads, 0, s>>>(c, io, B);
  return cudaGetLastError();
}

template <int ENV>
static cudaError_t launch_env(const EnvStepDev& c, int n, bool a64, const fg_env_step_io& io, long long B, cudaStream_t s,
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

cudaError_t launch_env_step(const EnvStepDev& c, int env_kind, int n_dof, bool a64, const fg_env_step_io& io, long long B,
                            cudaStream_t stream, const char** why) {
  switch (env_kind) {
    case FG_ENV_HOLE_REACHER: return launch_env<FG_ENV_HOLE_REACHER>(c, n_dof, a64, io, B, stream, why);
    case FG_ENV_VIAPOINT_REACHER: return launch_env<FG_ENV_VIAPOINT_REACHER>(c, n_dof, a64, io, B, stream, why);
    case FG_ENV_SIMPLE_REACHER: return launch_env<FG_ENV_SIMPLE_REACHER>(c, n_dof, a64, io, B, stream, why);
    default: *why = "env_kind has no step kernel"; return cudaSuccess;
  }
}

}  // namespace fg
