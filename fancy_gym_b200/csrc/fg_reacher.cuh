// One control step of the reference's classic-control reachers (HoleReacher, ViaPointReacher, SimpleReacher), defined once
// for the device: dynamics, collision tests, rewards and observation.  k_rollout (fg_rollout.cuh) runs it inside the fused
// black-box loop, k_env_step (fg_env_step.cu) once per launch; k_reset (fg_reset.cuh) shares the observation's context part.
//
// The arithmetic is the reference's, dtype for dtype (SURVEY.md App. A.6-Q7).  F64 is the dtype of the action: float64
// (a PD controller's torque, a float64 env.step action) or float32 (the clipped desired velocity / position, a float32
// env.step action); a64 always holds the action as float64, a32 the float32 action when !F64.
#pragma once
#include <type_traits>

#include "fg_device.cuh"

namespace fg {

// width of the step observation without the time_aware entry (the toy env observes one value)
__host__ __device__ constexpr int obs_dim(int env, int n) {   // hole: width, ee - goal, steps; viapoint: 2 + 2 + 1; simple 2 + 1
  return env == FG_ENV_TOY ? 1 : 3 * n + (env == FG_ENV_HOLE_REACHER ? 4 : env == FG_ENV_VIAPOINT_REACHER ? 5 : 3);
}

// float32(numpy.linspace(0,1,100)) into shared memory: i*(1/99) in float64, last forced to 1 (the wall samples)
template <int BD>
__device__ __forceinline__ void stage_line_points(float* s_m) {
  for (int i = threadIdx.x; i < kLinePoints; i += BD) s_m[i] = (i == kLinePoints - 1) ? 1.0f : (float)((double)i * (1.0 / 99.0));
}

// hole_reacher.py:152 (x - width/2), rounded once to float32
__device__ __forceinline__ Hole hole_of(const double (&cx)[4]) {
  return Hole{(float)(cx[0] - cx[1] / 2), (float)(cx[0] + cx[1] / 2), (float)(-cx[2])};
}

// Dynamics (no clip: that is the black-box wrapper's); returns sum(acc^2) of the velocity-controlled envs in the reference's
// dtype.  v is float32 where the caller carries the velocity of a velocity-controlled env with float32 actions as float32
// (it IS the last action); acc64: v holds float64 values (float64 actions, or the zeros of a reset), so acc is float64.
// r_dt = __frcp_rn(c.dt_f), r_dt64 = __drcp_rn(c.dt): computed by the caller, once outside its step loop.
template <int ENV, int N, bool F64, typename V>
__device__ __forceinline__ double reacher_dynamics(const ReacherCfg& c, float r_dt, double r_dt64, double (&q)[N], V (&v)[N],
                                                   const double (&a64)[N], const float (&a32)[N], bool acc64) {
  double acc_cost = 0.0;
  if constexpr (ENV == FG_ENV_HOLE_REACHER || ENV == FG_ENV_VIAPOINT_REACHER) {
    // base_reacher_direct.py:25-27
    if (acc64) {
#pragma unroll
      for (int i = 0; i < N; ++i) {
        const double ac = div_by64(a64[i] - (double)v[i], c.dt, r_dt64);
        acc_cost += ac * ac;
      }
    } else {                        // float32 action and float32 velocity
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
      if constexpr (std::is_same<V, float>::value) v[i] = a32[i]; else v[i] = a64[i];
      q[i] += F64 ? __dmul_rn(c.dt, a64[i]) : (double)__fmul_rn(c.dt_f, a32[i]);   // dt * v: float32 for a float32 v
    }
  } else if constexpr (ENV == FG_ENV_SIMPLE_REACHER) {
    // base_reacher_torque.py:25-26
#pragma unroll
    for (int i = 0; i < N; ++i) {
      v[i] += F64 ? __dmul_rn(c.dt, a64[i]) : (double)__fmul_rn(c.dt_f, a32[i]);
      q[i] += __dmul_rn(c.dt, v[i]);
    }
  }
  return acc_cost;
}

// np.sum(a ** 2) in the action's dtype: a float32 sum for a float32 action
template <int N, bool F64>
__device__ __forceinline__ typename std::conditional<F64, double, float>::type action_sq_sum(const double (&a64)[N],
                                                                                           const float (&a32)[N]) {
  if constexpr (F64) {
    double s = 0.0;
#pragma unroll
    for (int i = 0; i < N; ++i) s += a64[i] * a64[i];
    return s;
  } else {
    float s32 = 0.f;
#pragma unroll
    for (int i = 0; i < N; ++i) s32 = __fadd_rn(s32, __fmul_rn(a32[i], a32[i]));
    return s32;
  }
}

struct StepReward {
  double reward;
  double aux;           // deferred: the partial term collided_reward() completes
  bool collided, success;
  bool deferred;        // the step collided and its reward needs the float64 end effector: collided_reward()
  double info0, info1;  // SimpleReacher: reward_dist, reward_ctrl
};

// Collision tests and reward of the step that has just moved the arm to q (th: absolute link angles).  ee(ex, ey) yields the
// float64 end effector (base_reacher.py:95-103); it is asked for on the steps whose reward reports it.  latch_get / latch_put
// read and write the end effector latched by HoleReacher's rew_fct "unbounded".
template <int ENV, int N, bool F64, typename EE, typename LG, typename LP>
__device__ __forceinline__ StepReward reacher_reward(const ReacherCfg& c, const double (&q)[N], const double (&th)[N],
                                                     const double (&a64)[N], const float (&a32)[N], double acc_cost, int steps,
                                                     const double (&cx)[4], const Hole& hole, const float* s_m, EE ee,
                                                     LG latch_get, LP latch_put) {
  StepReward r{0.0, 0.0, false, false, false, 0.0, 0.0};
  if constexpr (ENV == FG_ENV_HOLE_REACHER) {
    float cs[N], sn[N];
#pragma unroll
    for (int i = 0; i < N; ++i) sincos_reduced(th[i], sn[i], cs[i]);
    bool selfc = false, wallc = false;
    if (!c.allow_self) selfc = self_collision<N>(q, th, cs, sn);                  // base_reacher.py:105-119
    if (!c.allow_wall) wallc = wall_collision<N>(s_m, cs, sn, hole, c.wall_mode);  // hole_reacher.py:148-179
    r.collided = selfc | wallc;
    if (c.rew_fct == 0) {
      // hr_simple_reward.py:35-53
      // ordinary steps: (-0.0 + x) + -0.0 == x for x = acc_cost * -5e-8 <= 0, so only the product is formed
      r.reward = __dmul_rn(acc_cost, -5e-8);
      if (r.collided) {           // the distance term: collided_reward()
        r.deferred = true;
        r.aux = r.reward;
        r.reward = 0.0;
      } else if (steps == 199) {
        double ex, ey;
        ee(ex, ey);
        const double dx = ex - cx[0], dy = ey - (-cx[2]);
        const double dist = sqrt(dx * dx + dy * dy);
        const double dist_cost = dist * dist;
        r.success = dist < 0.005;
        r.reward = __dadd_rn(__dadd_rn(__dmul_rn(dist_cost, -1.0), r.reward), __dmul_rn(0.0, -c.penalty));
      }
    } else if (c.rew_fct == 1) {
      // hr_dist_vel_acc_reward.py:20-60: distance / collision terms only on step 199 (a collision ends the episode, so
      // the latched flag and collision_dist are this step's); factors (-1, -1e-4, -1e-6, -penalty, 0)
      double dist_cost = 0.0, coll_cost = 0.0;
      if (steps == 199) {
        double ex, ey;
        ee(ex, ey);
        const double dx = ex - cx[0], dy = ey - (-cx[2]);
        const double dist = sqrt(dx * dx + dy * dy);
        dist_cost = dist * dist;
        coll_cost = r.collided ? dist * dist : 0.0;
        r.success = (dist < 0.005) && !r.collided;
      }
      const double vel_cost = (double)action_sq_sum<N, F64>(a64, a32);
      r.reward = __dadd_rn(__dadd_rn(__dadd_rn(__dmul_rn(dist_cost, -1.0), __dmul_rn(vel_cost, -1e-4)),
                                     __dmul_rn(acc_cost, -1e-6)), __dmul_rn(coll_cost, -c.penalty));
    } else {
      // hr_unbounded_reward.py:17-60: end effector latched at step 180 (or on collision); factors (1, -5e-6)
      if (r.collided) {           // latch + distance reward: collided_reward()
        r.deferred = true;
        r.aux = acc_cost;
      } else {
        double dist_reward = 0.0;
        if (steps == 180 || steps == 199) {
          double ex, ey;
          ee(ex, ey);
          if (steps == 180) {
            latch_put(ex, ey);
          }
          if (steps == 199) {
            double ee180x, ee180y;
            latch_get(ee180x, ee180y);
            const double dx = ee180x - cx[0], dy = ee180y - (-cx[2]);
            const double dist = sqrt(dx * dx + dy * dy);
            if (ey > 0) dist_reward = exp(-dist);
            else dist_reward = 1 - ee180y;
            r.success = true;
          }
        }
        r.reward = __dadd_rn(dist_reward, __dmul_rn(acc_cost, -5e-6));
      }
    }
  } else if constexpr (ENV == FG_ENV_VIAPOINT_REACHER) {
    // viapoint_reacher.py:79-107 (App. A.6-Q1/Q2: -inf start, `acc` is the action)
    if (!c.allow_self) {
      r.collided = joint_limits<N>(q);
      if (may_self_intersect<N>(q)) {      // (the link directions are only needed for the pair tests)
        float cs[N], sn[N];
#pragma unroll
        for (int i = 0; i < N; ++i) sincos_reduced(th[i], sn[i], cs[i]);
        r.collided |= links_intersect<N>(th, cs, sn);
      }
    }
    double act_term;
    if constexpr (F64) {
      act_term = 5e-8 * action_sq_sum<N, F64>(a64, a32);
    } else {   // float32 action: np.sum(acc**2) is float32 and 5e-8 * float32 stays float32
      act_term = (double)__fmul_rn(5e-8f, action_sq_sum<N, F64>(a64, a32));
    }
    if (!r.collided) {
      double dist = INFINITY;
      r.reward = -INFINITY;
      if (steps == 100 || steps == 199) {
        double ex, ey;
        ee(ex, ey);
        const double tx = (steps == 100) ? cx[0] : cx[2], ty = (steps == 100) ? cx[1] : cx[3];
        dist = sqrt((ex - tx) * (ex - tx) + (ey - ty) * (ey - ty));
      }
      r.success = dist < 0.005;
      r.reward -= dist * dist;
      r.reward -= act_term;
    } else {                    // -penalty - dist^2 - act_term: collided_reward()
      r.deferred = true;
      r.aux = act_term;
    }
  } else if constexpr (ENV == FG_ENV_SIMPLE_REACHER) {
    // simple_reacher.py:56-70 (collision flag is computed but unused)
    double rdist = 0.0;
    if (steps >= 199) {
      double ex, ey;
      ee(ex, ey);
      rdist = -sqrt((ex - cx[0]) * (ex - cx[0]) + (ey - cx[1]) * (ey - cx[1]));
    }
    const auto s = action_sq_sum<N, F64>(a64, a32);
    const double rctrl = (double)s;
    if constexpr (F64) {
      r.reward = rdist - rctrl;
    } else {   // float32 action: reward_ctrl float32; `0 - float32` stays float32 before steps>=199
      r.reward = (steps >= 199) ? rdist - rctrl : (double)(0.f - s);
    }
    r.info0 = rdist;
    r.info1 = rctrl;
  }
  return r;
}

// The reward of a step whose reacher_reward() was deferred, given the float64 end effector of that step.
template <int ENV, typename LP>
__device__ __forceinline__ double collided_reward(const ReacherCfg& c, const double (&cx)[4], double aux, double ex, double ey,
                                                  LP latch_put) {
  double reward = 0.0;
  if constexpr (ENV == FG_ENV_HOLE_REACHER) {
    if (c.rew_fct == 0) {          // hr_simple_reward.py:35-53 with collision_cost = 1
      const double dx = ex - cx[0], dy = ey - (-cx[2]);
      const double dist = sqrt(dx * dx + dy * dy);
      reward = __dadd_rn(__dadd_rn(__dmul_rn(dist * dist, -1.0), aux), __dmul_rn(1.0, -c.penalty));
    } else {                       // hr_unbounded_reward.py: the end effector is latched on the collision
      latch_put(ex, ey);
      const double dx = ex - cx[0], dy = ey - (-cx[2]);
      const double dist = sqrt(dx * dx + dy * dy);
      reward = __dadd_rn(0.25 * exp(-dist), __dmul_rn(aux, -5e-6));
    }
  } else if constexpr (ENV == FG_ENV_VIAPOINT_REACHER) {      // viapoint_reacher.py:96-101
    const double dist = sqrt((ex - cx[2]) * (ex - cx[2]) + (ey - cx[3]) * (ey - cx[3]));
    reward = -c.penalty;
    reward -= dist * dist;
    reward -= aux;
  }
  return reward;
}

// the env-specific part of _get_obs (float64, cast to float32) behind cos(q), sin(q), v; returns its width
__device__ __forceinline__ int obs_tail(int env, const double (&cx)[4], double ex, double ey, float* ob) {
  int no = 0;
  if (env == FG_ENV_HOLE_REACHER) {                   // hole_reacher.py:114-124
    ob[no++] = (float)cx[1];
    ob[no++] = (float)(ex - cx[0]);
    ob[no++] = (float)(ey - (-cx[2]));
  } else if (env == FG_ENV_VIAPOINT_REACHER) {        // viapoint_reacher.py:112-121
    ob[no++] = (float)(ex - cx[0]);
    ob[no++] = (float)(ey - cx[1]);
    ob[no++] = (float)(ex - cx[2]);
    ob[no++] = (float)(ey - cx[3]);
  } else {                                            // simple_reacher.py:75-83
    ob[no++] = (float)(ex - cx[0]);
    ob[no++] = (float)(ey - cx[1]);
  }
  return no;
}

// the step observation of a reacher (float64 trig, cast to float32 like _get_obs) given the end effector; returns its width
template <int ENV, int N, typename V>
__device__ __forceinline__ int reacher_obs(float* ob, const double (&q)[N], const V (&v)[N], const double (&cx)[4], double ex,
                                           double ey, int steps) {
#pragma unroll
  for (int i = 0; i < N; ++i) ob[i] = (float)cos(q[i]);
#pragma unroll
  for (int i = 0; i < N; ++i) ob[N + i] = (float)sin(q[i]);
#pragma unroll
  for (int i = 0; i < N; ++i) ob[2 * N + i] = (float)v[i];
  int no = 3 * N;
  no += obs_tail(ENV, cx, ex, ey, ob + no);
  ob[no++] = (float)steps;
  return no;
}

}  // namespace fg
