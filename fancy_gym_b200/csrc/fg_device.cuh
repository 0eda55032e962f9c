// Device-side building blocks of the fused movement-primitive rollout (sm_100a).
//
// One CUDA thread owns one environment for a whole plan segment: MP weights, joint state and
// the running return live in registers, the (shared) basis tables live in shared memory, and
// nothing per-step goes to HBM.  Arithmetic follows the reference's *mixed* precision
// (SURVEY.md App. A.6-Q7): the MP contraction and the finite-difference velocity are float32
// (FMA chain in index order == oracle/mp.py mode 'mirror'), joint angles are integrated in
// float64 from float32 increments exactly like base_reacher_direct.py:25-27, collision geometry
// is float32 built from float64-reduced angles, and everything that is *reported* (distance
// terms of the reward, end effector, observation) is recomputed in float64 on the few steps
// where the reference reports it.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <cmath>

#include "fancy_gym_b200.h"

namespace fg {

constexpr double kPi = 3.141592653589793115997963468544185161590576171875;   // numpy.pi
constexpr int kLinePoints = 100;                                             // hole_reacher.py:149

// The settings of one reacher env step (fg_reacher.cuh), filled from fg_config or fg_env_step_cfg.
struct ReacherCfg {
  double dt;        // python float 0.01
  float dt_f;       // float32(0.01): numpy's weak-scalar promotion when the action is float32
  int max_steps;    // <= 0: never truncates (fg_env_step)
  int allow_self, allow_wall, rew_fct, wall_mode;
  double penalty;
};

// Kernel-side copy of fg_config (passed by value as a __grid_constant__ kernel parameter).
struct DevCfg {
  int n_dof, T, K;
  ReacherCfg env;
  float act_lim;    // action-space bound as float32 (2*pi or 1000)
  double p[FG_MAX_DOF], d[FG_MAX_DOF];
  float tau, alpha, beta, wscale, gscale;
  int rel_goal, time_aware, ctrl;
  int n_obs_out, n_obs_full;
  int obs_index[FG_MAX_OBS];
  const float* tab_a;   // device
  const float* tab_b;   // device
  int cols_a, rows_b, cols_b;
  const float4* quad_rec;   // device: the tables re-packed per quad of time points for fg_trajgen (fg_trajgen.cuh), or null
  int quad_rec4;            // float4 per record
};

// Normalised RBFs at a LINEAR phase p: the functions of neighbouring centres differ by a ratio that is itself (almost) a
// geometric sequence,
//   phi_{k+1} = phi_k * r_k,   r_0 = exp(B_0 p + C_0) (1 + A_0 p^2),   r_{k+1} = r_k * q_k * (1 + (dA_k p + dB_k) p)
// (A, B, C: the coefficients of a_{k+1}(p) - a_k(p), a_k = -bw_k (p - c_k)^2 / 2; A, dA, dB ~ 1e-14: the centres are a float64
// linspace and every function has the bandwidth of its own spacing) — two exp() per time point instead of one per function.
// The float64 values differ from the direct evaluation's by a few hundred ulps at most; what the MP uses are the values
// ROUNDED TO FLOAT32, and the kernels fall back to the direct evaluation whenever a value sits within 2^12 float64 ulps of a
// float32 rounding boundary (8e-5 of the time points), so the float32 tables are bit-identical.
constexpr int kMaxRbfRec = 16;
struct RbfRec {
  int on;                     // 0: not applicable, every function is evaluated directly
  double a0, b0, c0;
  double q[kMaxRbfRec], da[kMaxRbfRec], db[kMaxRbfRec];
};

// host: the constants for n functions with centres cen[] and bandwidths bw[] (long double arithmetic)
inline void rbf_recurrence(RbfRec& r, const double* cen, const double* bw, int n, int phase_kind) {
  r.on = 0;
  if (phase_kind != 0 || n < 3 || n > kMaxRbfRec) return;
  long double A[kMaxRbfRec], B[kMaxRbfRec], C[kMaxRbfRec];
  for (int k = 0; k + 1 < n; ++k) {
    const long double b0 = bw[k], b1 = bw[k + 1], c0 = cen[k], c1 = cen[k + 1];
    A[k] = -(b1 - b0) / 2;
    B[k] = b1 * c1 - b0 * c0;
    C[k] = -(b1 * c1 * c1 - b0 * c0 * c0) / 2;
  }
  // every exponent stays far inside the range of exp() for a phase in [0, 1] (no function under- or overflows)
  for (int k = 0; k < n; ++k)
    for (int e = 0; e <= 1; ++e) {
      const long double d = (long double)e - cen[k];
      if (!(d * d * bw[k] / 2 <= 600.0L)) return;
    }
  auto absl = [](long double x) { return x < 0 ? -x : x; };
  if (!(absl(A[0]) <= 1e-9L) || !(absl(B[0]) + absl(C[0]) <= 600.0L)) return;
  for (int k = 0; k + 2 < n; ++k) {
    const long double dA = A[k + 1] - A[k], dB = B[k + 1] - B[k], dC = C[k + 1] - C[k];
    if (!(absl(dA) + absl(dB) <= 1e-9L) || !(absl(dC) <= 600.0L)) return;
    r.q[k] = (double)expl(dC);
    r.da[k] = (double)dA;
    r.db[k] = (double)dB;
  }
  r.a0 = (double)A[0];
  r.b0 = (double)B[0];
  r.c0 = (double)C[0];
  r.on = 1;
}

// phi[0 .. NT) by the recurrence (phi[0] exactly as the direct evaluation), normalised like the direct evaluation; returns
// true if one of the values phi[first .. NT) sits too close to a float32 rounding boundary (or is tiny): evaluate directly
template <int NT>
__device__ __forceinline__ bool rbf_recurrence_eval(const RbfRec& rc, const double* __restrict__ cen, const double* __restrict__ bw,
                                                    double ph, int first, double (&phi)[NT]) {
  const double d0 = ph - cen[0];
  phi[0] = exp(-((d0 * d0 * bw[0]) / 2));
  double r = exp(fma(rc.b0, ph, rc.c0));
  r = fma(r, rc.a0 * ph * ph, r);
  double sum = phi[0];
#pragma unroll
  for (int k = 0; k + 1 < NT; ++k) {
    phi[k + 1] = phi[k] * r;
    sum += phi[k + 1];
    if (k + 2 < NT) {
      const double rq = r * rc.q[k];
      r = fma(rq, fma(rc.da[k], ph, rc.db[k]) * ph, rq);
    }
  }
  const double rr = 1.0 / sum;
  bool tie = false;
#pragma unroll
  for (int k = 0; k < NT; ++k) {
    const double qq = phi[k] * rr;
    phi[k] = fma(fma(-qq, sum, phi[k]), rr, qq);
    if (k >= first) {
      // float32 keeps 23 of the 52 mantissa bits: round-to-nearest flips where the 29 dropped bits cross 2^28
      const unsigned dropped = (unsigned)__double2loint(phi[k]) & 0x1FFFFFFFu;
      tie |= (dropped - (0x10000000u - 4096u)) < 8192u;
      tie |= !(phi[k] > 1e-30);                      // (no float32 denormals / NaN on this path)
    }
  }
  return tie;
}

// Per-env phase evaluated INSIDE the fused rollout (learned tau / delay: fg_rollout_io.phase): constants of the phase / basis
// generators and the per-env inputs.  Passed by value next to DevCfg; n_total == 0: not used.
constexpr int kMaxRbfFused = 8;
struct PhaseConst {
  int n_total, first, phase_kind, exp_right_clip;
  double alpha_phase, basis_scale;
  double cen[kMaxRbfFused], bw[kMaxRbfFused];
  const float* tau;           // [B]
  const float* delay;         // [B]
  const float* times;         // [T] float32 time grid of the plan
  const int* n_steps_env;     // ragged plans: per-env number of points, or null
  const float* times_table;   // ragged plans: one grid row per possible length
  int times_stride;
  RbfRec rec;                 // linear phase: two exp() per time point instead of one per RBF (rbf_recurrence())
};

// ---- quad records of the closed-form trajectory kernel (packed on the host in fg_create) -------------------------
//   ProMP : 5 table rows (t0 .. t0+4; the 5th feeds the finite difference of row t0+3), 4 time increments, 4 reciprocals
//   ProDMP: 4 position rows, 4 velocity rows
// padded to an ODD number of float4 so that the lanes of a quarter warp, which read consecutive records, hit distinct
// shared-memory bank groups.
__host__ __device__ constexpr int traj_r4(int kw) { return (kw + 3) / 4; }
__host__ __device__ constexpr int traj_rec4(int mp, int kw) {
  return ((mp == FG_MP_PROMP) ? 5 * traj_r4(kw) + 2 : 8 * traj_r4(kw)) | 1;
}

// ------------------------------------------------------------------------------------------
// trigonometry: argument reduction in float64 (keeps *relative* accuracy of sin near multiples
// of pi, where the y<0 wall predicate and the collinear-arm orientation tests live), polynomial
// in float32.
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ void sincos_reduced(double th, float& s, float& c) {
  // k = nearest integer to th * 2/pi by the 1.5 * 2^52 shift: one DFMA + one DADD, and the quadrant is the low word of the
  // shifted sum (|k| < 2^31) — instead of DMUL + FRND.F64 + F2I.F64 (the two conversions run on the slow conversion path)
  constexpr double kShift = 6755399441055744.0;
  const double shifted = fma(th, 0.63661977236758138243, kShift);    // 2/pi
  const double kd = shifted - kShift;
  double r = fma(-kd, 1.57079632679489655800e+00, th);               // pi/2 hi
  r = fma(-kd, 6.12323399573676603587e-17, r);                       // pi/2 lo
  const float x = (float)r, x2 = x * x;                              // |x| <= pi/4
  float sp = fmaf(x2, -1.9515295891e-4f, 8.3321608736e-3f);
  sp = fmaf(sp, x2, -1.6666654611e-1f);
  sp = fmaf(sp * x2, x, x);
  float cp = fmaf(x2, 2.443315711809948e-5f, -1.388731625493765e-3f);
  cp = fmaf(cp, x2, 4.166664568298827e-2f);
  cp = fmaf(cp, x2, -0.5f);
  cp = fmaf(cp, x2, 1.0f);
  const int q = __double2loint(shifted);
  float ss = (q & 1) ? cp : sp;
  float cc = (q & 1) ? sp : cp;
  s = (q & 2) ? -ss : ss;
  c = ((q + 1) & 2) ? -cc : cc;
}

// sin of a *relative* link angle; exactly 0 for 0, relative accuracy ~1e-7 for tiny angles
__device__ __forceinline__ float sin_reduced(double phi) {
  const double kd = rint(phi * 0.31830988618379069122);              // 1/pi
  double r = fma(-kd, 3.14159265358979311600e+00, phi);
  r = fma(-kd, 1.22464679914735317723e-16, r);
  const float x = (float)r, x2 = x * x;                              // |x| <= pi/2
  float p = fmaf(x2, -2.5052108e-8f, 2.7557319e-6f);
  p = fmaf(p, x2, -1.9841270e-4f);
  p = fmaf(p, x2, 8.3333333e-3f);
  p = fmaf(p, x2, -1.6666667e-1f);
  p = fmaf(p * x2, x, x);
  return ((int)kd & 1) ? -p : p;
}

// x / d with a pre-computed r = RN(1/d) (__frcp_rn): one Newton step on the quotient gives the correctly
// rounded IEEE quotient for finite, non-denormal operands (Markstein) in 3 instructions instead of the
// ~13 of the generic division sequence.  The divisors on the hot path (time increments, dt, tau) are
// shared by all envs, so r is computed once per block / thread.
__device__ __forceinline__ float div_by(float x, float d, float r) {
  const float q = __fmul_rn(x, r);
  const float rem = fmaf(-q, d, x);
  return fmaf(rem, r, q);
}
// the same in float64 (r = __drcp_rn(d)): 3 instructions of the FP64 pipe instead of the ~35 of the generic division.  (For
// x = -0.0 it returns +0.0: its only caller squares the quotient.)
__device__ __forceinline__ double div_by64(double x, double d, double r) {
  const double q = __dmul_rn(x, r);
  const double rem = fma(-q, d, x);
  return fma(rem, r, q);
}

// ------------------------------------------------------------------------------------------
// self collision (base_reacher.py:105-119, utils.py:1-9)
// The reference tests ccw(A,B,C) = cross(B-A, C-A) > 1e-12 on joint positions.  With unit links
// every such cross product is a sum of sines of relative link angles:
//   ccw(J_i, J_i+1, J_m)   = sum_{l=i+1}^{m-1} sin(theta_l - theta_i)
//   ccw(J_a, J_j,  J_j+1)  = sum_{l=a}^{j-1}   sin(theta_j - theta_l)
// Evaluating it this way keeps float32 *relative* accuracy for (nearly) collinear links — the arm
// starts straight (q = [q0,0,..,0]) where the position form would be pure rounding noise around
// the 1e-12 threshold.  Exactly collinear links give exactly 0 -> "not ccw", as in the reference.
// ------------------------------------------------------------------------------------------
template <int N, bool ACCURATE>
__device__ __forceinline__ bool self_hits(const double (&th)[N], const float (&cs)[N], const float (&sn)[N],
                                          float& min_abs) {
  float S[N][N];   // S[i][l] = sin(th[l]-th[i]), i<l  (fully unrolled -> registers)
#pragma unroll
  for (int i = 0; i < N; ++i)
#pragma unroll
    for (int l = i + 1; l < N; ++l)
      S[i][l] = ACCURATE ? sin_reduced(th[l] - th[i]) : fmaf(sn[l], cs[i], -__fmul_rn(cs[l], sn[i]));
  bool hit = false;
  const float eps = 1e-12f;
  min_abs = 1e30f;
#pragma unroll
  for (int i = 0; i < N; ++i) {
#pragma unroll
    for (int j = i + 2; j < N; ++j) {
      float c3 = 0.f;                       // ccw(A,B,C): l = i+1 .. j-1
#pragma unroll
      for (int l = i + 1; l <= j - 1; ++l) c3 += S[i][l];
      const float c4 = c3 + S[i][j];        // ccw(A,B,D)
      float c2 = 0.f;                       // ccw(B,C,D): l = i+1 .. j-1
#pragma unroll
      for (int l = j - 1; l >= i + 1; --l) c2 += S[l][j];
      const float c1 = c2 + S[i][j];        // ccw(A,C,D): l = i .. j-1
      hit |= ((c1 > eps) != (c2 > eps)) & ((c3 > eps) != (c4 > eps));
      if (!ACCURATE) min_abs = fminf(fminf(min_abs, fminf(fabsf(c1), fabsf(c2))), fminf(fabsf(c3), fabsf(c4)));
    }
  }
  return hit;
}

// cs / sn: float32 cos / sin of the absolute link angles th (from the forward kinematics).  The orientation
// values are first formed from them (sin(a-b) = sin a cos b - cos a sin b, absolute error < 2e-6 on a sum);
// unless every one of them is farther than 8e-6 from zero — i.e. unless some links are (nearly) collinear —
// the decisions are already those of the accurate evaluation, which is only entered otherwise.
template <int N>
struct Angles {
  double th[N];
};
// the accurate evaluation is rare (nearly collinear links): kept out of the hot loop body, angles passed by value
template <int N>
__device__ __noinline__ bool self_hits_accurate(const Angles<N> a) {
  const float zero[N] = {};
  float unused;
  return self_hits<N, true>(a.th, zero, zero, unused);
}

// max / min that return NaN if either operand is NaN (PTX max.NaN / min.NaN, sm_80+; fmaxf / fminf return the other one):
// one FMNMX each, like fmaxf / fminf, and the same result for every other operand
__device__ __forceinline__ float fmax_nan(float a, float b) {
  float r;
  asm("max.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}
__device__ __forceinline__ float fmin_nan(float a, float b) {
  float r;
  asm("min.NaN.f32 %0, %1, %2;" : "=f"(r) : "f"(a), "f"(b));
  return r;
}

// any(q > pi) or any(q < -pi) (base_reacher.py:111): |q| > pi as an unsigned compare of the sign-stripped bit patterns
// (non-negative doubles order like integers).  Fast screen on the HIGH words only: non-negative float patterns order like the
// integers they are, so the largest sign-stripped high word is one FMNMX chain with |.| modifiers; only when it reaches pi's
// high word (|q| within 2^-20 of pi or beyond: rare) are the full 64-bit patterns compared.  The high word of |q| >= 2^1017
// (inf included) read as a float32 is a NaN: the max keeps it and the screen lets it through.  A NaN joint is not a limit
// (NaN > pi is False): its pattern lies above inf's.
template <int N>
__device__ __forceinline__ bool joint_limits(const double (&q)[N]) {
  bool lim = false;
  constexpr unsigned long long kPiBits = 0x400921FB54442D18ULL, kInfBits = 0x7FF0000000000000ULL;
  float hi_max = 0.f;
#pragma unroll
  for (int i = 0; i < N; ++i) hi_max = fmax_nan(hi_max, fabsf(__int_as_float(__double2hiint(q[i]))));
  if (!(hi_max < __int_as_float(0x400921FB))) {
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const unsigned long long bits = (unsigned long long)__double_as_longlong(q[i]) & 0x7FFFFFFFFFFFFFFFULL;
      lim |= (bits > kPiBits) & (bits <= kInfBits);
    }
  }
  return lim;
}

// Can two non-adjacent links touch at all?  If link i meets link j (j >= i + 2) at a point P, then P, joint i+1, ..., joint j is
// a closed polygon; the exterior angles of a closed polygon sum to at least 2 pi in absolute value and the one at P is below
// pi, so the joints between the two links turn by MORE than pi: sum_{l=i+1..j} |q_l| > pi (the relative joint angles are the
// exterior angles).  Hence, while sum_{l=1..N-1} |q_l| <= 3.0 (< pi, with room for the float32 sum), no pair of links intersects
// and every orientation test of the reference comes out "no hit"; the whole pair evaluation (18 orientation values for 5
// links, ~95 instructions) is skipped.  At sigma = 0.25 (BASELINE config 2) this holds on 99.8 % of the warp-steps.
constexpr float kTurnScreen = 3.0f;
template <int N>
__device__ __forceinline__ bool may_self_intersect(const double (&q)[N]) {
  if constexpr (N < 3) {
    return false;
  } else {
    float turn = 0.f;
#pragma unroll
    for (int i = 1; i < N; ++i) turn += fabsf((float)q[i]);
    return !(turn <= kTurnScreen);        // (a NaN angle takes the full evaluation)
  }
}

// the pair tests themselves: orientation values from the FK sin / cos first; the accurate evaluation only if one of them is
// within 8e-6 of zero (nearly collinear links)
template <int N>
__device__ __forceinline__ bool links_intersect(const double (&th)[N], const float (&cs)[N], const float (&sn)[N]) {
  float min_abs;
  bool hit = self_hits<N, false>(th, cs, sn, min_abs);
  if (min_abs <= 8e-6f) {
    Angles<N> a;
#pragma unroll
    for (int i = 0; i < N; ++i) a.th[i] = th[i];
    hit = self_hits_accurate<N>(a);
  }
  return hit;
}

template <int N>
__device__ __forceinline__ bool self_collision(const double (&q)[N], const double (&th)[N], const float (&cs)[N],
                                               const float (&sn)[N]) {
  bool hit = joint_limits<N>(q);
  if (may_self_intersect<N>(q)) hit |= links_intersect<N>(th, cs, sn);
  return hit;
}

// ------------------------------------------------------------------------------------------
// wall collision (hole_reacher.py:126-179): 100 samples s_m per link,
//   x_m = fma(cos, s_m, X_i), y_m = fma(sin, s_m, Y_i);  collided iff some sample has
//   (x<xl & y<0) | (x>xr & y<0) | (xl<x<xr & y<-depth)   (all strict).
// s_m (float32(linspace(0,1,100))) sits in shared memory.  Both coordinates are monotone in m
// even after rounding (fma is monotone in s), so every predicate holds on a prefix or a suffix
// of the sample index: the exact answer follows from six binary searches instead of 100
// evaluations (wall_mode 0); wall_mode 1 evaluates all samples literally.  Links whose lower
// end point is not below max(0,-depth) cannot collide and are skipped in both modes.
// ------------------------------------------------------------------------------------------
struct Hole {
  float xl, xr, nd;   // left edge, right edge, -depth
};

// number of samples m in [0,100) with f_m < tau (strict) or f_m <= tau, f_m = fma(k, s_m, off);
// `rev` walks the samples backwards so that the walked sequence is non-decreasing.
template <bool LE>
__device__ __forceinline__ int count_below(const float* __restrict__ s_m, float k, float off, float tau, bool rev) {
  int lo = 0, hi = kLinePoints;     // first walked index whose value is NOT below tau
#pragma unroll
  for (int it = 0; it < 7; ++it) {
    const int mid = min((lo + hi) >> 1, kLinePoints - 1);
    const int m = rev ? (kLinePoints - 1 - mid) : mid;
    const float f = fmaf(k, s_m[m], off);
    const bool below = LE ? (f <= tau) : (f < tau);
    const bool active = lo < hi;
    lo = (active && below) ? mid + 1 : lo;
    hi = (active && !below) ? mid : hi;
  }
  return lo;
}

struct Span {
  int lo, hi;   // [lo, hi) in forward sample order
};
__device__ __forceinline__ Span span_below(int n, bool rev) {       // {f < tau}
  return rev ? Span{kLinePoints - n, kLinePoints} : Span{0, n};
}
__device__ __forceinline__ Span span_above(int n_le, bool rev) {    // {f > tau}, n_le = #{f <= tau}
  return rev ? Span{0, kLinePoints - n_le} : Span{n_le, kLinePoints};
}
__device__ __forceinline__ bool overlap(Span a, Span b) { return max(a.lo, b.lo) < min(a.hi, b.hi); }
__device__ __forceinline__ bool overlap3(Span a, Span b, Span c) {
  return max(max(a.lo, b.lo), c.lo) < min(min(a.hi, b.hi), c.hi);
}

// Transition index by ESTIMATE + exact fix-up: the walked sequence g(i) = fma(k, s(i), off) is non-decreasing, so the
// count of samples below tau is the unique i with g(i-1) below and g(i) not below.  Solving the line for tau gives i to
// within a sample; the two fix-up loops then move it until the SAME float32 expressions the literal evaluation uses bracket
// it — whatever the estimate was (k == 0, inf, NaN included: they only cost iterations), the result is the binary search's.
// ~25 instructions instead of ~60; n_le (samples <= tau) continues from n_lt (samples < tau): one more evaluation.
__device__ __forceinline__ float walked(const float* __restrict__ s_m, float k, float off, int i, bool rev) {
  return fmaf(k, s_m[rev ? (kLinePoints - 1 - i) : i], off);
}
__device__ __forceinline__ int count_lt_est(const float* __restrict__ s_m, float k, float r99k, float off, float tau, bool rev) {
  float e = (tau - off) * r99k;                        // sample coordinate where the line crosses tau
  e = rev ? (float)(kLinePoints - 1) - e : e;
  int i = (int)fminf(fmaxf(e, -1.0f), (float)kLinePoints) + 1;      // (fmaxf drops a NaN estimate)
  i = min(max(i, 0), kLinePoints);
  while (i > 0 && !(walked(s_m, k, off, i - 1, rev) < tau)) --i;
  while (i < kLinePoints && walked(s_m, k, off, i, rev) < tau) ++i;
  return i;
}
__device__ __forceinline__ int count_le_from(const float* __restrict__ s_m, float k, float off, float tau, bool rev, int n_lt) {
  int i = n_lt;                                        // samples == tau follow the ones below it
  while (i < kLinePoints && walked(s_m, k, off, i, rev) <= tau) ++i;
  return i;
}

// (out of line: up to N calls per step share ONE copy of the searches — the fused kernel's loop body otherwise exceeds the
//  instruction cache; measured "no_instruction" stalls, profiles/README.md)
static __device__ __noinline__ bool link_wall_search(const float* __restrict__ s_m, float c, float s, float X, float Y, const Hole h) {
  const bool rx = c < 0.f, ry = s < 0.f;
  const float rc = __fdividef((float)(kLinePoints - 1), c), rs = __fdividef((float)(kLinePoints - 1), s);   // estimates only
  const int n_lt_l = count_lt_est(s_m, c, rc, X, h.xl, rx), n_le_l = count_le_from(s_m, c, X, h.xl, rx, n_lt_l);
  const int n_lt_r = count_lt_est(s_m, c, rc, X, h.xr, rx), n_le_r = count_le_from(s_m, c, X, h.xr, rx, n_lt_r);
  const Span A = span_below(n_lt_l, rx);           // x <  xl
  const Span Bx = span_above(n_le_r, rx);          // x >  xr
  const Span Gl = span_above(n_le_l, rx);          // x >  xl
  const Span Lr = span_below(n_lt_r, rx);          // x <  xr
  const Span C = span_below(count_lt_est(s_m, s, rs, Y, 0.f, ry), ry);           // y <  0
  const Span D = span_below(count_lt_est(s_m, s, rs, Y, h.nd, ry), ry);          // y < -depth
  return overlap(A, C) | overlap(Bx, C) | overlap3(Gl, Lr, D);
}

// the round-1 formulation (six 7-step binary searches), kept as wall_mode 3 for A/B runs
static __device__ __noinline__ bool link_wall_bisect(const float* __restrict__ s_m, float c, float s, float X, float Y, const Hole h) {
  const bool rx = c < 0.f, ry = s < 0.f;
  const Span A = span_below(count_below<false>(s_m, c, X, h.xl, rx), rx);          // x <  xl
  const Span Bx = span_above(count_below<true>(s_m, c, X, h.xr, rx), rx);          // x >  xr
  const Span Gl = span_above(count_below<true>(s_m, c, X, h.xl, rx), rx);          // x >  xl
  const Span Lr = span_below(count_below<false>(s_m, c, X, h.xr, rx), rx);         // x <  xr
  const Span C = span_below(count_below<false>(s_m, s, Y, 0.f, ry), ry);           // y <  0
  const Span D = span_below(count_below<false>(s_m, s, Y, h.nd, ry), ry);          // y < -depth
  return overlap(A, C) | overlap(Bx, C) | overlap3(Gl, Lr, D);
}

__device__ __forceinline__ bool wall_sample_hit(float x, float y, const Hole& h) {
  return ((x < h.xl) & (y < 0.f)) | ((x > h.xr) & (y < 0.f)) | ((x > h.xl) & (x < h.xr) & (y < h.nd));
}

static __device__ __noinline__ bool link_wall_brute(const float* __restrict__ s_m, float c, float s, float X, float Y, const Hole h) {
  bool hit = false;
#pragma unroll 4
  for (int m = 0; m < kLinePoints; ++m) {
    const float sm = s_m[m];
    const float x = fmaf(c, sm, X), y = fmaf(s, sm, Y);
    hit |= wall_sample_hit(x, y, h);
  }
  return hit;
}

template <int N>
__device__ __forceinline__ bool wall_collision(const float* __restrict__ s_m, const float (&cs)[N],
                                               const float (&sn)[N], const Hole& h, int wall_mode) {
  bool hit = false;
  const float ythr = fmaxf(0.f, h.nd);
  // ONE test whether any link reaches below the ground line at all (the common case in the sigma = 0.25 regime is
  // "none"): a link's lower end is one of its two joints, so "some link has min(Y_i, Y_i+1) < ythr" is "the lowest joint is
  // below ythr" — the joint heights and one FMNMX chain; the x positions and the per-link tests are only formed behind it
  float Ys[N + 1];
  Ys[0] = 0.f;
#pragma unroll
  for (int i = 0; i < N; ++i) Ys[i + 1] = fmaf(sn[i], 1.0f, Ys[i]);      // sample m=99 (s=1) == next joint
  float ymin = 0.f;
#pragma unroll
  for (int i = 1; i <= N; ++i) ymin = fminf(ymin, Ys[i]);
  if (ymin < ythr || wall_mode == 2) {           // mode 2: no skipping at all
    float X = 0.f;
#pragma unroll
    for (int i = 0; i < N; ++i) {
      const float Xn = fmaf(cs[i], 1.0f, X);
      if (wall_mode == 2 || fminf(Ys[i], Ys[i + 1]) < ythr) {
        if (wall_mode == 0) {
          // The two ends of the link ARE samples (s_0 = 0: (X, Y_i); s_99 = 1: the next joint, the same fma), and every
          // other sample lies between them in both coordinates (monotone in s).  So: an end that collides decides "hit"
          // (the step an episode ends on: the lower end is below the ground next to the hole); both ends strictly inside
          // the hole's column and not below its floor decide "no hit" (an arm reaching into the hole).  Only links that
          // straddle an edge of the hole go through the searches.  (A NaN coordinate fails every comparison: searches.)
          if (!hit) {
            const float y0 = Ys[i], y1 = Ys[i + 1];
            const bool end_hit = wall_sample_hit(X, y0, h) | wall_sample_hit(Xn, y1, h);
            const bool inside = (fminf(X, Xn) > h.xl) & (fmaxf(X, Xn) < h.xr) & (fminf(y0, y1) >= h.nd);
            if (end_hit) hit = true;
            else if (!inside) hit = link_wall_search(s_m, cs[i], sn[i], X, y0, h);
          }
        } else {
          hit |= (wall_mode == 3) ? link_wall_bisect(s_m, cs[i], sn[i], X, Ys[i], h)
                                  : link_wall_brute(s_m, cs[i], sn[i], X, Ys[i], h);
        }
      }
      X = Xn;
    }
  }
  return hit;
}

// float64 forward kinematics of the end effector, for the steps on which the reference *reports*
// a distance / end effector / observation (base_reacher.py:95-103, :137-139)
template <int N>
__device__ __noinline__ double2 end_effector64_ool(const Angles<N> a) {
  double ex = 0.0, ey = 0.0;
#pragma unroll
  for (int i = 0; i < N; ++i) {
    double s, c;
    sincos(a.th[i], &s, &c);
    ex += c;
    ey += s;
  }
  return make_double2(ex, ey);
}
// executed on a handful of steps per episode: one out-of-line copy instead of three inlined double-precision sincos chains
template <int N>
__device__ __forceinline__ void end_effector64(const double (&th)[N], double& ex, double& ey) {
  Angles<N> a;
#pragma unroll
  for (int i = 0; i < N; ++i) a.th[i] = th[i];
  const double2 e = end_effector64_ool<N>(a);
  ex = e.x;
  ey = e.y;
}

}  // namespace fg
