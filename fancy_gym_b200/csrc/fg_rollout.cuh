// Fused black-box rollout kernel (K1-K3 of SURVEY.md §2.1): one thread runs one environment at a time.
//
// Replaces, for B envs at once, the Python loop of BlackBoxWrapper.step
// (fancy_gym/black_box/black_box_wrapper.py:150-217): trajectory evaluation (get_trajectory
// :96-120 -> mp_pytorch), controller (:176-177), np.clip (:178-179), env.step
// (base_reacher_direct.py:20-38 / base_reacher_torque.py:20-37), reward, termination, TimeLimit
// truncation and reward aggregation (:215-216) — and, when the caller hands over the parameters of several plans
// (fg_rollout_io.n_plans), the re-planning loop around it (:197-203): plan after plan inside ONE launch.
//
// Scheduling.  An env's whole state lives in registers while it runs.  Episodes end at different steps (collisions), so a
// block RE-PACKS its live envs whenever that frees a whole warp: every env owns a shared-memory slot, threads park their
// env's state there, the block compacts the list of live slots and threads 0 .. n_live-1 pick the live envs up again —
// warps beyond that stop issuing.  Envs that have stopped wait in their slot; the work that is only done once per episode
// (float64 end effector, the distance term of the reward of the step that collided, the observation, all global stores)
// is done for 32 of them at a time by otherwise idle warps instead of one lane at a time inside the step loop.  Which env a
// thread runs never changes what is computed for that env: results are bit-identical to one-thread-per-env execution
// (tests/test_gpu_digests.py).
#pragma once
#ifdef FG_ROLLOUT_CHECK
#include <cstdio>
#endif
#include "fg_reacher.cuh"

namespace fg {

#ifndef FG_ROLLOUT_THREADS
#define FG_ROLLOUT_THREADS 128
#endif
constexpr int kRolloutThreads = FG_ROLLOUT_THREADS;
constexpr int kRolloutWarps = kRolloutThreads / 32;

__host__ __device__ constexpr int pad4(int n) { return (n + 3) & ~3; }

// per-dof weight slots: ProMP K, DMP K + goal, ProDMP [y_b, tau*dy_b, w_0..w_K-1, g]
__host__ __device__ constexpr int weight_slots(int mp, int K) {
  return mp == FG_MP_PROMP ? K : mp == FG_MP_DMP ? K + 1 : mp == FG_MP_PRODMP ? K + 3 : 0;
}

// ---- an env's parked state: 32-bit words of one shared-memory slot (word-major: word w of slot s sits at [w * BD + s]) ----
template <int ENV, int MP, bool MOTOR, int N, int KC>
struct SlotLayout {
  // In the velocity-controlled envs with a float32 action (velocity / position controller) the joint velocity IS the last
  // float32 action (or the zeros of reset), so it is carried as float32; PD-controlled / torque envs keep the float64 value.
  static constexpr bool VF = !MOTOR && (ENV == FG_ENV_HOLE_REACHER || ENV == FG_ENV_VIAPOINT_REACHER);
  // The register-resident-weights instantiation (KC > 0) is dispatched for velocity / motor control only (position control
  // takes the run-time-K variant, fg_rollout_launch.cuh): without a motor law the action IS the desired velocity, so the
  // desired position is dead weight in the loop — no copies of it, no select per joint, for ProDMP no position contraction.
  static constexpr bool VEL_ONLY = (KC > 0) && !MOTOR;
  static constexpr bool CARRY = (MP == FG_MP_PROMP || MP == FG_MP_DMP);   // ProMP: pos[t+1], vel; DMP: integrator state
  // desired position / velocity of the last executed step (condition_on_desired): carried unless it can be re-evaluated
  static constexpr bool LASTDES = !(VEL_ONLY && (MP == FG_MP_PROMP || MP == FG_MP_PRODMP));
  static constexpr int W_Q = 0;
  static constexpr int W_V = W_Q + 2 * N;
  static constexpr int W_CARRY = W_V + (VF ? N : 2 * N);
  static constexpr int W_LAST = W_CARRY + (CARRY ? 2 * N : 0);
  static constexpr int W_INFO = W_LAST + (LASTDES ? 2 * N : 0);
  // 2 doubles: SimpleReacher reward_dist / reward_ctrl of the last step; HoleReacher: the end effector latched by rew_fct "unbounded"
  static constexpr bool INFO = (ENV == FG_ENV_SIMPLE_REACHER || ENV == FG_ENV_HOLE_REACHER);
  static constexpr int W_SCAL = W_INFO + (INFO ? 4 : 0);
  // env index within the block, episode step, plan, current / end / last table row of the plan, status + result bits
  enum { S_B = 0, S_STEPS, S_K, S_TR, S_TREND, S_TRLAST, S_FLAGS, S_RET, S_AUX = S_RET + 2, S_COUNT = S_AUX + 2 };
  static constexpr int WORDS = W_SCAL + S_COUNT;
};

// status (bits 0-1 of the flags word) and result bits of a slot
constexpr unsigned kSlotEmpty = 0u, kSlotLive = 1u, kSlotPending = 2u, kSlotStatusMask = 3u;
constexpr unsigned kSlotTerminated = 4u, kSlotTruncated = 8u, kSlotSuccess = 16u, kSlotCollided = 32u, kSlotDeferred = 64u;

// shared memory layout (32-bit words); what the step loop touches sits at compile-time addresses:
//   [control words: want, n_live, warps that run, queue dry, queue base, -, -, -, per-warp live / pending counts] [live list | pending list: 2 * BD uint16]
//   [s_m 100 (+4)] [tab_a rows * pad4(cols_a)] [tab_b rows_b * pad4(cols_b)] [1/tab_b pad4(rows_b)]
//   [w  slots * n_dof * BD] [slot state  WORDS * BD]
constexpr int kCtlWords = (8 + 2 * kRolloutWarps + 15) & ~15;
constexpr int kListWords = kRolloutThreads;            // 2 * BD uint16
constexpr int kSmWords = (kLinePoints + 3) & ~3;
constexpr int kFixedWords = kCtlWords + kListWords + kSmWords;
__host__ __device__ inline size_t rollout_smem_bytes(int T, int cols_a, int rows_b, int cols_b, int w_per_thread, int slot_words,
                                                     int threads) {
  const size_t words = kFixedWords + (size_t)T * pad4(cols_a) + (size_t)rows_b * pad4(cols_b) + pad4(rows_b) +
                       (size_t)w_per_thread * threads + (size_t)slot_words * threads;
#ifdef FG_ROLLOUT_CHECK
  return (words + 3 * (size_t)threads) * sizeof(float);
#endif
  return words * sizeof(float);
}

// KC > 0: the number of weighted basis functions is a compile-time constant (the registry default 5): the per-env
//         weights live in REGISTERS and the (float4-padded) table rows are fetched with vector broadcast loads.
// KC == 0: run-time K; weights stay in shared memory (k-major, slot-minor: conflict free).
// DBG: the verbose>=2 variant that also writes the per-step actions / observations / rewards (black_box_wrapper.py:208-213).
#ifndef FG_ROLLOUT_MINB
#define FG_ROLLOUT_MINB 4   // <= 128 registers: 4 blocks of 128 threads per SM (65 536 envs need 443 resident threads per SM)
#endif
// NTX > 0: per-env phase (learned tau / delay): the basis row of every step is evaluated in the thread from the env's own tau /
//          delay (NTX RBFs in total, the last KC of them weighted) instead of read from the shared tables — the arithmetic of
//          k_trajgen_phase_warp + k_dmp_integrate_phase (fg_trajgen_phase.cu), without the 8 KB / env round trip through HBM.
template <int ENV, int MP, bool MOTOR, int N, int KC, bool DBG, int NTX = 0>
__global__ void __launch_bounds__(kRolloutThreads, FG_ROLLOUT_MINB)
k_rollout(const __grid_constant__ DevCfg c, const __grid_constant__ fg_rollout_io io, const long long B,
          const int seg_steps, unsigned* __restrict__ queue, const int warps_lo, const int blocks_extra,
          const __grid_constant__ PhaseConst pc) {
  static_assert(NTX == 0 || ((MP == FG_MP_PROMP || MP == FG_MP_DMP) && KC > 0 && NTX >= KC && NTX <= kMaxRbfFused),
                "per-env phase: ProMP / DMP with register-resident weights");
  using SL = SlotLayout<ENV, MP, MOTOR, N, KC>;
  constexpr bool VF = SL::VF, VEL_ONLY = SL::VEL_ONLY;
  extern __shared__ __align__(16) float smem[];
  const int RT = c.T;                          // rows of the staged tables (all plans of the launch, one after the other)
  const int K = (KC > 0) ? KC : c.K;
  const int CA = (KC > 0) ? weight_slots(MP, KC) : c.cols_a;   // table columns == weight slots per dof
  const int RA = pad4(CA), RB = pad4(c.cols_b);
  constexpr int BD = kRolloutThreads;
  volatile int* ctl = reinterpret_cast<volatile int*>(smem);                     // [0] want, [1] n_live, [2] warps bound
  int* wcount = reinterpret_cast<int*>(smem) + 8;                                // [warps] live | [warps] pending
  unsigned short* live_list = reinterpret_cast<unsigned short*>(smem + kCtlWords);
  unsigned short* pend_list = live_list + BD;
  float* s_m = smem + kCtlWords + kListWords;
  float* tabA = smem + kFixedWords;
  float* tabB = tabA + RT * RA;
  float* tabR = tabB + c.rows_b * RB;          // ProMP: reciprocals of the time increments
  float* wsm = tabR + pad4(c.rows_b);
  constexpr bool HAS_W = (MP != FG_MP_TRAJ);
  const int WS = weight_slots(MP, K);                     // slots per dof
  unsigned* sst = reinterpret_cast<unsigned*>(wsm + (HAS_W ? WS * N * BD : 0));
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  // The step loop polls control word 0 once per step.  Through the generic pointer every poll re-derives the shared window
  // (S2UR SR_CgaCtaId + ULEA: ~6 % of the kernel's stall samples); the 32-bit shared address is formed once instead.
  const unsigned ctl_saddr = (unsigned)__cvta_generic_to_shared(smem);
  auto want_repack = [&]() -> int {
    int v_;
    asm volatile("ld.volatile.shared.s32 %0, [%1];" : "=r"(v_) : "r"(ctl_saddr) : "memory");
    return v_;
  };

#ifdef FG_ROLLOUT_CHAOS
  // test build: random per-lane / per-warp delays at every scheduling point (tools/race_probe.py, profiles/README.md "Sanitizer")
  unsigned chaos_state = (unsigned)clock64() * 2654435761u + (blockIdx.x * BD + tid) * 40503u + 12345u;
  auto chaos = [&](unsigned one_in, unsigned max_ns) {
    chaos_state = chaos_state * 1664525u + 1013904223u;
    if (((chaos_state >> 16) % one_in) == 0) __nanosleep((chaos_state >> 8) % max_ns);
  };
#define FG_CHAOS(a, b) chaos(a, b)
#else
#define FG_CHAOS(a, b)
#endif

  // ---- stage the shared tables (coalesced reads, rows zero-padded to float4) ----
  for (int i = tid; i < RT * RA; i += BD) {
    const int r = i / max(RA, 1), col = i - r * RA;
    tabA[i] = (col < c.cols_a) ? c.tab_a[r * c.cols_a + col] : 0.f;
  }
  for (int i = tid; i < c.rows_b * RB; i += BD) {
    const int r = i / max(RB, 1), col = i - r * RB;
    tabB[i] = (col < c.cols_b) ? c.tab_b[r * c.cols_b + col] : 0.f;
  }
  if constexpr (MP == FG_MP_PROMP)
    for (int i = tid; i < c.rows_b; i += BD) tabR[i] = __frcp_rn(c.tab_b[i]);
  stage_line_points<BD>(s_m);

  // Envs per block: `warps_lo` warps, one more in the first `blocks_extra` blocks (the launcher uses full blocks: 4 / 0).
  const int bi = (int)blockIdx.x;
  const long long b0 = 32LL * ((long long)warps_lo * bi + min(bi, blocks_extra));
  const int n_here = 32 * (warps_lo + (bi < blocks_extra ? 1 : 0));
  const int n_plans = io.n_plans > 1 ? io.n_plans : 1;
  // io.plan_T: points of ONE plan (the "last point" rules of ProMP / DMP); == c.T unless several plans share the tables

  // ---- stage this block's MP parameters of the first plan: coalesced read of [BD, P], stored slot-major ----
  const int KP = (MP == FG_MP_PROMP) ? K : K + 1;         // params per dof
  const int P = N * KP;
  const long long PS = (long long)n_plans * P;            // params of one env: [n_plans, P]
  auto put_param = [&](int slot, int idx, float val) {
    const int d = idx / KP, k = idx % KP;
    if constexpr (MP == FG_MP_DMP) val = __fmul_rn(val, (k < K) ? c.wscale : c.gscale);
    wsm[(d * WS + ((MP == FG_MP_PRODMP) ? k + 2 : k)) * BD + slot] = val;
  };
  if constexpr (HAS_W) {
    const long long nblk = max(0LL, min((long long)n_here, B - b0));
    for (long long f = tid; f < nblk * P; f += BD) {
      const int th = (int)(f / P), idx = (int)(f % P);
      put_param(th, idx, io.params[(b0 + th) * PS + idx]);
    }
  }
  if (tid == 0) {
    ctl[0] = 0;
    ctl[1] = 0;
    ctl[2] = 0;
    ctl[3] = 0;        // work queue exhausted
  }
  __syncthreads();

  // ---- registers of the env this thread currently runs -------------------------------------------------------------
  int own = tid;                  // its slot (also where its weights sit in wsm)
  long long b = b0 + tid;
  double q[N], v[N];
  float vf[N];
  int steps = 0, k = 0;
  int tr = 0, tr_end = 0, tr_last = 0;   // table row of the current step, of the end of this plan's segment, of the plan's last point
  unsigned fl = kSlotEmpty;
  double ret = 0.0;
  double info0 = 0, info1 = 0;
  float carry_a[N], carry_b[N];     // ProMP: pos[t+1], vel[t]; DMP: y, scaled-time velocity
  float pos[N], vel[N];             // desired position / velocity of the current step
  Hole hole{};
  double cx[4] = {0, 0, 0, 0};
  // rew_fct "unbounded": the end effector latched at step 180 (hr_unbounded_reward.py:35-36) lives in the env's slot, not in
  // registers (it is touched on two steps of an episode)
  auto latch_put = [&](double x, double y) {
    unsigned* z = sst + SL::W_INFO * BD + own;
    z[0] = (unsigned)__double2loint(x); z[BD] = (unsigned)__double2hiint(x);
    z[2 * BD] = (unsigned)__double2loint(y); z[3 * BD] = (unsigned)__double2hiint(y);
  };
  auto latch_get = [&](double& x, double& y) {
    const unsigned* z = sst + SL::W_INFO * BD + own;
    x = __hiloint2double((int)z[BD], (int)z[0]);
    y = __hiloint2double((int)z[3 * BD], (int)z[2 * BD]);
  };

  // ---- per-env weights: registers (KC > 0) or shared memory (KC == 0) ----
  constexpr int WSC = (KC > 0) ? weight_slots(MP, KC) : 1;
  constexpr int RAC = pad4(WSC) > 0 ? pad4(WSC) : 4;
  float wreg[N][(KC > 0 && HAS_W) ? WSC : 1];
#define WSM(d, k_) wsm[((d) * WS + (k_)) * BD + own]
  auto fetch_weights = [&]() {
    if constexpr (KC > 0 && HAS_W) {
#pragma unroll
      for (int d = 0; d < N; ++d)
#pragma unroll
        for (int kk = 0; kk < WSC; ++kk) wreg[d][kk] = WSM(d, kk);
    }
  };
  // dot(table row, weights of dof d): FMA chain in index order, accumulator starts at 0 (oracle 'mirror' mode)
  auto dot_row = [&](const float* row, int d, int n) -> float {
    float acc = 0.f;
    if constexpr (KC > 0) {
      float r[RAC];
#pragma unroll
      for (int j = 0; j < RAC / 4; ++j) {
        const float4 x = reinterpret_cast<const float4*>(row)[j];
        r[4 * j] = x.x; r[4 * j + 1] = x.y; r[4 * j + 2] = x.z; r[4 * j + 3] = x.w;
      }
#pragma unroll
      for (int kk = 0; kk < WSC; ++kk)
        if (kk < n) acc = fmaf(r[kk], wreg[d][kk], acc);
    } else {
      for (int kk = 0; kk < n; ++kk) acc = fmaf(row[kk], WSM(d, kk), acc);
    }
    return acc;
  };
  auto weight = [&](int d, int kk) -> float {
    if constexpr (KC > 0) return wreg[d][kk]; else return WSM(d, kk);
  };
  const float r_tau = __frcp_rn(c.tau), r_dt = __frcp_rn(c.env.dt_f);
  const double r_dt64 = __drcp_rn(c.env.dt);

  // ---- per-env phase (NTX > 0): this env's tau / delay / time grid, and the basis row of one time point -----------------
  float tau_b = c.tau, delay_b = 0.f, r_tau_b = r_tau;
  const float* tm = pc.times;
  constexpr int KCC = (KC > 0) ? KC : 1;
  auto load_phase = [&]() -> int {          // returns the number of points of this env's plan
    int T_b = c.T;
    if constexpr (NTX > 0) {
      tau_b = pc.tau[b];
      delay_b = pc.delay[b];
      r_tau_b = __frcp_rn(tau_b);
      if (pc.n_steps_env) {
        T_b = min(max(pc.n_steps_env[b], 2), c.T);
        tm = pc.times_table + (long long)T_b * pc.times_stride;
      }
    }
    return T_b;
  };
  auto scaled_time = [&](int t_) -> float {   // left-bounded linear phase, float32 elementwise ops of the library
    return fmaxf(div_by(__fsub_rn(tm[t_], delay_b), tau_b, r_tau_b), 0.f);
  };
  // coefficients of the KC weighted basis functions at time point t_: float64 phase / RBFs rounded once (exactly eval_basis of
  // fg_trajgen_phase.cu), ProMP: * weights_scale, DMP: canonical x * basis (* the scale when it sits on the basis)
  auto eval_row = [&](int t_, float (&coef)[KCC]) {
    if constexpr (NTX > 0) {
      const float un = div_by(__fsub_rn(tm[t_], delay_b), tau_b, r_tau_b);
      const float z = fminf(fmaxf(un, 0.f), (pc.phase_kind && !pc.exp_right_clip) ? INFINITY : 1.f);
      const double ph = pc.phase_kind ? exp(-pc.alpha_phase * (double)z) : (double)z;
      double phi[NTX];
      bool direct = true;
      if constexpr (MP == FG_MP_PROMP && NTX >= 3) {
        // the recurrence of fg_device.cuh (two exp() instead of NTX); a value too close to a float32 rounding boundary
        // sends the time point through the direct evaluation below
        if (pc.rec.on) direct = rbf_recurrence_eval<NTX>(pc.rec, pc.cen, pc.bw, ph, NTX - KCC, phi);
      }
      if (direct) {
        double sum = 0.0;
#pragma unroll
        for (int kk = 0; kk < NTX; ++kk) {
          const double dd = ph - pc.cen[kk];
          phi[kk] = exp(-((dd * dd * pc.bw[kk]) / 2));
          sum += phi[kk];
        }
        if (NTX > 1) {
          const double rr = 1.0 / sum;
#pragma unroll
          for (int kk = 0; kk < NTX; ++kk) {
            const double qq = phi[kk] * rr;
            phi[kk] = fma(fma(-qq, sum, phi[kk]), rr, qq);
          }
        }
      }
#pragma unroll
      for (int kk = 0; kk < KCC; ++kk) {
        const double f_ = phi[NTX - KCC + kk];         // the weighted functions are the last KC (zero padding in front)
        coef[kk] = (MP == FG_MP_PROMP) ? __fmul_rn((float)f_, c.wscale) : (float)(ph * f_ * pc.basis_scale);
      }
    }
  };
  auto dot_coef = [&](const float (&coef)[KCC], int d) -> float {      // FMA chain in index order, accumulator starts at 0
    float acc = 0.f;
    if constexpr (KC > 0 && HAS_W) {
#pragma unroll
      for (int kk = 0; kk < KCC; ++kk) acc = fmaf(coef[kk], wreg[d][kk], acc);
    }
    return acc;
  };

  // ---- the env's context (read again whenever a thread picks an env up: a few L2 hits per re-packing) ----
  auto load_context = [&]() {
    if constexpr (ENV != FG_ENV_TOY) {
      cx[0] = io.ctx[b * 4 + 0]; cx[1] = io.ctx[b * 4 + 1]; cx[2] = io.ctx[b * 4 + 2]; cx[3] = io.ctx[b * 4 + 3];
    }
    if constexpr (ENV == FG_ENV_HOLE_REACHER) hole = hole_of(cx);
  };
  auto plan_seg = [&](int kk) -> int {       // steps plan kk may execute (ragged sub-trajectories: per env)
    if (io.n_plans > 1) return io.plan_seg[kk];
    return io.seg_steps_env ? min(seg_steps, io.seg_steps_env[b]) : seg_steps;
  };

  // ---- start of a plan: boundary condition (black_box_wrapper.py:110-114, float32 like the library) + MP set-up ----
  auto plan_setup = [&](const float (&ybc)[N], const float (&vbc)[N]) {
    if constexpr (MP == FG_MP_PRODMP) {
#pragma unroll
      for (int d = 0; d < N; ++d) {
        WSM(d, 0) = ybc[d];
        WSM(d, 1) = __fmul_rn(vbc[d], c.tau);
        if (c.rel_goal) WSM(d, K + 2) = __fadd_rn(WSM(d, K + 2), ybc[d]);
      }
    }
    fetch_weights();
    if constexpr (MP == FG_MP_DMP) {
#pragma unroll
      for (int d = 0; d < N; ++d) {
        carry_a[d] = ybc[d];
        carry_b[d] = __fmul_rn(vbc[d], tau_b);
      }
    }
    if constexpr (MP == FG_MP_PROMP) {
      float coef0[KCC];
      eval_row(tr, coef0);
#pragma unroll
      for (int d = 0; d < N; ++d) {
        carry_a[d] = (NTX > 0) ? dot_coef(coef0, d) : dot_row(tabA + tr * RA, d, K);
        carry_b[d] = 0.f;             // (a one-point plan has zero velocity; otherwise overwritten at the first step)
      }
    }
  };

  // full step observation (float64 trig, cast to float32 like _get_obs) given the end effector; returns its width
  auto build_obs = [&](float* obs, double ex, double ey) -> int {
    int no = 0;
    if constexpr (ENV == FG_ENV_TOY) obs[no++] = -1.0f;
    else if constexpr (VF) no = reacher_obs<ENV, N>(obs, q, vf, cx, ex, ey, steps);
    else no = reacher_obs<ENV, N>(obs, q, v, cx, ex, ey, steps);
    if (c.time_aware) obs[no++] = (float)((double)steps / (double)c.env.max_steps);
    return no;
  };
  auto end_effector_now = [&](double& ex, double& ey) {
    if constexpr (ENV == FG_ENV_TOY) {
      ex = ey = 0.0;
    } else {
      double th[N];
      th[0] = q[0];
#pragma unroll
      for (int i = 1; i < N; ++i) th[i] = th[i - 1] + q[i];
      end_effector64<N>(th, ex, ey);
    }
  };

  // ---- the multi-GPU gather, fused: this env's result row goes straight into every peer's gather buffer (NVLink stores;
  // ---- the block layout is that of a contiguous result block: return f64 [B] | length i32 [B] | flags u8 [B] | 4 x u8 [B]) ----
  auto peer_store = [&](double r_, int len_, unsigned char f_) {
    for (int r = 0; r < io.n_peers; ++r) {
      unsigned char* base = static_cast<unsigned char*>(io.peer_bufs[r]) + io.peer_offset;
      reinterpret_cast<double*>(base)[b] = r_;
      reinterpret_cast<int*>(base + 8 * B)[b] = len_;
      base[12 * B + b] = f_;
      base[13 * B + b] = (f_ & FG_FLAG_TERMINATED) != 0;
      base[14 * B + b] = (f_ & FG_FLAG_TRUNCATED) != 0;
      base[15 * B + b] = (f_ & FG_FLAG_SUCCESS) != 0;
      base[16 * B + b] = (f_ & FG_FLAG_COLLIDED) != 0;
    }
  };
  // ---- results of plan kk of this env (what one step() call of the reference returns) ----
  auto write_plan_outputs = [&](int kk, int len, unsigned f, const float* obs, double i0, double i1) {
    const long long o = (long long)kk * B + b;
    io.ret[o] = ret;
    io.length[o] = len;
    const unsigned char fbyte = ((f & kSlotTerminated) ? FG_FLAG_TERMINATED : 0u) | ((f & kSlotTruncated) ? FG_FLAG_TRUNCATED : 0u) |
                                ((f & kSlotSuccess) ? FG_FLAG_SUCCESS : 0u) | ((f & kSlotCollided) ? FG_FLAG_COLLIDED : 0u);
    io.flags[o] = fbyte;
    if (io.flag_bytes) {
      unsigned char* fb = io.flag_bytes + (long long)kk * 4 * B;
      fb[b] = (f & kSlotTerminated) != 0;
      fb[B + b] = (f & kSlotTruncated) != 0;
      fb[2 * B + b] = (f & kSlotSuccess) != 0;
      fb[3 * B + b] = (f & kSlotCollided) != 0;
    }
    if (io.n_peers > 0) peer_store(ret, len, fbyte);
    for (int j = 0; j < c.n_obs_out; ++j) io.obs[o * c.n_obs_out + j] = obs[c.obs_index[j]];
    io.info[o * 4 + 0] = i0;
    io.info[o * 4 + 1] = i1;
    double lx = 0.0, ly = 0.0;
    if constexpr (ENV == FG_ENV_HOLE_REACHER) latch_get(lx, ly);
    io.info[o * 4 + 2] = lx;
    io.info[o * 4 + 3] = ly;
  };
  // the desired state of the last executed step (tl - 1) of the current plan (condition_on_desired)
  auto last_desired = [&](float (&lp)[N], float (&lv)[N]) {
    if constexpr (SL::LASTDES) {
#pragma unroll
      for (int i = 0; i < N; ++i) { lp[i] = pos[i]; lv[i] = vel[i]; }
    } else {
      // the desired position is not carried through the loop in this instantiation: the same FMA chain, once, here
      const float* row = tabA + (tr - 1) * RA;
      float coefl[KCC];
      eval_row(tr - 1, coefl);
#pragma unroll
      for (int i = 0; i < N; ++i) {
        lp[i] = (NTX > 0) ? dot_coef(coefl, i) : dot_row(row, i, MP == FG_MP_PROMP ? K : K + 3);
        if constexpr (MP == FG_MP_PROMP) lv[i] = carry_b[i];
        else lv[i] = div_by(dot_row(tabB + (tr - 1) * RB, i, K + 3), c.tau, r_tau);
      }
    }
  };

  // ---- parking / picking up an env --------------------------------------------------------------------------------
  auto park = [&]() {
    unsigned* s = sst + own;
#pragma unroll
    for (int i = 0; i < N; ++i) {
      s[(SL::W_Q + 2 * i) * BD] = (unsigned)__double2loint(q[i]);
      s[(SL::W_Q + 2 * i + 1) * BD] = (unsigned)__double2hiint(q[i]);
      if constexpr (VF) {
        s[(SL::W_V + i) * BD] = __float_as_uint(vf[i]);
      } else {
        s[(SL::W_V + 2 * i) * BD] = (unsigned)__double2loint(v[i]);
        s[(SL::W_V + 2 * i + 1) * BD] = (unsigned)__double2hiint(v[i]);
      }
      if constexpr (SL::CARRY) {
        s[(SL::W_CARRY + i) * BD] = __float_as_uint(carry_a[i]);
        s[(SL::W_CARRY + N + i) * BD] = __float_as_uint(carry_b[i]);
      }
      if constexpr (SL::LASTDES) {
        s[(SL::W_LAST + i) * BD] = __float_as_uint(pos[i]);
        s[(SL::W_LAST + N + i) * BD] = __float_as_uint(vel[i]);
      }
    }
    if constexpr (ENV == FG_ENV_SIMPLE_REACHER) {
      s[(SL::W_INFO + 0) * BD] = (unsigned)__double2loint(info0); s[(SL::W_INFO + 1) * BD] = (unsigned)__double2hiint(info0);
      s[(SL::W_INFO + 2) * BD] = (unsigned)__double2loint(info1); s[(SL::W_INFO + 3) * BD] = (unsigned)__double2hiint(info1);
    }
    unsigned* z = s + SL::W_SCAL * BD;
    z[SL::S_B * BD] = (unsigned)b;
    z[SL::S_STEPS * BD] = (unsigned)steps;
    z[SL::S_K * BD] = (unsigned)k;
    z[SL::S_TR * BD] = (unsigned)tr;
    z[SL::S_TREND * BD] = (unsigned)tr_end;
    z[SL::S_TRLAST * BD] = (unsigned)tr_last;
    z[SL::S_FLAGS * BD] = fl;
    z[SL::S_RET * BD] = (unsigned)__double2loint(ret); z[(SL::S_RET + 1) * BD] = (unsigned)__double2hiint(ret);
  };
  auto pick_up = [&](int slot) {
    own = slot;
    const unsigned* s = sst + own;
#pragma unroll
    for (int i = 0; i < N; ++i) {
      q[i] = __hiloint2double((int)s[(SL::W_Q + 2 * i + 1) * BD], (int)s[(SL::W_Q + 2 * i) * BD]);
      if constexpr (VF) {
        vf[i] = __uint_as_float(s[(SL::W_V + i) * BD]);
        v[i] = 0.0;
      } else {
        v[i] = __hiloint2double((int)s[(SL::W_V + 2 * i + 1) * BD], (int)s[(SL::W_V + 2 * i) * BD]);
        vf[i] = 0.f;
      }
      if constexpr (SL::CARRY) {
        carry_a[i] = __uint_as_float(s[(SL::W_CARRY + i) * BD]);
        carry_b[i] = __uint_as_float(s[(SL::W_CARRY + N + i) * BD]);
      }
      if constexpr (SL::LASTDES) {
        pos[i] = __uint_as_float(s[(SL::W_LAST + i) * BD]);
        vel[i] = __uint_as_float(s[(SL::W_LAST + N + i) * BD]);
      }
    }
    if constexpr (ENV == FG_ENV_SIMPLE_REACHER) {
      info0 = __hiloint2double((int)s[(SL::W_INFO + 1) * BD], (int)s[(SL::W_INFO + 0) * BD]);
      info1 = __hiloint2double((int)s[(SL::W_INFO + 3) * BD], (int)s[(SL::W_INFO + 2) * BD]);
    }
    const unsigned* z = s + SL::W_SCAL * BD;
    b = (long long)z[SL::S_B * BD];
    steps = (int)z[SL::S_STEPS * BD];
    k = (int)z[SL::S_K * BD];
    tr = (int)z[SL::S_TR * BD];
    tr_end = (int)z[SL::S_TREND * BD];
    tr_last = (int)z[SL::S_TRLAST * BD];
    fl = z[SL::S_FLAGS * BD];
    ret = __hiloint2double((int)z[(SL::S_RET + 1) * BD], (int)z[SL::S_RET * BD]);
    load_context();
    load_phase();
    fetch_weights();
  };

  // ---- end of an episode / of the launch for this env: everything that is done once (runs for packed lanes) ----------
  // the reward of a step that collided is completed when the env is finished: what it needs from that step goes straight to
  // the env's slot (a rare path: not a loop-carried register)
  auto defer = [&](double a) {
    unsigned* z = sst + (SL::W_SCAL + SL::S_AUX) * BD + own;
    z[0] = (unsigned)__double2loint(a);
    z[BD] = (unsigned)__double2hiint(a);
  };
  auto finish = [&]() {
    const int tl = (NTX > 0) ? tr : tr - (tr_last - (io.plan_T - 1));      // steps this plan executed
    const unsigned* za = sst + (SL::W_SCAL + SL::S_AUX) * BD + own;
    const double aux = __hiloint2double((int)za[BD], (int)za[0]);
    double ex, ey;
    end_effector_now(ex, ey);
    if (fl & kSlotDeferred) {
      // the reward of the step that collided (its distance term needs the float64 end effector): the last addend of the return
      const double reward = collided_reward<ENV>(c.env, cx, aux, ex, ey, latch_put);
      ret += reward;
      if constexpr (DBG) {
        if (io.dbg_rewards) io.dbg_rewards[b * c.T + tl - 1] = reward;
      }
    }
    const bool stopped = (fl & (kSlotTerminated | kSlotTruncated)) != 0;
    if (!io.keep_state) {
      if constexpr (ENV != FG_ENV_TOY) {
#pragma unroll
        for (int i = 0; i < N; ++i) {
          io.q[b * N + i] = q[i];
          io.v[b * N + i] = VF ? (double)vf[i] : v[i];
        }
      }
      io.steps[b] = steps;
      io.done[b] = stopped ? 1 : 0;
    }
    if (io.write_cond && tl > 0 && (stopped || io.write_cond == 2)) {
      float lp[N], lv[N];
      last_desired(lp, lv);
#pragma unroll
      for (int i = 0; i < N; ++i) {
        io.cond_pos[b * N + i] = lp[i];
        io.cond_vel[b * N + i] = lv[i];
      }
    }
    float obs[FG_MAX_OBS];
    build_obs(obs, ex, ey);
    if constexpr (ENV == FG_ENV_HOLE_REACHER || ENV == FG_ENV_VIAPOINT_REACHER) {
      info0 = ex;
      info1 = ey;
    }
    write_plan_outputs(k, tl, fl, obs, info0, info1);
    // plans after the one the episode ended in never run: they report 0 steps and keep the last observation / infos
    const double r_keep = ret;
    ret = 0.0;
    for (int kk = k + 1; kk < n_plans; ++kk) write_plan_outputs(kk, 0, 0u, obs, info0, info1);
    ret = r_keep;
  };

  // ---- start env `b` in slot `own` (its parameters of the first plan are in wsm already): true if it runs ----
  auto start_env = [&]() -> bool {
    if (io.done[b]) {   // episode already over: frozen (oracle/blackbox.py keeps such envs untouched)
      for (int kk = 0; kk < n_plans; ++kk) {
        const long long o = (long long)kk * B + b;
        io.ret[o] = 0.0;
        io.length[o] = 0;
        io.flags[o] = 0;
        if (io.flag_bytes)
          for (int i = 0; i < 4; ++i) io.flag_bytes[((long long)kk * 4 + i) * B + b] = 0;
        if (io.prev_obs)
          for (int j = 0; j < c.n_obs_out; ++j) io.obs[o * c.n_obs_out + j] = io.prev_obs[b * c.n_obs_out + j];
        if (io.prev_info)
          for (int j = 0; j < 4; ++j) io.info[o * 4 + j] = io.prev_info[b * 4 + j];
      }
      if (io.n_peers > 0) peer_store(0.0, 0, 0);
      fl = kSlotEmpty;
      return false;
    }
#pragma unroll
    for (int i = 0; i < N; ++i) {
      if constexpr (ENV == FG_ENV_TOY) {   // ToyWrapper: current_pos = 1, current_vel = 0 (test_black_box.py:48-56)
        q[i] = 1.0;
        v[i] = 0.0;
        vf[i] = 0.f;
      } else {
        q[i] = io.q[b * N + i];
        v[i] = io.v[b * N + i];
        vf[i] = (float)v[i];
      }
    }
    steps = io.steps[b];
    k = 0;
    ret = 0.0;
    load_context();
    if constexpr (ENV == FG_ENV_HOLE_REACHER) {
      if (c.env.rew_fct == 2 && steps > 0) latch_put(io.info[b * 4 + 2], io.info[b * 4 + 3]);   // a later plan segment of the episode
      else latch_put(0.0, 0.0);
    }
    float ybc[N], vbc[N];
#pragma unroll
    for (int i = 0; i < N; ++i) {
      if (io.use_cond) {
        ybc[i] = io.cond_pos[b * N + i];
        vbc[i] = io.cond_vel[b * N + i];
      } else {
        ybc[i] = (float)q[i];
        vbc[i] = VF ? vf[i] : (float)v[i];
      }
    }
    tr = io.n_plans > 1 ? io.plan_row0[0] : 0;
    tr_end = tr + plan_seg(0);
    const int T_b = load_phase();
    tr_last = tr + ((NTX > 0) ? T_b : io.plan_T) - 1;
    plan_setup(ybc, vbc);
    fl = kSlotLive;
    if (tr_end <= tr) fl = kSlotPending;  // nothing to execute: reports 0 steps
    return fl == kSlotLive;
  };

  // =================================================================================================================
  // initial binding: thread tid <-> slot tid <-> env b0 + tid
  // =================================================================================================================
  {
    bool live = false;
    if (tid < n_here && b < B) live = start_env();
    const unsigned m = __ballot_sync(0xffffffffu, live);
    if (lane == 0 && m) {
      atomicAdd(const_cast<int*>(&ctl[1]), __popc(m));
      atomicAdd(const_cast<int*>(&ctl[2]), 1);       // warps that run something
    }
    if (fl == kSlotEmpty) sst[(SL::W_SCAL + SL::S_FLAGS) * BD + tid] = kSlotEmpty;
  }
  __syncthreads();
  // (envs that were already done / a ragged last block: re-pack right away when that frees a warp)
  if (tid == 0 && ((ctl[1] + 31) >> 5) < ctl[2]) ctl[0] = 1;
  bool have = (fl == kSlotLive);          // this thread is running an env
  bool bound = (fl != kSlotEmpty);        // this thread holds an env's state in its registers (running or just stopped)
  __syncthreads();

  // =================================================================================================================
#ifdef FG_ROLLOUT_NAMED_BARRIERS
#define FG_BAR(id) asm volatile("bar.sync " #id ", %0;" ::"n"(kRolloutThreads) : "memory")
#else
#define FG_BAR(id) __syncthreads()
#endif
#ifdef FG_ROLLOUT_CHECK
  int rnd = 0;
#endif
  for (;;) {
    // ------------------------------------------------------------------ run until the block wants to re-pack
    // (a lane whose env stops leaves the loop and waits for its warp; a warp without a running lane goes straight to the
    //  barrier of the re-packing and sleeps there)
    for (;;) {
      // success / collided of the last executed step (what the plan reports when its segment simply runs out)
      bool success = false, collided = false;
      while (have && tr < tr_end && want_repack() == 0) {
        FG_CHAOS(16, 4000);
        {
        const int t = tr;
        // ---------------------------------------------------------------- desired pos / vel at point t of the plan
        if constexpr (MP == FG_MP_PROMP) {
#pragma unroll
          for (int d = 0; d < N; ++d) pos[d] = carry_a[d];
          if (t < tr_last) {
            const float* row = tabA + (t + 1) * RA;
            float dtt, rdt;
            float coef[KCC];
            if constexpr (NTX > 0) {
              eval_row(t + 1, coef);
              dtt = __fsub_rn(tm[t + 1], tm[t]);
              rdt = __frcp_rn(dtt);
            } else {
              dtt = tabB[t * RB];
              rdt = tabR[t];
            }
#pragma unroll
            for (int d = 0; d < N; ++d) {
              const float acc = (NTX > 0) ? dot_coef(coef, d) : dot_row(row, d, K);
              carry_a[d] = acc;
              carry_b[d] = div_by(__fsub_rn(acc, pos[d]), dtt, rdt);     // (pos[t+1]-pos[t]) / (times[t+1]-times[t])
            }
          }                     // t == T - 1: vel[T-1] = vel[T-2] — the registers simply keep the previous step's values
#pragma unroll
          for (int d = 0; d < N; ++d) vel[d] = carry_b[d];
        } else if constexpr (MP == FG_MP_DMP) {
#pragma unroll
          for (int d = 0; d < N; ++d) {
            pos[d] = carry_a[d];
            vel[d] = div_by(carry_b[d], tau_b, r_tau_b);
          }
          if (t < tr_last) {   // semi-implicit Euler in scaled time (oracle/mp.py DMP._integrate)
            const float* row = tabA + t * RA;
            float h;
            float coef[KCC];
            if constexpr (NTX > 0) {
              eval_row(t, coef);
              h = __fsub_rn(scaled_time(t + 1), scaled_time(t));
            } else {
              h = tabB[t * RB];
            }
#pragma unroll
            for (int d = 0; d < N; ++d) {
              const float f = (NTX > 0) ? dot_coef(coef, d) : dot_row(row, d, K);
              const float g = weight(d, K);
              float a = __fmul_rn(c.beta, __fsub_rn(g, carry_a[d]));
              a = __fmul_rn(c.alpha, __fsub_rn(a, carry_b[d]));
              a = __fadd_rn(a, f);
              carry_b[d] = __fadd_rn(carry_b[d], __fmul_rn(h, a));
              carry_a[d] = __fadd_rn(carry_a[d], __fmul_rn(h, carry_b[d]));
            }
          }
        } else if constexpr (MP == FG_MP_PRODMP) {
          const float* rp = tabA + t * RA;
          const float* rv = tabB + t * RB;
#pragma unroll
          for (int d = 0; d < N; ++d) {
            if constexpr (!VEL_ONLY) pos[d] = dot_row(rp, d, K + 3);
            vel[d] = div_by(dot_row(rv, d, K + 3), c.tau, r_tau);
          }
        } else {
#pragma unroll
          for (int d = 0; d < N; ++d) {
            pos[d] = io.traj_pos[(b * c.T + t) * N + d];
            vel[d] = io.traj_vel[(b * c.T + t) * N + d];
          }
        }

        // ---------------------------------------------------------------- controller + clip + dynamics
        double a64[N];
        float a32[N];
        if constexpr (MOTOR) {    // pd_controller.py:28: float64 because c_pos / c_vel are float64
#pragma unroll
          for (int i = 0; i < N; ++i) {
            const double tq = __dadd_rn(__dmul_rn(c.p[i], (double)pos[i] - q[i]), __dmul_rn(c.d[i], (double)vel[i] - v[i]));
            // np.clip(tq, -lim, lim): one compare on |tq| and a sign transplant instead of the two NaN-aware fmin / fmax
            // sequences (~16 instructions per joint; they were 21 % of the SimpleReacher kernel)
            const double lim = (double)c.act_lim;
            a64[i] = (fabs(tq) > lim) ? copysign(lim, tq) : tq;
          }
        } else {
#pragma unroll
          for (int i = 0; i < N; ++i) {
            const float des = (VEL_ONLY || c.ctrl == FG_CTRL_VELOCITY) ? vel[i] : pos[i];
            // np.clip(des, -lim, lim) keeps a NaN, which fminf / fmaxf would turn into -lim
            a32[i] = fmin_nan(fmax_nan(des, -c.act_lim), c.act_lim);
            a64[i] = (double)a32[i];
          }
        }

        // v is float64 (zeros at reset / float64 actions) unless it holds the previous float32 action
        double acc_cost;
        if constexpr (VF) acc_cost = reacher_dynamics<ENV, N, MOTOR>(c.env, r_dt, r_dt64, q, vf, a64, a32, MOTOR || steps == 0);
        else acc_cost = reacher_dynamics<ENV, N, MOTOR>(c.env, r_dt, r_dt64, q, v, a64, a32, MOTOR || steps == 0);

        // ---------------------------------------------------------------- geometry, collisions, reward
        double reward = 0.0;
        bool terminated = false, deferred = false;
        success = collided = false;
        if constexpr (ENV == FG_ENV_TOY) {
          reward = 1.0;
        } else {
          double th[N];
          th[0] = q[0];
#pragma unroll
          for (int i = 1; i < N; ++i) th[i] = th[i - 1] + q[i];
          // the float64 end effector only on the steps whose reward reports it
          const StepReward r = reacher_reward<ENV, N, MOTOR>(c.env, q, th, a64, a32, acc_cost, steps, cx, hole, s_m,
                                                             [&](double& ex, double& ey) { end_effector64<N>(th, ex, ey); },
                                                             latch_get, latch_put);
          reward = r.reward;
          collided = r.collided;
          success = r.success;
          deferred = r.deferred;
          if (deferred) defer(r.aux);   // the rest of this reward is added when the env is finished (see finish())
          if constexpr (ENV == FG_ENV_SIMPLE_REACHER) {
            info0 = r.info0;
            info1 = r.info1;
          } else {
            terminated = collided;
          }
        }
        steps += 1;
        const bool truncated = steps >= c.env.max_steps;       // gymnasium TimeLimit (App. A.6-Q12)
        ret += reward;            // (+0.0 for a deferred step: the return is never -0.0, so this leaves it as it is)

        if constexpr (DBG) {
          if (io.dbg_rewards && !deferred) io.dbg_rewards[b * c.T + t] = reward;
          if (io.dbg_actions) {
#pragma unroll
            for (int i = 0; i < N; ++i) io.dbg_actions[(b * c.T + t) * N + i] = a64[i];
          }
          if (io.dbg_state) {
#pragma unroll
            for (int i = 0; i < N; ++i) {
              io.dbg_state[(b * c.T + t) * 2 * N + i] = q[i];
              io.dbg_state[(b * c.T + t) * 2 * N + N + i] = VF ? (double)vf[i] : v[i];
            }
          }
          if (io.dbg_obs) {
            float so[FG_MAX_OBS];
            double ex, ey;
            end_effector_now(ex, ey);
            const int n_full = build_obs(so, ex, ey);
            for (int j = 0; j < n_full; ++j) io.dbg_obs[(b * c.T + t) * n_full + j] = so[j];
          }
        }
        tr = t + 1;
        if (terminated || truncated) {
          // this env's episode is over: it waits in its slot until it is finished (see finish()); when the block's live envs now
          // fit into fewer warps, ask for a re-packing
          fl = kSlotPending | (terminated ? kSlotTerminated : 0u) | (truncated ? kSlotTruncated : 0u) |
               (success ? kSlotSuccess : 0u) | (collided ? kSlotCollided : 0u) | (deferred ? kSlotDeferred : 0u);
          have = false;
          const int left = atomicSub(const_cast<int*>(&ctl[1]), 1) - 1;
          if (((left + 31) >> 5) < ctl[2]) ctl[0] = 1;
        }
        }
      }
      // ---- the lanes of the warp are together again.  A plan whose segment ran out: a re-planning break
      // (black_box_wrapper.py:197-203: this plan's results, then the next plan) or the end of this launch for the env
      FG_CHAOS(2, 20000);
      if (!(have && tr >= tr_end)) break;
      FG_CHAOS(2, 20000);
      fl = kSlotLive | (success ? kSlotSuccess : 0u) | (collided ? kSlotCollided : 0u);
      if (k + 1 < n_plans) {
        double ex, ey;
        end_effector_now(ex, ey);
        float obs[FG_MAX_OBS];
        build_obs(obs, ex, ey);
        if constexpr (ENV == FG_ENV_HOLE_REACHER || ENV == FG_ENV_VIAPOINT_REACHER) {
          info0 = ex;
          info1 = ey;
        }
        write_plan_outputs(k, tr - (tr_last - (io.plan_T - 1)), fl, obs, info0, info1);
        float ybc[N], vbc[N];
        if (io.write_cond) {            // condition_on_desired: the next plan starts from the DESIRED state of the break
          last_desired(ybc, vbc);
        } else {
#pragma unroll
          for (int i = 0; i < N; ++i) {
            ybc[i] = (float)q[i];
            vbc[i] = VF ? vf[i] : (float)v[i];
          }
        }
        k += 1;
        ret = 0.0;
        fl = kSlotLive;
        tr = io.plan_row0[k];
        tr_end = tr + plan_seg(k);
        tr_last = tr + io.plan_T - 1;
        if constexpr (HAS_W) {          // this env's parameters of plan k (its own row: a handful of L2 reads per plan)
          const float* pk = io.params + b * PS + (long long)k * P;
          for (int idx = 0; idx < P; ++idx) put_param(own, idx, pk[idx]);
        }
        plan_setup(ybc, vbc);
      } else {
        fl = (fl & ~kSlotStatusMask) | kSlotPending;
        have = false;
        const int left = atomicSub(const_cast<int*>(&ctl[1]), 1) - 1;
        if (((left + 31) >> 5) < ctl[2]) ctl[0] = 1;
      }
    }

    // ------------------------------------------------------------------ re-pack (block-uniform)
    FG_CHAOS(2, 50000);
    if (bound) park();
    FG_CHAOS(2, 50000);
#ifdef FG_ROLLOUT_CHECK
    int* chk = reinterpret_cast<int*>(sst + SL::WORDS * BD);
    chk[tid] = rnd;
#endif
    FG_BAR(1);                            // every env of the block is in its slot; nobody reads the control words any more
#ifdef FG_ROLLOUT_CHECK
    for (int w = 0; w < kRolloutWarps; ++w)
      if (chk[w * 32 + lane] != rnd)
        printf("B1 skew: block %d thread %d round %d sees thread %d in round %d\n", (int)blockIdx.x, tid, rnd, w * 32 + lane, chk[w * 32 + lane]);
#endif
    FG_CHAOS(2, 20000);
    const unsigned st = sst[(SL::W_SCAL + SL::S_FLAGS) * BD + tid] & kSlotStatusMask;
#ifdef FG_ROLLOUT_CHECK
    {
      const unsigned am = __activemask();
      if (am != 0xffffffffu) printf("diverged at the scan: block %d thread %d activemask %08x\n", (int)blockIdx.x, tid, am);
    }
#endif
    const unsigned lm = __ballot_sync(0xffffffffu, st == kSlotLive), pm = __ballot_sync(0xffffffffu, st == kSlotPending);
    if (lane == 0) {
      wcount[warp] = __popc(lm);
      wcount[kRolloutWarps + warp] = __popc(pm);
    }
#ifdef FG_ROLLOUT_CHECK
    chk[BD + tid] = rnd;
#endif
    FG_BAR(2);
#ifdef FG_ROLLOUT_CHECK
    for (int w = 0; w < kRolloutWarps; ++w)
      if (chk[BD + w * 32 + lane] != rnd)
        printf("B2 skew: block %d thread %d round %d sees thread %d in round %d\n", (int)blockIdx.x, tid, rnd, w * 32 + lane, chk[BD + w * 32 + lane]);
#endif
    FG_CHAOS(2, 20000);
    int lbase = 0, pbase = 0, n_live = 0, n_pend = 0;
#pragma unroll
    for (int w = 0; w < kRolloutWarps; ++w) {
      const int a = wcount[w], p_ = wcount[kRolloutWarps + w];
      if (w < warp) {
        lbase += a;
        pbase += p_;
      }
      n_live += a;
      n_pend += p_;
    }
    const unsigned lt = (1u << lane) - 1u;
    if (st == kSlotLive) live_list[lbase + __popc(lm & lt)] = (unsigned short)tid;
    if (st == kSlotPending) pend_list[pbase + __popc(pm & lt)] = (unsigned short)tid;
    // Stopped envs are finished 32 at a time by the threads from the top of the block (warps that have nothing to run),
    // or all of them once nothing is running any more.  With a work queue (more envs than resident threads) every thread
    // that finishes an env starts the next env of the queue in the same slot: the block stays full until the queue is empty.
    const bool do_finish = n_pend > 0 && (n_pend >= 32 || n_live == 0);
    const int n_fin = do_finish ? n_pend : 0;
    if (tid == 0) {
      unsigned base = 0xffffffffu;
      if (queue && n_fin > 0 && ctl[3] == 0) {
        base = atomicAdd(queue, (unsigned)n_fin);
        if ((long long)base + (long long)gridDim.x * BD >= B) ctl[3] = 1;       // the queue has run dry
      }
      ctl[4] = (int)base;
      ctl[0] = 0;
      ctl[1] = n_live;          // (+ the envs started from the queue: added by their threads below)
      ctl[2] = 0;               // warps that run something: counted below
    }
#ifdef FG_ROLLOUT_CHECK
    chk[2 * BD + tid] = rnd;
#endif
    FG_BAR(3);                            // the lists are complete
#ifdef FG_ROLLOUT_CHECK
    for (int w = 0; w < kRolloutWarps; ++w)
      if (chk[2 * BD + w * 32 + lane] != rnd)
        printf("B3 skew: block %d thread %d round %d sees thread %d in round %d\n", (int)blockIdx.x, tid, rnd, w * 32 + lane, chk[2 * BD + w * 32 + lane]);
    rnd += 1;
#endif
    FG_CHAOS(2, 50000);
    have = bound = false;
    if (tid < n_live) {
      pick_up(live_list[tid]);
      have = bound = true;
    } else if (BD - 1 - tid < n_fin) {
      const int j = BD - 1 - tid;
      pick_up(pend_list[j]);
      FG_CHAOS(2, 100000);
      finish();
      FG_CHAOS(2, 100000);
      fl = kSlotEmpty;
      const unsigned base = (unsigned)ctl[4];
      const long long nb = (long long)gridDim.x * BD + (long long)base + j;
      if (queue && base != 0xffffffffu && nb < B) {        // the next env of the queue, in the slot that has just become free
        b = nb;
        if constexpr (HAS_W) {
          const float* pk = io.params + b * PS;
          for (int idx = 0; idx < P; ++idx) put_param(own, idx, pk[idx]);
        }
        if (start_env()) {
          have = true;
          atomicAdd(const_cast<int*>(&ctl[1]), 1);
        }
        bound = fl != kSlotEmpty;
      }
      if (!bound) sst[(SL::W_SCAL + SL::S_FLAGS) * BD + own] = kSlotEmpty;
    }
    if (__any_sync(0xffffffffu, have) && lane == 0) atomicAdd(const_cast<int*>(&ctl[2]), 1);
    if (n_live == 0) {
      if (!(queue && n_fin > 0)) break;   // every stopped env has just been finished and nothing was started
      // nothing was running: did the queue hand out envs?  (only in this case does anybody wait for the finishing threads;
      // the vote is the barrier's own: the live counter may already be counted down again by an env that has just started)
      if (!__syncthreads_or(have)) {
        // no: the block ends, unless an env was started that has nothing to execute (it is pending: one more pass)
        if (!__syncthreads_or(bound)) break;
        if (tid == 0) ctl[0] = 1;
        __syncthreads();
      }
    }
  }
  if (queue && tid == 0) {                // the last block of the launch resets the queue for the next launch
    const unsigned done_blocks = atomicAdd(queue + 1, 1u);
    if (done_blocks == gridDim.x - 1) {
      queue[0] = 0u;
      queue[1] = 0u;
    }
  }
#undef WSM
#undef FG_BAR
}

}  // namespace fg
