// Device-side episode reset: task-context sampling that reproduces numpy's Generator(PCG64(SeedSequence(seed)))
// streams bit for bit, so that env i of a batch reset with seed s is the reference env reset with seed s + i
// (gymnasium.utils.seeding.np_random; draw order of hole_reacher.py:60-112, viapoint_reacher.py:45-77,
// simple_reacher.py:46-96, base_reacher.py:73-93).  One thread per env; the stream state (40 bytes) lives in HBM between
// resets because an unseeded reset continues the env's stream.
//
// numpy algorithms restated (numpy/random/bit_generator.pyx, src/pcg64/pcg64.h, src/distributions/distributions.c):
// see oracle/np_rng.py, which is pinned against numpy and is the specification of this file.
#pragma once
#include "fg_reacher.cuh"

namespace fg {

typedef unsigned __int128 u128;

struct Pcg64 {
  u128 state, inc;
  uint32_t has32, buf32;

  __device__ __forceinline__ void step() {
    const u128 mult = ((u128)0x2360ED051FC65DA4ULL << 64) | 0x4385DF649FCCF645ULL;
    state = state * mult + inc;
  }
  __device__ void seed(uint64_t s) {
    // SeedSequence(s): entropy = the 32-bit words of s (at least one), pool of 4
    uint32_t ent[2] = {(uint32_t)s, (uint32_t)(s >> 32)};
    const int n_ent = ent[1] ? 2 : 1;
    uint32_t hc = 0x43B0D7E5u, pool[4];
    auto hashmix = [&](uint32_t v) {
      v ^= hc;
      hc *= 0x931E8875u;
      v *= hc;
      return v ^ (v >> 16);
    };
    auto mix = [](uint32_t x, uint32_t y) {
      const uint32_t r = 0xCA01F9DDu * x - 0x4973F715u * y;
      return r ^ (r >> 16);
    };
#pragma unroll
    for (int i = 0; i < 4; ++i) pool[i] = hashmix(i < n_ent ? ent[i & 1] : 0u);
#pragma unroll
    for (int i_src = 0; i_src < 4; ++i_src)
#pragma unroll
      for (int i_dst = 0; i_dst < 4; ++i_dst)
        if (i_src != i_dst) pool[i_dst] = mix(pool[i_dst], hashmix(pool[i_src]));
    uint32_t hb = 0x8B51F9DDu, w[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      uint32_t v = pool[i & 3] ^ hb;
      hb *= 0x58F38DEDu;
      v *= hb;
      w[i] = v ^ (v >> 16);
    }
    const uint64_t s0 = w[0] | ((uint64_t)w[1] << 32), s1 = w[2] | ((uint64_t)w[3] << 32);
    const uint64_t s2 = w[4] | ((uint64_t)w[5] << 32), s3 = w[6] | ((uint64_t)w[7] << 32);
    const u128 initstate = ((u128)s0 << 64) | s1, initseq = ((u128)s2 << 64) | s3;
    inc = (initseq << 1) | 1;      // pcg_setseq_128_srandom_r
    state = 0;
    step();
    state += initstate;
    step();
    has32 = 0;
    buf32 = 0;
  }
  __device__ __forceinline__ uint64_t next64() {
    step();
    const uint64_t hi = (uint64_t)(state >> 64), lo = (uint64_t)state;
    const uint64_t x = hi ^ lo;
    const unsigned rot = (unsigned)(hi >> 58);
    return (x >> rot) | (x << ((64u - rot) & 63u));
  }
  __device__ __forceinline__ uint32_t next32() {      // pcg64_next32: low half now, high half buffered
    if (has32) {
      has32 = 0;
      return buf32;
    }
    const uint64_t n = next64();
    has32 = 1;
    buf32 = (uint32_t)(n >> 32);
    return (uint32_t)n;
  }
  __device__ __forceinline__ double next_double() { return (double)(next64() >> 11) * (1.0 / 9007199254740992.0); }
  // random_uniform: lower + range * next_double, no contraction (numpy's baseline build has none)
  __device__ __forceinline__ double uniform(double low, double high) {
    return __dadd_rn(low, __dmul_rn(high - low, next_double()));
  }
  __device__ __forceinline__ int choice2() { return (int)(next32() >> 31); }    // integers(0, 2): Lemire, top bit

  __device__ __forceinline__ void load(const uint64_t* p) {
    state = ((u128)p[0] << 64) | p[1];
    inc = ((u128)p[2] << 64) | p[3];
    has32 = (uint32_t)(p[4] >> 32) & 1u;
    buf32 = (uint32_t)p[4];
  }
  __device__ __forceinline__ void store(uint64_t* p) const {
    p[0] = (uint64_t)(state >> 64); p[1] = (uint64_t)state;
    p[2] = (uint64_t)(inc >> 64); p[3] = (uint64_t)inc;
    p[4] = ((uint64_t)has32 << 32) | buf32;
  }
};

struct ResetCfg {
  int env_kind, n_dof, random_start, time_aware;
  double fixed[4];
  int has_fixed[4];
  int n_obs_out;
  int obs_index[FG_MAX_OBS];
};

__global__ void __launch_bounds__(128)
k_reset(const __grid_constant__ ResetCfg c, const __grid_constant__ fg_reset_io io, const long long B) {
  const long long b = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  if (io.mask && !io.mask[b]) return;
  const int N = c.n_dof;
  const double total = (double)N;      // link lengths are all 1 (base_reacher.py:19)
  Pcg64 g;
  const uint64_t seed = io.seeds ? (uint64_t)io.seeds[b] : (uint64_t)(io.seed0 + b);
  if (io.reseed) g.seed(seed); else g.load(io.rng_state + b * 5);

  auto first_joint = [&](double fixed_start) {     // base_reacher.py:81-86
    return c.random_start ? g.uniform(kPi / 4, 3 * kPi / 4) : fixed_start;
  };
  auto draw_in_ring = [&](double half, double lo, double hi, double& x, double& y) {
    // `goal = [total, total]; while norm(goal) >= hi or norm(goal) <= lo: goal = uniform(-half, half, size=2)`
    x = total; y = total;
    for (;;) {
      const double r = sqrt(x * x + y * y);
      if (!(r >= hi || r <= lo)) break;
      x = g.uniform(-half, half);
      y = g.uniform(-half, half);
    }
  };

  double ctx[4] = {0, 0, 0, 0}, q0;
  if (c.env_kind == FG_ENV_HOLE_REACHER) {
    // hole_reacher.py:60-71: seed -> _generate_hole (:79-112) -> base reset on the same stream
    const double width = c.has_fixed[1] ? c.fixed[1] : g.uniform(0.15, 0.5);
    double x;
    if (c.has_fixed[0]) {
      x = c.fixed[0];
    } else {
      const double direction = g.choice2() ? 1.0 : -1.0;
      x = direction * g.uniform(width / 2, 3.5);
    }
    const double depth = c.has_fixed[2] ? c.fixed[2] : g.uniform(1.0, 1.0);
    q0 = first_joint(kPi / 2);
    ctx[0] = x; ctx[1] = width; ctx[2] = depth;
  } else {
    // viapoint_reacher.py:45-53 / simple_reacher.py:46-54: _generate_goal(), seeded reset, _generate_goal(), seeded reset.
    // Seeded: the first goal comes from the stale stream and is discarded; start angle = first variate of the fresh stream,
    // goal from the variates after it; the stream is then restarted and advanced by the start-angle draw (App. A.6-Q4).
    // Unseeded: goal, start, goal, start on the one running stream.
    const bool via = c.env_kind == FG_ENV_VIAPOINT_REACHER;
    const double start = via ? kPi / 2 : 0.0;       // simple_reacher.py:29 starts at zeros
    auto goals = [&]() {
      if (via) {
        if (c.has_fixed[0]) { ctx[0] = c.fixed[0]; ctx[1] = c.fixed[1]; }
        else draw_in_ring(0.5 * total, -1.0, 0.5 * total, ctx[0], ctx[1]);            // norm(via) >= 0.5*total rejected
        if (c.has_fixed[2]) { ctx[2] = c.fixed[2]; ctx[3] = c.fixed[3]; }
        else draw_in_ring(total, 0.5 * total, total, ctx[2], ctx[3]);
      } else {
        if (c.has_fixed[0]) { ctx[0] = c.fixed[0]; ctx[1] = c.fixed[1]; }
        else draw_in_ring(total, -1.0, total, ctx[0], ctx[1]);
      }
    };
    if (io.reseed) {
      q0 = first_joint(start);
      goals();
      g.seed(seed);
      first_joint(start);
    } else {
      goals();
      first_joint(start);
      goals();
      q0 = first_joint(start);
    }
  }
  g.store(io.rng_state + b * 5);

  // ---- state ----
  for (int i = 0; i < N; ++i) {
    io.q[b * N + i] = i == 0 ? q0 : 0.0;
    io.v[b * N + i] = 0.0;
  }
  io.steps[b] = 0;
  io.done[b] = 0;
#pragma unroll
  for (int i = 0; i < 4; ++i) io.ctx[b * 4 + i] = ctx[i];

  // ---- initial observation (_get_obs of the three envs, float64 -> float32), context-masked ----
  float obs[FG_MAX_OBS];
  const double cq = cos(q0), sq = sin(q0);
  double ex = 0.0, ey = 0.0;
  for (int i = 0; i < N; ++i) {       // every link has the absolute angle q0
    ex += cq;
    ey += sq;
    obs[i] = i == 0 ? (float)cq : 1.0f;
    obs[N + i] = i == 0 ? (float)sq : 0.0f;
    obs[2 * N + i] = 0.0f;
  }
  int no = 3 * N;
  no += obs_tail(c.env_kind, ctx, ex, ey, obs + no);
  obs[no++] = 0.0f;                       // steps
  if (c.time_aware) obs[no++] = 0.0f;     // elapsed / max_episode_steps
  if (io.obs)
    for (int j = 0; j < c.n_obs_out; ++j) io.obs[b * c.n_obs_out + j] = obs[c.obs_index[j]];
}

}  // namespace fg
