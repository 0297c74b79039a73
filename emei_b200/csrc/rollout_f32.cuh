// Fused T-step rollouts (float32): cart-pole / analytic inverted-pendulum family and charged ball.
//
// Replaces the canonical caller of step(): the collection loop of zoo/util.py:33-93
//     obs = env.reset(); while not done: a = policy(obs) | action_space.sample(); step; record; ...
// for a batch of independent envs, with gym's TimeLimit (register_env.py max_episode_steps: truncated when
// the episode step count reaches the limit) and auto-reset (zoo/util.py:52-54) done in-kernel.
//
// One thread owns its envs (two for the cart-pole family, whose pair shares packed f32x2 arithmetic; one for
// the charged ball) for the whole horizon: state, episode step counter and
// episode return live in registers across all T steps, so HBM is touched only for what the caller asks
// for -- the action stream (teacher-forced policy) and/or the transition records in the reference's
// dataset layout (observations, next_observations, actions, rewards, dones, timeouts; zoo/util.py:62-67).
// With the built-in uniform random policy and no records a rollout moves < 100 bytes per env in total.
//
// Arithmetic per step is the step kernels' (cartpole_f32.cuh / charged_ball_f32.cuh): a rollout equals T
// calls of emei_*_step_f32 plus the bookkeeping, bit for bit (tests/test_gpu_parity.py).
//
// The kernel is written once over a `Dyn` policy (the env family): Dyn::Buffers (state arrays), Dyn::Regs
// (one env in registers), load/store/observation/step/reset.
#pragma once
#include "rollout.cuh"

namespace emei {

// In-rollout reset sample of one env row.
// Uniform family (cartpole.py:131-132,153-156: U(low, high) per coordinate, + pi on the swing-up angle): the lean
// float32 sampler of the rollout kernels -- ONE Philox block per reset, coordinate c = fma(high - low, u_c, low)
// with u_c the top 24 bits of word c.  A reset is a divergent branch that a third of all warp-steps take under
// the random policy, so its length is paid by the whole warp: the 53-bit double construction of the init kernels
// (two blocks, four double conversions) cost ~360 warp instructions per event, this one ~110
// (mirror: oracle/rollout_oracle.py reset_sample_uniform).
// Gaussian family (mujoco_env.py:137-140): the arithmetic of init_gaussian_kernel (kernels.cuh).
static __device__ __noinline__ float4 rollout_init_state(const RolloutConsts<4>& r, unsigned long long env, unsigned long long seed) {
  float v[4];
  if (r.init_kind == 0) {
    uint32_t w[4];
    Philox::generate(seed, env, 0u, kPurposeRolloutReset, w);
    const float lo = static_cast<float>(r.init_low), span = static_cast<float>(r.init_high) - lo;
#pragma unroll
    for (int c = 0; c < 4; ++c) {
      v[c] = fmaf(span, static_cast<float>(w[c] >> 8) * (1.0f / 16777216.0f), lo);
      if (c == r.init_pi_column) v[c] = static_cast<float>(static_cast<double>(v[c]) + 3.141592653589793238462643383279502884);
    }
  } else {
#pragma unroll
    for (int pr = 0; pr < 2; ++pr) gaussian_initial_pair<float>(r.mean, r.sigma, seed, env, pr, v[2 * pr], v[2 * pr + 1]);
  }
  return make_float4(v[0], v[1], v[2], v[3]);
}

// same arithmetic as init_charged_ball_kernel<float> (kernels.cuh; charged_ball.py:84-94), one env
static __device__ __noinline__ CBRegs rollout_init_charged_ball(float radius, unsigned long long env, unsigned long long seed) {
  CBRegs e;
  float f[4];
  charged_ball_initial_sample<float>(seed, env, radius, e.theta, e.omega, f);
  e.on = true;
  e.f = make_float4(f[0], f[1], f[2], f[3]);
  cb_prepare(e);
  return e;
}

// w[j] for a run-time j without putting the array in local memory
__device__ __forceinline__ uint32_t select_word(const uint32_t (&w)[4], unsigned j) {
  const uint32_t lo = (j & 1u) ? w[1] : w[0], hi = (j & 1u) ? w[3] : w[2];
  return (j & 2u) ? hi : lo;
}

__device__ __forceinline__ double block_sum_double(double v, double* smem /*[kBlock/32]*/) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) smem[warp] = v;
  __syncthreads();
  double t = lane < kBlock / 32 ? smem[lane] : 0.0;
  return warp_sum(t);  // valid in every lane of every warp
}

// ------------------------------------------------------------------------------------------------
// env families
// ------------------------------------------------------------------------------------------------
template <bool IP, int AK, int FR>
struct CartPoleDyn {
  using Consts = CartPoleF32Consts;
  using ActT = typename ActionStorage<AK>::type;
  static constexpr bool kDiscrete = AK <= EMEI_ACTION_DISCRETE_I64;
  // TWO envs per thread: the dynamics of the pair run in packed f32x2 registers (the step kernel's arithmetic,
  // f32::cartpole_integrate<f2>), which halves the issue slots of the integration; policy, TimeLimit bookkeeping and
  // resets stay per env.
  static constexpr int kEnvsPerThread = 2;
  static constexpr bool kSpareReset = true;  // resets are frequent and per env: keep the next sample ready (kernel comment)
  static constexpr int kMinBlocks = 3;  // 80 registers, no spills; 4 CTAs/SM (64 registers, 128 B of spills) measured the same 101 G env-steps/s
  struct Buffers {
    float4* state;
  };
  struct Regs {
    float4 y;
  };
  __device__ __forceinline__ static void load(Regs& e, const Buffers& b, uint32_t i) { e.y = b.state[i]; }
  __device__ __forceinline__ static void blank(Regs& e) { e.y = make_float4(0.f, 0.f, 0.f, 0.f); }
  __device__ __forceinline__ static void store(const Regs& e, const Buffers& b, uint32_t i) { b.state[i] = e.y; }
  __device__ __forceinline__ static float4 observation(const Regs& e) {
    return IP ? make_float4(e.y.x, wrap_pi_f32(e.y.y), e.y.z, e.y.w) : e.y;
  }
  // one step of the pair: same bits as two lanes of cartpole_step_f32_tma_kernel / as cartpole_step_one per env
  __device__ __forceinline__ static void step(Regs (&e)[2], const float (&a)[2], const Consts& k, float (&rew)[2],
                                              bool (&terminated)[2], float4 (&next_obs)[2]) {
    using f32::f2;
    const uint32_t flip = ip_flip(IP, k.variant);
    const float fa = action_to_f_mt<IP, AK>(a[0], k), fb = action_to_f_mt<IP, AK>(a[1], k);
    const float4 ya = e[0].y, yb = e[1].y;
    f2 X = f32::f2_pack(ya.x, yb.x), V, TH, W = f32::f2_pack(ya.w, yb.w);
    if constexpr (!IP) {
      V = f32::f2_pack(ya.y, yb.y);
      TH = f32::f2_pack(ya.z, yb.z);
    } else {
      TH = f32::f2_pack(ya.y, yb.y);
      V = f32::f2_pack(ya.z, yb.z);
    }
    const float th0a = fabsf(IP ? ya.y : ya.z), th0b = fabsf(IP ? yb.y : yb.z);
    f32::LaneMax<f2> dmax;
    const f2 C = f32::cartpole_integrate<f2, FR>(X, V, TH, W, f32::f2_pack(-fa, -fb), flip, k.k, k.freq_rate, dmax);
    float4 na, nb;
    {
      float t0, t1;
      f32::f2_unpack(X, na.x, nb.x);
      f32::f2_unpack(W, na.w, nb.w);
      f32::f2_unpack(V, t0, t1);
      if constexpr (!IP) { na.y = t0; nb.y = t1; } else { na.z = t0; nb.z = t1; }
      f32::f2_unpack(TH, t0, t1);
      if constexpr (!IP) { na.z = t0; nb.z = t1; } else { na.y = t0; nb.y = t1; }
    }
    float ca, cb;
    f32::f2_unpack(C, ca, cb);
    if constexpr (IP) {
      ca = f32::u2f(f32::f2u(ca) ^ flip);
      cb = f32::u2f(f32::f2u(cb) ^ flip);
    }
    const bool ok_a = th0a <= f32::kSinCosSaneMax && dmax.a <= f32::kDeltaMax;
    const bool ok_b = th0b <= f32::kSinCosSaneMax && dmax.b <= f32::kDeltaMax;
    if (!(ok_a && ok_b)) {  // cold: the integrator's guard tripped (f32math.cuh)
      if (!ok_a) {
        na = integrate_libm<IP, FR>(ya, fa, flip, k.k, k.freq_rate, &ca);
        if constexpr (IP) ca = f32::u2f(f32::f2u(ca) ^ flip);
      }
      if (!ok_b) {
        nb = integrate_libm<IP, FR>(yb, fb, flip, k.k, k.freq_rate, &cb);
        if constexpr (IP) cb = f32::u2f(f32::f2u(cb) ^ flip);
      }
    }
    bool nd_a, nd_b;
    cartpole_outcome<IP>(na, ca, k, rew[0], nd_a, next_obs[0]);
    cartpole_outcome<IP>(nb, cb, k, rew[1], nd_b, next_obs[1]);
    e[0].y = na;
    e[1].y = nb;
    terminated[0] = !nd_a;
    terminated[1] = !nd_b;
  }
  __device__ __forceinline__ static void reset(Regs& e, const RolloutConsts<4>& r, const Consts&, unsigned long long env, unsigned long long seed) {
    e.y = rollout_init_state(r, env, seed);
  }
  __device__ __forceinline__ static float4 pack(const Regs& e) { return e.y; }
  __device__ __forceinline__ static void unpack(Regs& e, const float4& v) { e.y = v; }
};

struct ChargedBallBuffers {
  uint8_t* on_circle;
  float2* circle;
  float4* free_state;
};

// FR: compile-time sub-step count (0 = k.freq_rate at run time)
template <int AK, int FR>
struct ChargedBallDyn {
  using Consts = ChargedBallF32Consts;
  using ActT = typename ActionStorage<AK>::type;
  static constexpr bool kDiscrete = AK <= EMEI_ACTION_DISCRETE_I64;
  static constexpr int kMinBlocks = 4;
  using Buffers = ChargedBallBuffers;
  using Regs = CBRegs;
  static constexpr int kEnvsPerThread = 1;
  static constexpr bool kSpareReset = false;  // the charged ball never terminates: every env resets at the same TimeLimit step
  __device__ __forceinline__ static void blank(Regs&) {}
  __device__ __forceinline__ static void load(Regs& e, const Buffers& b, uint32_t i) {
    e.on = b.on_circle[i] != 0;
    const float2 c2 = b.circle[i];
    e.theta = c2.x;
    e.omega = c2.y;
    e.f = b.free_state[i];
    cb_prepare(e);
  }
  __device__ __forceinline__ static void store(const Regs& e, const Buffers& b, uint32_t i) {
    b.on_circle[i] = e.on ? 1 : 0;
    b.circle[i] = make_float2(e.theta, e.omega);
    b.free_state[i] = e.f;
  }
  __device__ __forceinline__ static float4 observation(const Regs& e) { return e.f; }  // charged_ball.py:96-97
  __device__ __forceinline__ static void step(Regs (&e)[1], const float (&a)[1], const Consts& k, float (&rew)[1],
                                              bool (&terminated)[1], float4 (&next_obs)[1]) {
    rew[0] = cb_env_step<FR>(e[0], cb_field<AK>(a[0], k), k);
    terminated[0] = false;  // charged_ball.py:110-111
    next_obs[0] = e[0].f;
  }
  __device__ __forceinline__ static void reset(Regs& e, const RolloutConsts<4>&, const Consts& k, unsigned long long env, unsigned long long seed) {
    e = rollout_init_charged_ball(k.r, env, seed);
  }
  __device__ __forceinline__ static float4 pack(const Regs& e) { return e.f; }  // unused (kSpareReset = false)
  __device__ __forceinline__ static void unpack(Regs&, const float4&) {}
};

// ------------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------------
// One thread owns E = Dyn::kEnvsPerThread envs for the whole horizon: envs i0 + e * kBlock of its CTA's block of
// E * kBlock envs (every access stays coalesced per e).
template <class Dyn, bool RECORD>
__global__ void __launch_bounds__(kBlock, Dyn::kMinBlocks)
    rollout_f32_kernel(const typename Dyn::Buffers b, const RolloutIO<float> io, uint32_t n, const typename Dyn::Consts k,
                       const RolloutConsts<4> r) {
  using ActT = typename Dyn::ActT;
  constexpr int E = Dyn::kEnvsPerThread;
  const uint32_t i0 = blockIdx.x * (kBlock * E) + threadIdx.x;
  const ActT* __restrict__ act_in = static_cast<const ActT*>(io.actions);
  ActT* __restrict__ act_out = static_cast<ActT*>(io.rec_act);

  // reward sums in double: a thread's partial sums must not depend on how a horizon is split into launches
  double r_sum = 0.0, fin_ret = 0.0;
  unsigned n_term = 0, n_trunc = 0, n_fin = 0, fin_len = 0;
  // Spare reset samples (families whose episodes end at different steps in different envs).  A reset is a divergent
  // call of ~110 warp instructions (one Philox block + conversions; the Gaussian family: two blocks, log, sqrt,
  // sincospi in double), and under a random policy 36 % of the 32-env warp-steps hold at least one env that needs it,
  // so every env-step paid ~45 instructions for an event that 1.4 % of them take.  The sample of an env's NEXT
  // episode depends only on (seed, env, episode index + 1), so it is drawn ahead of time, all lanes of a warp that
  // lack one in the same pass every kSpareWindow steps, and parked in shared memory; a reset is then one 128-bit
  // load, and only an env that ends two episodes inside one window takes the divergent call.  Same samples, same bits.
  constexpr bool SPARE = Dyn::kSpareReset;
  constexpr int kSpareWindow = 16;
  __shared__ float4 s_spare[SPARE ? E : 1][SPARE ? kBlock : 1];
  const bool use_spare = SPARE && r.auto_reset && r.horizon >= kSpareWindow;
  const int max_steps = r.max_episode_steps > 0 ? r.max_episode_steps : 0x7fffffff;  // gym TimeLimit; 0 = none
  pdl_trigger();
  pdl_wait();
  if (i0 < n) {
    typename Dyn::Regs ev[E];
    uint32_t idx[E];
    bool live[E];
    int ep_step[E], ep_idx[E];
    float ep_ret[E], a_next[E];
    uint32_t w[E][4], cur[E];
    bool have_spare[E];
#pragma unroll
    for (int e = 0; e < E; ++e) {
      cur[e] = 0u;
      have_spare[e] = false;
      idx[e] = i0 + static_cast<uint32_t>(e) * kBlock;
      live[e] = idx[e] < n;
      ep_step[e] = ep_idx[e] = 0;
      ep_ret[e] = a_next[e] = 0.f;
      w[e][0] = w[e][1] = w[e][2] = w[e][3] = 0u;
      if (live[e]) {
        Dyn::load(ev[e], b, idx[e]);
        ep_step[e] = io.ep_step[idx[e]];
        ep_ret[e] = io.ep_return[idx[e]];
        ep_idx[e] = io.ep_index[idx[e]];
        if (!r.random_policy) a_next[e] = static_cast<float>(__ldg(act_in + idx[e]));
      } else {
        Dyn::blank(ev[e]);  // a dead lane of the pair computes on zeros; nothing of it is stored or counted
      }
    }
    const uint32_t t0_lo = static_cast<uint32_t>(r.t0);  // positions inside a Philox block need the low bits only
    for (int t = 0; t < r.horizon; ++t) {
      float a[E];
      const uint32_t tl = t0_lo + static_cast<uint32_t>(t);  // low word of the global step r.t0 + t (uniform)
      if constexpr (SPARE) {
        if (use_spare && (t & (kSpareWindow - 1)) == 0) {  // uniform
#pragma unroll
          for (int e = 0; e < E; ++e) {
            if (live[e] && !have_spare[e]) {
              typename Dyn::Regs nxt = ev[e];
              Dyn::reset(nxt, r, k, r.env_offset + idx[e], reset_seed(r.seed_reset, ep_idx[e] + 1));
              s_spare[e][threadIdx.x] = Dyn::pack(nxt);
              have_spare[e] = true;
            }
          }
        }
      }
#pragma unroll
      for (int e = 0; e < E; ++e) {
        // ---- policy
        if (r.random_policy) {  // env.action_space.sample() (zoo/util.py:57): Discrete(2) bit / Box uniform
          // counter-based stream per (seed_action, env): Discrete(2) consumes ONE bit per step (a 128-bit Philox
          // block lasts 128 steps: block tg >> 7, word (tg >> 5) & 3, bit tg & 31), Box one 32-bit word per step
          // (block tg >> 2, word tg & 3, top 24 bits -> [low, high)).  The refresh tests depend on the step number
          // only, so they are uniform branches; between refreshes a Discrete step costs a mask and a shift of the
          // current word.  rollout_ref_kernel keeps its own copy of this stream (DESIGN.md 4.6).
          if constexpr (Dyn::kDiscrete) {
            if (t == 0 || (tl & 31u) == 0) {
              if (t == 0 || (tl & 127u) == 0)
                Philox::generate(r.seed_action, r.env_offset + idx[e],
                                 static_cast<uint32_t>((r.t0 + static_cast<unsigned long long>(t)) >> 7), kPurposeRolloutAction, w[e]);
              cur[e] = select_word(w[e], (tl >> 5) & 3u) >> (tl & 31u);
            }
            a[e] = static_cast<float>(cur[e] & 1u);
            cur[e] >>= 1;
          } else {
            if (t == 0 || (tl & 3u) == 0)
              Philox::generate(r.seed_action, r.env_offset + idx[e],
                               static_cast<uint32_t>((r.t0 + static_cast<unsigned long long>(t)) >> 2), kPurposeRolloutAction, w[e]);
            const uint32_t word = select_word(w[e], tl & 3u);
            a[e] = fmaf(r.act_high - r.act_low, static_cast<float>(word >> 8) * (1.0f / 16777216.0f), r.act_low);
          }
        } else {
          a[e] = a_next[e];
          if (live[e] && t + 1 < r.horizon) a_next[e] = static_cast<float>(__ldg(act_in + static_cast<size_t>(t + 1) * n + idx[e]));
        }
        if constexpr (RECORD) {
          if (live[e]) {
            const size_t rec = static_cast<size_t>(t) * n + idx[e];
            reinterpret_cast<float4*>(io.rec_obs)[rec] = Dyn::observation(ev[e]);
            act_out[rec] = static_cast<ActT>(a[e]);
          }
        }
      }
      // ---- dynamics + reward + terminal (the step kernel's arithmetic)
      float rew[E];
      bool terminated[E];
      float4 next_obs[E];
      Dyn::step(ev, a, k, rew, terminated, next_obs);
#pragma unroll
      for (int e = 0; e < E; ++e) {
        if (!live[e]) continue;
        // ---- TimeLimit + bookkeeping (zoo/util.py:58-73; gym TimeLimit: truncated = elapsed >= max)
        ep_step[e] += 1;
        ep_ret[e] += rew[e];
        const bool truncated = ep_step[e] >= max_steps;
        const bool done = terminated[e] || truncated;
        if constexpr (RECORD) {
          const size_t rec = static_cast<size_t>(t) * n + idx[e];
          reinterpret_cast<float4*>(io.rec_next)[rec] = next_obs[e];
          io.rec_rew[rec] = rew[e];
          io.rec_done[rec] = done ? 1 : 0;
          io.rec_timeout[rec] = truncated ? 1 : 0;
        }
        r_sum += static_cast<double>(rew[e]);
        if (done) {
          n_term += terminated[e] ? 1u : 0u;
          n_trunc += truncated ? 1u : 0u;
          if (r.auto_reset) {
            n_fin += 1u;
            fin_ret += static_cast<double>(ep_ret[e]);
            fin_len += static_cast<unsigned>(ep_step[e]);
            ep_idx[e] += 1;
            if (SPARE && have_spare[e]) {  // the sample drawn ahead of time for exactly this episode index
              Dyn::unpack(ev[e], s_spare[e][threadIdx.x]);
              have_spare[e] = false;
            } else {
              Dyn::reset(ev[e], r, k, r.env_offset + idx[e], reset_seed(r.seed_reset, ep_idx[e]));
            }
            ep_step[e] = 0;
            ep_ret[e] = 0.f;
          }
        }
      }
    }
#pragma unroll
    for (int e = 0; e < E; ++e) {
      if (!live[e]) continue;
      Dyn::store(ev[e], b, idx[e]);
      io.ep_step[idx[e]] = ep_step[e];
      io.ep_return[idx[e]] = ep_ret[e];
      io.ep_index[idx[e]] = ep_idx[e];
    }
  }
  if (io.stats != nullptr) {  // uniform across the grid
    __shared__ double s_red[kBlock / 32];
    const double vals[6] = {r_sum, static_cast<double>(n_term), static_cast<double>(n_trunc),
                            static_cast<double>(n_fin), fin_ret, static_cast<double>(fin_len)};
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      const double tot = block_sum_double(vals[j], s_red);
      if (threadIdx.x == 0) atomicAdd(&io.stats[j], tot);
    }
  }
}

template <class Dyn>
inline void launch_rollout(const typename Dyn::Buffers& b, const RolloutIO<float>& io, int64_t n, const typename Dyn::Consts& k,
                           const RolloutConsts<4>& r, cudaStream_t s) {
  const int grid = grid_for(n, kBlock * Dyn::kEnvsPerThread);
  if (io.rec_obs != nullptr)
    launch_pdl(rollout_f32_kernel<Dyn, true>, grid, kBlock, s, b, io, static_cast<uint32_t>(n), k, r);
  else
    launch_pdl(rollout_f32_kernel<Dyn, false>, grid, kBlock, s, b, io, static_cast<uint32_t>(n), k, r);
}

template <bool IP, int FR>
inline void launch_cartpole_rollout(int ak, float* state, const RolloutIO<float>& io, int64_t n, const CartPoleF32Consts& k,
                                    const RolloutConsts<4>& r, cudaStream_t s) {
  float4* st = reinterpret_cast<float4*>(state);
  switch (ak) {
#define EMEI_AK(A)                                                           \
  case A: {                                                                  \
    typename CartPoleDyn<IP, A, FR>::Buffers b = {st};                       \
    launch_rollout<CartPoleDyn<IP, A, FR>>(b, io, n, k, r, s);               \
  } break;
    EMEI_AK(EMEI_ACTION_DISCRETE_U8)
    EMEI_AK(EMEI_ACTION_DISCRETE_I32)
    EMEI_AK(EMEI_ACTION_DISCRETE_I64)
    EMEI_AK(EMEI_ACTION_CONTINUOUS_F32)
    EMEI_AK(EMEI_ACTION_CONTINUOUS_F64)
#undef EMEI_AK
  }
}

inline void launch_charged_ball_rollout(int ak, uint8_t* on_circle, float* circle, float* free_state, const RolloutIO<float>& io,
                                        int64_t n, const ChargedBallF32Consts& k, const RolloutConsts<4>& r, cudaStream_t s) {
  switch (ak) {
#define EMEI_AK(A)                                                                                                       \
  case A: {                                                                                                              \
    ChargedBallBuffers b = {on_circle, reinterpret_cast<float2*>(circle), reinterpret_cast<float4*>(free_state)}; \
    if (k.freq_rate == 1) launch_rollout<ChargedBallDyn<A, 1>>(b, io, n, k, r, s); /* BASELINE configs[3]: no sub-step loop */ \
    else launch_rollout<ChargedBallDyn<A, 0>>(b, io, n, k, r, s);                                                         \
  } break;
    EMEI_AK(EMEI_ACTION_DISCRETE_U8)
    EMEI_AK(EMEI_ACTION_DISCRETE_I32)
    EMEI_AK(EMEI_ACTION_DISCRETE_I64)
    EMEI_AK(EMEI_ACTION_CONTINUOUS_F32)
    EMEI_AK(EMEI_ACTION_CONTINUOUS_F64)
#undef EMEI_AK
  }
}

}  // namespace emei
