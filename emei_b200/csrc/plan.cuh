// Sampling-based MPC over the true dynamics (CEM / MPPI, DESIGN.md 4.10): one launch scores B x K candidate action
// sequences of H steps from B start states, one launch refits the [H, B] plan distribution from the returns.
//
// Candidate (b, k) draws its actions from Philox keyed by (seed, (env_offset + b) * 2^32 + k) with purpose kPurposePlanAction
// (host mirror: tests/test_plan.py plan_actions):
//   continuous: step t takes the Box-Muller pair of block t >> 1 (cs for even t, sn for odd t), a = clamp(R(mean + std z))
//               with the product and the sum rounded in double and the clamp in R;
//   discrete:   step t takes word t & 3 of block t >> 2, a = ((w >> 8) 2^-24 < float(p)) ? 1 : 0.
// Per step the arithmetic is the one the env's own rollout() uses for that (family, precision), so a candidate's rewards are
// bit-equal to a teacher-forced rollout of the same actions (the lean float32 cart-pole step, ChargedBallDyn, the reference
// family structs of rollout_ref.cuh).  The return sum_{t<H} gamma^t r_t is accumulated in double with every operation rounded
// on its own; the reward of the step that terminates counts, later steps do not.
//
// The update regenerates the chosen candidates' actions from the same counters instead of reading them back, so the two
// launches move 8 bytes per candidate between them.
#pragma once
#include <type_traits>

#include "rollout_ref.cuh"
#include "trajectory.cuh"

namespace emei {

constexpr int kPlanMaxCandidates = 4096;

// the kernel form of emei_plan_params
struct PlanConsts {
  unsigned long long seed, env_offset;
  double gamma, temperature, momentum, min_std;
  float low, high;
  int method, elites, kind;
};

inline int check_plan_params(const emei_plan_params& q, int64_t K) {
  if (!action_kind_valid(q.action_kind)) return EMEI_ERR_BAD_ACTION_KIND;
  if (q.method != EMEI_PLAN_CEM && q.method != EMEI_PLAN_MPPI) return EMEI_ERR_BAD_PARAM;
  if (q.method == EMEI_PLAN_CEM && (q.elites < 1 || q.elites > K)) return EMEI_ERR_BAD_PARAM;
  if (q.method == EMEI_PLAN_MPPI && !(q.temperature > 0.0)) return EMEI_ERR_BAD_PARAM;
  if (!(q.gamma >= 0.0 && q.gamma <= 1.0) || !(q.momentum >= 0.0 && q.momentum < 1.0) || !(q.min_std >= 0.0)) return EMEI_ERR_BAD_PARAM;
  if (q.action_kind >= EMEI_ACTION_CONTINUOUS_F32 && !(q.action_low <= q.action_high)) return EMEI_ERR_BAD_PARAM;
  return EMEI_OK;
}

// sizes first (every entry point): B, H >= 0 and 1 <= K <= 4096
inline int check_plan_sizes(int64_t B, int64_t K, int64_t H) {
  if (B < 0 || H < 0 || H > 0x7fffffff || K < 1 || K > kPlanMaxCandidates) return EMEI_ERR_BAD_SIZE;
  return EMEI_OK;
}

inline PlanConsts make_plan_consts(const emei_plan_params& q) {
  return {q.seed, q.env_offset, q.gamma, q.temperature, q.momentum, q.min_std, q.action_low, q.action_high, q.method, q.elites,
          q.action_kind};
}

__device__ __forceinline__ unsigned long long plan_env_word(const PlanConsts& c, int64_t b, int64_t k) {
  return ((c.env_offset + static_cast<unsigned long long>(b)) << 32) | static_cast<unsigned long long>(k);
}

// the continuous action from the step's standard normal z: R(mean + std z) in double, then clamped in R (plan_clamp); a
// float32 action array in a float64 plan holds the float32 rounding of that value, and the step consumes what the array holds
template <typename R>
__device__ __forceinline__ R plan_clamp(R a, const PlanConsts& c) {
  const R lo = static_cast<R>(c.low), hi = static_cast<R>(c.high);
  a = a < lo ? lo : (a > hi ? hi : a);
  if (sizeof(R) == 8 && c.kind == EMEI_ACTION_CONTINUOUS_F32) a = static_cast<R>(static_cast<float>(a));
  return a;
}
template <typename R>
__device__ __forceinline__ R plan_continuous(R mean, R std, double z, const PlanConsts& c) {
  return plan_clamp<R>(static_cast<R>(__dadd_rn(static_cast<double>(mean), __dmul_rn(static_cast<double>(std), z))), c);
}

__device__ __forceinline__ float plan_discrete(uint32_t word, float p) {
  return static_cast<float>(word >> 8) * (1.0f / 16777216.0f) < p ? 1.0f : 0.0f;
}

// The per-candidate random state across steps: one Philox block serves two continuous / four discrete steps.
struct PlanDraw {
  uint32_t w[4];
  double rad, cs, sn;
  template <bool DISC>
  __device__ __forceinline__ void refill(const PlanConsts& c, unsigned long long env, int64_t t) {
    if constexpr (DISC)
      Philox::generate(c.seed, env, static_cast<uint32_t>(t >> 2), kPurposePlanAction, w);
    else
      philox_normal_pair(c.seed, env, static_cast<uint32_t>(t >> 1), kPurposePlanAction, rad, cs, sn);
  }
  template <bool DISC>
  __device__ __forceinline__ static bool starts_block(int64_t t) {
    return DISC ? (t & 3) == 0 : (t & 1) == 0;
  }
  // action of step t (its block drawn): the probability / mean and std of that step
  template <bool DISC, typename R>
  __device__ __forceinline__ R action(const PlanConsts& c, int64_t t, R m, R s) const {
    if constexpr (DISC)
      return static_cast<R>(plan_discrete(select_word(w, static_cast<unsigned>(t) & 3u), static_cast<float>(m)));
    else
      return plan_continuous<R>(m, s, __dmul_rn(rad, (t & 1) ? sn : cs), c);
  }
};

template <typename R>
__device__ __forceinline__ void plan_store(void* p, int64_t i, int kind, R a) {
  switch (kind) {
    case EMEI_ACTION_DISCRETE_U8: static_cast<uint8_t*>(p)[i] = static_cast<uint8_t>(a); break;
    case EMEI_ACTION_DISCRETE_I32: static_cast<int32_t*>(p)[i] = static_cast<int32_t>(a); break;
    case EMEI_ACTION_DISCRETE_I64: static_cast<long long*>(p)[i] = static_cast<long long>(a); break;
    case EMEI_ACTION_CONTINUOUS_F32: static_cast<float*>(p)[i] = static_cast<float>(a); break;
    default: static_cast<double*>(p)[i] = static_cast<double>(a); break;
  }
}

// ---------------------------------------------------------------------------------------------
// families: the start state's load and the rollout's step of one env, given the action value the array would hold; the
// observation of the start state (observe) and of every state a step reaches (step's o) is the one the env's step()
// returns there (the closed-loop policies of policy.cuh act on it; the plan eval discards it)
// ---------------------------------------------------------------------------------------------
struct PlanRowsF32 {
  const float* rows;
};
struct PlanChargedBallF32State {
  const uint8_t* on_circle;
  const float* circle;
  const float* free_state;
};

template <bool IP, int FR, bool DISC>
struct PlanCartPoleF32 {  // the lean float32 step of emei_cartpole_rollout_f32 (cartpole_step_one == a lane of its pair)
  using Real = float;
  using Consts = CartPoleF32Consts;
  using Regs = float4;
  using State = PlanRowsF32;
  static constexpr int AK = DISC ? EMEI_ACTION_DISCRETE_U8 : EMEI_ACTION_CONTINUOUS_F32;
  static constexpr int kObs = 4;
  __device__ __forceinline__ static void load(Regs& y, const State& s, int64_t b) { y = reinterpret_cast<const float4*>(s.rows)[b]; }
  // the observation step() would return in state y (CartPoleDyn::observation)
  __device__ __forceinline__ static void observe(const Regs& y, const Consts&, float (&o)[kObs]) {
    o[0] = y.x, o[1] = IP ? wrap_pi_f32(y.y) : y.y, o[2] = y.z, o[3] = y.w;
  }
  __device__ __forceinline__ static float step(Regs& y, float a, const Consts& k, bool& terminated, float (&o)[kObs]) {
    float rew;
    bool notdone;
    float4 obs;
    cartpole_step_one<IP, FR>(y, action_to_f_mt<IP, AK>(a, k), ip_flip(IP, k.variant), k, rew, notdone, obs);
    terminated = !notdone;
    o[0] = obs.x, o[1] = obs.y, o[2] = obs.z, o[3] = obs.w;
    return rew;
  }
  __device__ __forceinline__ static float step(Regs& y, float a, const Consts& k, bool& terminated) {
    float o[kObs];
    return step(y, a, k, terminated, o);
  }
};

template <int FR, bool DISC>
struct PlanChargedBallF32 {  // the load and step of ChargedBallDyn (emei_charged_ball_rollout_f32)
  using Real = float;
  static constexpr int AK = DISC ? EMEI_ACTION_DISCRETE_U8 : EMEI_ACTION_CONTINUOUS_F32;
  using Consts = ChargedBallF32Consts;
  using Regs = CBRegs;
  using State = PlanChargedBallF32State;
  __device__ __forceinline__ static void load(Regs& e, const State& s, int64_t b) {
    e.on = s.on_circle[b] != 0;
    const float2 c2 = reinterpret_cast<const float2*>(s.circle)[b];
    e.theta = c2.x;
    e.omega = c2.y;
    e.f = reinterpret_cast<const float4*>(s.free_state)[b];
    cb_prepare(e);
  }
  static constexpr int kObs = 4;
  __device__ __forceinline__ static void observe(const Regs& e, const Consts&, float (&o)[kObs]) {
    o[0] = e.f.x, o[1] = e.f.y, o[2] = e.f.z, o[3] = e.f.w;  // charged_ball.py:96-97
  }
  __device__ __forceinline__ static float step(Regs& e, float a, const Consts& k, bool& terminated, float (&o)[kObs]) {
    terminated = false;  // charged_ball.py:110-111
    const float rew = cb_env_step<FR>(e, cb_field<AK>(a, k), k);
    observe(e, k, o);
    return rew;
  }
  __device__ __forceinline__ static float step(Regs& e, float a, const Consts& k, bool& terminated) {
    float o[kObs];
    return step(e, a, k, terminated, o);
  }
};

// the reference-arithmetic families of rollout_ref.cuh (float64 cart-pole / IP / charged ball, I2P in both precisions)
template <class Fam, bool DISC>
struct PlanRef {
  using Real = typename Fam::Real;
  using Consts = typename Fam::Consts;
  using Regs = typename Fam::Regs;
  using State = typename Fam::Buffers;
  using ActC = std::conditional_t<DISC, uint8_t, Real>;  // the element the drive reads, as a teacher-forced rollout does
  static constexpr int AK = DISC ? EMEI_ACTION_DISCRETE_U8 : (sizeof(Real) == 4 ? EMEI_ACTION_CONTINUOUS_F32 : EMEI_ACTION_CONTINUOUS_F64);
  static constexpr int kObs = Fam::kObs;
  __device__ __forceinline__ static void load(Regs& e, const State& s, int64_t b) { Fam::load(e, s, b); }
  __device__ __forceinline__ static void observe(const Regs& e, const Consts& k, Real (&o)[kObs]) { Fam::observation(e, k, o); }
  __device__ __forceinline__ static Real step(Regs& e, Real a, const Consts& k, bool& terminated, Real (&o)[kObs]) {
    const ActC av = static_cast<ActC>(a);
    RefAction ra;
    ra.value = 0.f;
    ra.index = 0;
    const NoiseConsts z = {};
    Real rew;
    Fam::step(e, Fam::drive(k, &av, ra, AK), k, z, 0ull, 0ull, rew, terminated, o);
    return rew;
  }
  __device__ __forceinline__ static Real step(Regs& e, Real a, const Consts& k, bool& terminated) {
    Real o[kObs];
    return step(e, a, k, terminated, o);
  }
};

// ---------------------------------------------------------------------------------------------
// eval: one candidate per thread, k fastest (a warp shares b: the mean / std loads are broadcasts)
// ---------------------------------------------------------------------------------------------
template <class F, bool DISC>
__global__ void __launch_bounds__(kBlock)
    plan_eval_kernel(const typename F::State s, const typename F::Real* __restrict__ mean, const typename F::Real* __restrict__ std,
                     double* __restrict__ returns, void* __restrict__ actions_out, int64_t B, int64_t K, int64_t H, const PlanConsts c,
                     const typename F::Consts k) {
  using R = typename F::Real;
  const int64_t n = B * K;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * kBlock;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x; i < n; i += stride) {
    const int64_t b = i / K;
    const unsigned long long env = plan_env_word(c, b, i - b * K);
    typename F::Regs e;
    F::load(e, s, b);
    R m = mean[b], sd = DISC ? R(0) : std[b];
    double ret = 0.0, disc = 1.0;
    bool live = true;
    PlanDraw d;
    for (int64_t t = 0; t < H; ++t) {
      R m_next = R(0), sd_next = R(0);  // step t+1's distribution, requested before step t's math
      if (t + 1 < H) {
        m_next = mean[(t + 1) * B + b];
        if (!DISC) sd_next = std[(t + 1) * B + b];
      }
      if (PlanDraw::starts_block<DISC>(t)) d.refill<DISC>(c, env, t);
      const R a = d.action<DISC, R>(c, t, m, sd);
      if (actions_out != nullptr) plan_store<R>(actions_out, t * n + i, c.kind, a);
      if (live) {
        bool terminated;
        const R rew = F::step(e, a, k, terminated);
        ret = __dadd_rn(ret, __dmul_rn(disc, static_cast<double>(rew)));
        disc = __dmul_rn(disc, c.gamma);
        if (terminated) {
          live = false;
          if (actions_out == nullptr) break;
        }
      }
      m = m_next, sd = sd_next;
    }
    returns[i] = ret;
  }
}

template <class F, bool DISC, typename C>
inline void launch_plan_eval(const typename F::State& s, const typename F::Real* mean, const typename F::Real* std, double* returns,
                             void* actions_out, int64_t B, int64_t K, int64_t H, const PlanConsts& c, const C& k, cudaStream_t st) {
  plan_eval_kernel<F, DISC><<<resident_grid(plan_eval_kernel<F, DISC>, B * K), kBlock, 0, st>>>(s, mean, std, returns, actions_out, B, K,
                                                                                                 H, c, k);
}

// the checks every eval entry point applies, in order, after its own family's params check
template <typename R>
inline int plan_eval_args(const R* mean, const R* std, double* returns, const emei_plan_params& q) {
  EMEI_CHECK_PTR(mean);
  EMEI_CHECK_PTR(returns);
  if (q.action_kind >= EMEI_ACTION_CONTINUOUS_F32) EMEI_CHECK_PTR(std);
  return EMEI_OK;
}

template <typename R>
int cartpole_plan_eval(const R* state0, const R* mean, const R* std, double* returns, void* actions_out, int64_t B, int64_t K, int64_t H,
                       const emei_plan_params* q, const emei_cartpole_params* p, emei_stream_t stream) {
  if (const int e = check_plan_sizes(B, K, H)) return e;
  EMEI_CHECK_PTR(q);
  EMEI_CHECK_PTR(p);
  if (const int e = check_cartpole_params(*p)) return e;
  if (const int e = check_plan_params(*q, K)) return e;
  if (B == 0 || H == 0) return EMEI_OK;
  EMEI_CHECK_PTR(state0);
  if (const int e = plan_eval_args(mean, std, returns, *q)) return e;
  EMEI_CHECK_ALIGN16(state0);
  emei_cartpole_params pk = *p;
  pk.action_kind = q->action_kind;  // the plan's actions drive the step
  const PlanConsts c = make_plan_consts(*q);
  const bool disc = q->action_kind <= EMEI_ACTION_DISCRETE_I64, ip = p->variant >= EMEI_IP_REBOUND_BALANCING;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if constexpr (sizeof(R) == 4) {  // the float32 rollout's instantiations (emei_cartpole_rollout_f32)
#define EMEI_GO(IPV, FRV)                                                                                                         \
  do {                                                                                                                            \
    const PlanRowsF32 s = {state0};                                                           \
    const CartPoleF32Consts k = make_cartpole_f32_consts(pk);                                                                     \
    if (disc) launch_plan_eval<PlanCartPoleF32<IPV, FRV, true>, true>(s, mean, std, returns, actions_out, B, K, H, c, k, st);   \
    else launch_plan_eval<PlanCartPoleF32<IPV, FRV, false>, false>(s, mean, std, returns, actions_out, B, K, H, c, k, st);      \
  } while (0)
    if (!ip) {
      if (p->freq_rate == 1) EMEI_GO(false, 1);
      else if (p->freq_rate == 4) EMEI_GO(false, 4);
      else EMEI_GO(false, 0);
    } else {
      if (p->freq_rate == 1) EMEI_GO(true, 1);
      else if (p->freq_rate == 4) EMEI_GO(true, 4);
      else EMEI_GO(true, 0);
    }
#undef EMEI_GO
  } else {
    const CartPoleConsts<R> k = make_cartpole_consts<R>(pk);
#define EMEI_GO(IPV)                                                                                                              \
  do {                                                                                                                            \
    const typename RefCartPole<R, IPV>::Buffers s = {const_cast<R*>(state0)};                                                     \
    if (disc) launch_plan_eval<PlanRef<RefCartPole<R, IPV>, true>, true>(s, mean, std, returns, actions_out, B, K, H, c, k, st);  \
    else launch_plan_eval<PlanRef<RefCartPole<R, IPV>, false>, false>(s, mean, std, returns, actions_out, B, K, H, c, k, st);     \
  } while (0)
    if (ip) EMEI_GO(true); else EMEI_GO(false);
#undef EMEI_GO
  }
  return launch_status();
}

template <typename R>
int i2p_plan_eval(const R* state0, const R* mean, const R* std, double* returns, void* actions_out, int64_t B, int64_t K, int64_t H,
                  const emei_plan_params* q, const emei_i2p_params* p, emei_stream_t stream) {
  if (const int e = check_plan_sizes(B, K, H)) return e;
  EMEI_CHECK_PTR(q);
  EMEI_CHECK_PTR(p);
  if (const int e = check_i2p_params(*p)) return e;
  if (const int e = check_plan_params(*q, K)) return e;
  if (q->action_kind <= EMEI_ACTION_DISCRETE_I64) return EMEI_ERR_BAD_ACTION_KIND;  // the double pendulum's tasks act on a Box
  if (B == 0 || H == 0) return EMEI_OK;
  EMEI_CHECK_PTR(state0);
  if (const int e = plan_eval_args(mean, std, returns, *q)) return e;
  EMEI_CHECK_ALIGN16(state0);
  emei_i2p_params pk = *p;
  pk.action_kind = q->action_kind;
  const PlanConsts c = make_plan_consts(*q);
  const I2PConsts<R> k = make_i2p_consts<R>(pk);
  const typename RefI2P<R>::Buffers s = {const_cast<R*>(state0)};
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  launch_plan_eval<PlanRef<RefI2P<R>, false>, false>(s, mean, std, returns, actions_out, B, K, H, c, k, st);
  return launch_status();
}

template <typename R>
int charged_ball_plan_eval(const uint8_t* on_circle, const R* circle, const R* free_state, const R* mean, const R* std, double* returns,
                           void* actions_out, int64_t B, int64_t K, int64_t H, const emei_plan_params* q, const emei_charged_ball_params* p,
                           emei_stream_t stream) {
  if (const int e = check_plan_sizes(B, K, H)) return e;
  EMEI_CHECK_PTR(q);
  EMEI_CHECK_PTR(p);
  if (const int e = check_charged_ball_params(*p)) return e;
  if (const int e = check_plan_params(*q, K)) return e;
  if (B == 0 || H == 0) return EMEI_OK;
  EMEI_CHECK_PTR(on_circle);
  EMEI_CHECK_PTR(circle);
  EMEI_CHECK_PTR(free_state);
  if (const int e = plan_eval_args(mean, std, returns, *q)) return e;
  EMEI_CHECK_ALIGN16(circle);
  EMEI_CHECK_ALIGN16(free_state);
  emei_charged_ball_params pk = *p;
  pk.action_kind = q->action_kind;
  const PlanConsts c = make_plan_consts(*q);
  const bool disc = q->action_kind <= EMEI_ACTION_DISCRETE_I64;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if constexpr (sizeof(R) == 4) {  // emei_charged_ball_rollout_f32's instantiations
    const ChargedBallF32Consts k = make_cb_f32_consts(pk);
#define EMEI_GO(FRV)                                                                                                              \
  do {                                                                                                                            \
    const PlanChargedBallF32State s = {on_circle, circle, free_state};                                      \
    if (disc) launch_plan_eval<PlanChargedBallF32<FRV, true>, true>(s, mean, std, returns, actions_out, B, K, H, c, k, st);      \
    else launch_plan_eval<PlanChargedBallF32<FRV, false>, false>(s, mean, std, returns, actions_out, B, K, H, c, k, st);         \
  } while (0)
    if (p->freq_rate == 1) EMEI_GO(1); else EMEI_GO(0);
#undef EMEI_GO
  } else {
    const ChargedBallConsts<R> k = make_cb_consts<R>(pk);
    const typename RefChargedBall<R>::Buffers s = {const_cast<uint8_t*>(on_circle), const_cast<R*>(circle), const_cast<R*>(free_state)};
    if (disc)
      launch_plan_eval<PlanRef<RefChargedBall<R>, true>, true>(s, mean, std, returns, actions_out, B, K, H, c, k, st);
    else
      launch_plan_eval<PlanRef<RefChargedBall<R>, false>, false>(s, mean, std, returns, actions_out, B, K, H, c, k, st);
  }
  return launch_status();
}

// ---------------------------------------------------------------------------------------------
// update: one CTA per start state
// ---------------------------------------------------------------------------------------------
// the candidates' total order as an unsigned key: larger return first, NaN below every number (key 0), -0 == +0
__device__ __forceinline__ unsigned long long plan_order_key(double r) {
  if (isnan(r)) return 0ull;
  const unsigned long long u = static_cast<unsigned long long>(__double_as_longlong(__dadd_rn(r, 0.0)));
  return (u >> 63) ? ~u : (u | 0x8000000000000000ull);
}
// does (ka, ia) rank before (kb, ib): larger key, then smaller index
__device__ __forceinline__ bool plan_before(unsigned long long ka, int ia, unsigned long long kb, int ib) {
  return ka > kb || (ka == kb && ia < ib);
}

// Sorts the Kp (a power of two) pairs (s_key, s_idx) of shared memory into plan_before order by a bitonic network.  Called by
// every thread of the CTA; ends on a barrier.
__device__ __forceinline__ void plan_sort(unsigned long long* s_key, uint16_t* s_idx, int Kp) {
  const int tid = threadIdx.x;
  for (int size = 2; size <= Kp; size <<= 1) {
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      for (int i = tid; i < (Kp >> 1); i += kBlock) {
        const int lo = 2 * i - (i & (stride - 1)), hi = lo + stride;
        const unsigned long long kl = s_key[lo], kh = s_key[hi];
        const int il = s_idx[lo], ih = s_idx[hi];
        const bool swap = (lo & size) == 0 ? plan_before(kh, ih, kl, il) : plan_before(kl, il, kh, ih);
        if (swap) {
          s_key[lo] = kh, s_key[hi] = kl;
          s_idx[lo] = static_cast<uint16_t>(ih), s_idx[hi] = static_cast<uint16_t>(il);
        }
      }
      __syncthreads();
    }
  }
}

// The refit of start state b, one warp per Philox block of steps (S = 4 discrete / 2 continuous steps per block).
template <typename R, bool DISC>
__device__ __forceinline__ void plan_refit(R* mean_io, R* std_io, int64_t B, int64_t b, int64_t H, int K, int L, double W, bool cem,
                                           const uint16_t* s_idx, const double* s_w, const PlanConsts& c) {
  constexpr int S = DISC ? 4 : 2;
  const int lane = threadIdx.x & 31;
  const int64_t nblk = (H + S - 1) / S;
  for (int64_t blk = threadIdx.x >> 5; blk < nblk; blk += kBlock / 32) {
    const int64_t t0 = blk * S;
    R m[S], sd[S];
    double s1[S], s2[S];
#pragma unroll
    for (int q = 0; q < S; ++q) {
      const bool in = t0 + q < H;
      m[q] = in ? mean_io[(t0 + q) * B + b] : R(0);
      sd[q] = (in && !DISC) ? std_io[(t0 + q) * B + b] : R(0);
      s1[q] = s2[q] = 0.0;
    }
    for (int j = lane; j < L; j += 32) {  // pass 1: sum w a
      const int kk = cem ? static_cast<int>(s_idx[j]) : j;
      PlanDraw d;
      d.refill<DISC>(c, plan_env_word(c, b, kk), t0);
      const double w = cem ? 1.0 : s_w[kk];
#pragma unroll
      for (int q = 0; q < S; ++q) s1[q] += w * static_cast<double>(d.action<DISC, R>(c, t0 + q, m[q], sd[q]));
    }
    double fit[S];
#pragma unroll
    for (int q = 0; q < S; ++q) fit[q] = warp_sum(s1[q]) / W;  // the xor tree leaves the total in every lane
    if (!DISC) {
      for (int j = lane; j < L; j += 32) {  // pass 2: sum w (a - fit_mean)^2, the actions regenerated
        const int kk = cem ? static_cast<int>(s_idx[j]) : j;
        PlanDraw d;
        d.refill<DISC>(c, plan_env_word(c, b, kk), t0);
        const double w = cem ? 1.0 : s_w[kk];
#pragma unroll
        for (int q = 0; q < S; ++q) {
          const double dv = static_cast<double>(d.action<DISC, R>(c, t0 + q, m[q], sd[q])) - fit[q];
          s2[q] += w * dv * dv;
        }
      }
#pragma unroll
      for (int q = 0; q < S; ++q) s2[q] = warp_sum(s2[q]);
    }
#pragma unroll
    for (int q = 0; q < S; ++q) {
      const int64_t t = t0 + q;
      if (lane != q || t >= H) continue;
      const double alpha = c.momentum, beta = 1.0 - c.momentum;
      if (DISC) {
        double p = alpha * static_cast<double>(m[q]) + beta * fit[q];
        p = p < 0.0 ? 0.0 : (p > 1.0 ? 1.0 : p);
        mean_io[t * B + b] = static_cast<R>(p);
      } else {
        const double ns = alpha * static_cast<double>(sd[q]) + beta * sqrt(s2[q] / W);
        mean_io[t * B + b] = static_cast<R>(alpha * static_cast<double>(m[q]) + beta * fit[q]);
        std_io[t * B + b] = static_cast<R>(ns > c.min_std ? ns : c.min_std);
      }
    }
  }
}

template <typename R>
__global__ void __launch_bounds__(kBlock)
    plan_update_kernel(const double* __restrict__ returns, R* __restrict__ mean_io, R* __restrict__ std_io, void* __restrict__ best_actions,
                       double* __restrict__ best_return, int64_t B, int K, int Kp, int64_t H, const PlanConsts c) {
  __shared__ union {
    unsigned long long key[kPlanMaxCandidates];  // CEM: the order keys
    double w[kPlanMaxCandidates];                // MPPI: the weights
  } s_kw;
  __shared__ uint16_t s_idx[kPlanMaxCandidates];
  unsigned long long* s_key = s_kw.key;
  double* s_w = s_kw.w;
  __shared__ unsigned long long s_bk[kBlock / 32];
  __shared__ int s_bi[kBlock / 32];
  __shared__ double s_red[kBlock / 32];
  __shared__ int s_best;
  __shared__ double s_wsum;
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const bool disc = c.kind <= EMEI_ACTION_DISCRETE_I64;
  const bool cem = c.method == EMEI_PLAN_CEM;
  for (int64_t b = blockIdx.x; b < B; b += gridDim.x) {
    const double* r = returns + b * K;
    // ---- order keys and the argmax candidate
    unsigned long long bk = 0ull;
    int bi = 0x7fffffff;
    for (int j = tid; j < Kp; j += kBlock) {
      const unsigned long long key = j < K ? plan_order_key(r[j]) : 0ull;
      s_key[j] = key;
      s_idx[j] = static_cast<uint16_t>(j < K ? j : 0xffff);
      if (j < K && plan_before(key, j, bk, bi)) bk = key, bi = j;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const unsigned long long ok = __shfl_xor_sync(0xffffffffu, bk, o);
      const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
      if (plan_before(ok, oi, bk, bi)) bk = ok, bi = oi;
    }
    if (lane == 0) s_bk[warp] = bk, s_bi[warp] = bi;
    __syncthreads();
    if (tid == 0) {
      for (int w = 1; w < kBlock / 32; ++w)
        if (plan_before(s_bk[w], s_bi[w], bk, bi)) bk = s_bk[w], bi = s_bi[w];
      s_best = bi;
    }
    __syncthreads();
    const int best = s_best;
    // ---- selection: CEM sorts (key desc, index asc) by a bitonic network; MPPI forms exp((R - max R) / lambda)
    if (cem) {
      plan_sort(s_key, s_idx, Kp);
    } else {
      const double rmax = r[best];
      double part = 0.0;
      for (int j = tid; j < K; j += kBlock) {  // a weight that is not a number counts 0
        double w = exp((r[j] - rmax) / c.temperature);
        w = isnan(w) ? 0.0 : w;
        s_w[j] = w;
        part += w;
      }
      // every thread holds the same total (block_sum_double reduces in one fixed order in every warp), so the branch is uniform
      // and s_wsum is written once, before the barrier that publishes it
      const double tot = block_sum_double(part, s_red);
      const bool uniform = !(tot > 0.0);  // every weight 0 (no finite maximum): uniform weights
      if (uniform)
        for (int j = tid; j < K; j += kBlock) s_w[j] = 1.0;
      if (tid == 0) s_wsum = uniform ? static_cast<double>(K) : tot;
      __syncthreads();
    }
    // ---- the argmax candidate's actions, from the distribution before this update
    if (best_actions != nullptr || best_return != nullptr) {
      if (best_return != nullptr && tid == 0) best_return[b] = r[best];
      if (best_actions != nullptr) {
        const unsigned long long env = plan_env_word(c, b, best);
        for (int64_t t = tid; t < H; t += kBlock) {
          const R m = mean_io[t * B + b], s = disc ? R(0) : std_io[t * B + b];
          PlanDraw d;
          R a;
          if (disc) {
            d.refill<true>(c, env, t);
            a = d.action<true, R>(c, t, m, s);
          } else {
            d.refill<false>(c, env, t);
            a = d.action<false, R>(c, t, m, s);
          }
          plan_store<R>(best_actions, t * B + b, c.kind, a);
        }
      }
      __syncthreads();
    }
    // ---- refit: warp w takes the Philox blocks of steps w, w + 8, ...; lanes take the chosen candidates j = lane, lane + 32, ...
    // (CEM: the elites in rank order; MPPI: k order), then a fixed shuffle tree.  Two passes (the mean, then the squared
    // deviations from it): a one-pass variance cancels when the weights concentrate on a few candidates.
    const int L = cem ? c.elites : K;
    const double W = cem ? static_cast<double>(c.elites) : s_wsum;
    if (disc)
      plan_refit<R, true>(mean_io, std_io, B, b, H, K, L, W, cem, s_idx, s_w, c);
    else
      plan_refit<R, false>(mean_io, std_io, B, b, H, K, L, W, cem, s_idx, s_w, c);
    __syncthreads();  // shared memory is reused by the next start state
  }
}

template <typename R>
int plan_update(const double* returns, R* mean_io, R* std_io, void* best_actions, double* best_return, int64_t B, int64_t K, int64_t H,
                const emei_plan_params* q, emei_stream_t stream) {
  if (const int e = check_plan_sizes(B, K, H)) return e;
  EMEI_CHECK_PTR(q);
  if (const int e = check_plan_params(*q, K)) return e;
  if (B == 0 || H == 0) return EMEI_OK;
  EMEI_CHECK_PTR(returns);
  EMEI_CHECK_PTR(mean_io);
  if (q->action_kind >= EMEI_ACTION_CONTINUOUS_F32) EMEI_CHECK_PTR(std_io);
  int Kp = 1;
  while (Kp < K) Kp <<= 1;
  const int64_t cap = static_cast<int64_t>(sm_count()) * 16;
  const int grid = static_cast<int>(B < cap ? B : cap);
  plan_update_kernel<R><<<grid, kBlock, 0, static_cast<cudaStream_t>(stream)>>>(
      returns, mean_io, std_io, best_actions, best_return, B, static_cast<int>(K), Kp, H, make_plan_consts(*q));
  return launch_status();
}

}  // namespace emei
