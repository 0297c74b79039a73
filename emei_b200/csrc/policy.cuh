// Policy search over the true dynamics (DESIGN.md 4.11): closed-loop returns of linear feedback policies, and the ARS
// (Mania, Guy & Recht 2018, V1-t) perturbation and update around one policy.
//
// A policy theta = (w_0 .. w_{D-1}, c) acts on the observation step() returns in the current state:
//   u = c; u = u + w_j double(obs_j), j ascending, every product and sum rounded on its own;
//   continuous: a = clamp(R(u)) as plan_clamp; discrete: a = u > 0 ? 1 : 0.
// Per step the eval calls the plan eval's family adapters (plan.cuh), i.e. the device function of the env's own rollout(),
// so the rewards of (c, e) equal a teacher-forced rollout of its actions bit for bit.
//
// Direction k draws delta_k from Philox keyed by (seed, k) with purpose kPurposePolicyPerturb (host mirror: tests/test_policy.py
// policy_directions): block j gives delta_{2j} = rad cs and delta_{2j+1} = rad sn.  The update regenerates the directions
// it steps along instead of reading params back.
#pragma once
#include <cmath>

#include "plan.cuh"

namespace emei {

constexpr int kPolicyMaxDirections = EMEI_POLICY_MAX_DIRECTIONS;
constexpr int kPolicyMaxParams = EMEI_POLICY_MAX_PARAMS;

// sizes first (every eval entry point): 0 <= C, E <= 2^31 (C E < 2^62 fits the 64-bit index), 0 <= H < 2^31
inline int check_policy_sizes(int64_t C, int64_t E, int64_t H) {
  if (C < 0 || E < 0 || C > (int64_t(1) << 31) || E > (int64_t(1) << 31) || H < 0 || H > 0x7fffffff) return EMEI_ERR_BAD_SIZE;
  return EMEI_OK;
}

inline int check_policy_eval_params(const emei_policy_params& q) {
  if (!action_kind_valid(q.action_kind)) return EMEI_ERR_BAD_ACTION_KIND;
  if (!(q.gamma >= 0.0 && q.gamma <= 1.0)) return EMEI_ERR_BAD_PARAM;
  if (q.action_kind >= EMEI_ACTION_CONTINUOUS_F32 && !(q.action_low <= q.action_high)) return EMEI_ERR_BAD_PARAM;
  return EMEI_OK;
}

// the eval's constants in the planner's form (gamma, the action box and kind: what plan_clamp / plan_store read)
inline PlanConsts make_policy_consts(const emei_policy_params& q) {
  PlanConsts c = {};
  c.gamma = q.gamma;
  c.low = q.action_low;
  c.high = q.action_high;
  c.kind = q.action_kind;
  return c;
}

// direction k's coordinates 2j and 2j + 1
__device__ __forceinline__ void policy_delta_pair(unsigned long long seed, int k, int j, double& d0, double& d1) {
  double rad, cs, sn;
  philox_normal_pair(seed, static_cast<unsigned long long>(k), static_cast<uint32_t>(j), kPurposePolicyPerturb, rad, cs, sn);
  d0 = __dmul_rn(rad, cs);
  d1 = __dmul_rn(rad, sn);
}

// ---------------------------------------------------------------------------------------------
// eval: one (candidate c, episode e) pair per thread, e fastest (a warp shares theta_c: its loads are broadcasts; the start
// loads, the returns and the actions are coalesced)
// ---------------------------------------------------------------------------------------------
template <class F, bool DISC>
__device__ __forceinline__ typename F::Real policy_action(const double (&th)[F::kObs + 1], const typename F::Real (&o)[F::kObs],
                                                          const PlanConsts& c) {
  using R = typename F::Real;
  double u = th[F::kObs];
#pragma unroll
  for (int j = 0; j < F::kObs; ++j) u = __dadd_rn(u, __dmul_rn(th[j], static_cast<double>(o[j])));
  if constexpr (DISC)
    return u > 0.0 ? R(1) : R(0);
  else
    return plan_clamp<R>(static_cast<R>(u), c);
}

template <class F, bool DISC>
__global__ void __launch_bounds__(kBlock)
    policy_eval_kernel(const typename F::State s, const double* __restrict__ params, double* __restrict__ returns,
                       void* __restrict__ actions_out, int64_t C, int64_t E, int64_t H, const PlanConsts c, const typename F::Consts k) {
  using R = typename F::Real;
  constexpr int D = F::kObs;
  const int64_t n = C * E;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * kBlock;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x; i < n; i += stride) {
    const int64_t cand = i / E;
    double th[D + 1];
#pragma unroll
    for (int j = 0; j <= D; ++j) th[j] = params[cand * (D + 1) + j];
    typename F::Regs e;
    F::load(e, s, i - cand * E);
    R o[D];
    F::observe(e, k, o);
    double ret = 0.0, disc = 1.0;
    bool live = true;
    for (int64_t t = 0; t < H; ++t) {
      const R a = policy_action<F, DISC>(th, o, c);
      if (actions_out != nullptr) plan_store<R>(actions_out, t * n + i, c.kind, a);
      bool terminated;
      const R rew = F::step(e, a, k, terminated, o);  // after termination only to keep actions_out a teacher-forcing record
      if (live) {
        ret = __dadd_rn(ret, __dmul_rn(disc, static_cast<double>(rew)));
        disc = __dmul_rn(disc, c.gamma);
        if (terminated) {
          live = false;
          if (actions_out == nullptr) break;
        }
      }
    }
    returns[i] = ret;
  }
}

template <class F, bool DISC, typename K>
inline void launch_policy_eval(const typename F::State& s, const double* params, double* returns, void* actions_out, int64_t C, int64_t E,
                               int64_t H, const PlanConsts& c, const K& k, cudaStream_t st) {
  policy_eval_kernel<F, DISC><<<resident_grid(policy_eval_kernel<F, DISC>, C * E), kBlock, 0, st>>>(s, params, returns, actions_out, C, E,
                                                                                                     H, c, k);
}

// the checks every eval entry point applies first, in order, with its family's params check
template <typename P>
inline int policy_eval_head(int64_t C, int64_t E, int64_t H, const emei_policy_params* q, const P* p, int (*check_family)(const P&)) {
  if (const int e = check_policy_sizes(C, E, H)) return e;
  EMEI_CHECK_PTR(q);
  EMEI_CHECK_PTR(p);
  if (const int e = check_family(*p)) return e;
  return check_policy_eval_params(*q);
}

template <typename R>
int cartpole_policy_eval(const R* state0, const double* params, double* returns, void* actions_out, int64_t C, int64_t E, int64_t H,
                         const emei_policy_params* q, const emei_cartpole_params* p, emei_stream_t stream) {
  if (const int e = policy_eval_head(C, E, H, q, p, check_cartpole_params)) return e;
  if (C == 0 || E == 0 || H == 0) return EMEI_OK;
  EMEI_CHECK_PTR(state0);
  EMEI_CHECK_PTR(params);
  EMEI_CHECK_PTR(returns);
  EMEI_CHECK_ALIGN16(state0);
  emei_cartpole_params pk = *p;
  pk.action_kind = q->action_kind;  // the policy's actions drive the step
  const PlanConsts c = make_policy_consts(*q);
  const bool disc = q->action_kind <= EMEI_ACTION_DISCRETE_I64, ip = p->variant >= EMEI_IP_REBOUND_BALANCING;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if constexpr (sizeof(R) == 4) {  // the float32 rollout's instantiations (emei_cartpole_rollout_f32)
#define EMEI_GO(IPV, FRV)                                                                                                          \
  do {                                                                                                                             \
    const PlanRowsF32 s = {state0};                                                                                                \
    const CartPoleF32Consts k = make_cartpole_f32_consts(pk);                                                                      \
    if (disc) launch_policy_eval<PlanCartPoleF32<IPV, FRV, true>, true>(s, params, returns, actions_out, C, E, H, c, k, st);       \
    else launch_policy_eval<PlanCartPoleF32<IPV, FRV, false>, false>(s, params, returns, actions_out, C, E, H, c, k, st);          \
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
#define EMEI_GO(IPV)                                                                                                               \
  do {                                                                                                                             \
    const typename RefCartPole<R, IPV>::Buffers s = {const_cast<R*>(state0)};                                                      \
    if (disc) launch_policy_eval<PlanRef<RefCartPole<R, IPV>, true>, true>(s, params, returns, actions_out, C, E, H, c, k, st);    \
    else launch_policy_eval<PlanRef<RefCartPole<R, IPV>, false>, false>(s, params, returns, actions_out, C, E, H, c, k, st);       \
  } while (0)
    if (ip) EMEI_GO(true); else EMEI_GO(false);
#undef EMEI_GO
  }
  return launch_status();
}

template <typename R>
int i2p_policy_eval(const R* state0, const double* params, double* returns, void* actions_out, int64_t C, int64_t E, int64_t H,
                    const emei_policy_params* q, const emei_i2p_params* p, emei_stream_t stream) {
  if (const int e = policy_eval_head(C, E, H, q, p, check_i2p_params)) return e;
  if (q->action_kind <= EMEI_ACTION_DISCRETE_I64) return EMEI_ERR_BAD_ACTION_KIND;  // the double pendulum's tasks act on a Box
  if (C == 0 || E == 0 || H == 0) return EMEI_OK;
  EMEI_CHECK_PTR(state0);
  EMEI_CHECK_PTR(params);
  EMEI_CHECK_PTR(returns);
  EMEI_CHECK_ALIGN16(state0);
  emei_i2p_params pk = *p;
  pk.action_kind = q->action_kind;
  const typename RefI2P<R>::Buffers s = {const_cast<R*>(state0)};
  launch_policy_eval<PlanRef<RefI2P<R>, false>, false>(s, params, returns, actions_out, C, E, H, make_policy_consts(*q),
                                                       make_i2p_consts<R>(pk), static_cast<cudaStream_t>(stream));
  return launch_status();
}

template <typename R>
int charged_ball_policy_eval(const uint8_t* on_circle, const R* circle, const R* free_state, const double* params, double* returns,
                             void* actions_out, int64_t C, int64_t E, int64_t H, const emei_policy_params* q,
                             const emei_charged_ball_params* p, emei_stream_t stream) {
  if (const int e = policy_eval_head(C, E, H, q, p, check_charged_ball_params)) return e;
  if (C == 0 || E == 0 || H == 0) return EMEI_OK;
  EMEI_CHECK_PTR(on_circle);
  EMEI_CHECK_PTR(circle);
  EMEI_CHECK_PTR(free_state);
  EMEI_CHECK_PTR(params);
  EMEI_CHECK_PTR(returns);
  EMEI_CHECK_ALIGN16(circle);
  EMEI_CHECK_ALIGN16(free_state);
  emei_charged_ball_params pk = *p;
  pk.action_kind = q->action_kind;
  const PlanConsts c = make_policy_consts(*q);
  const bool disc = q->action_kind <= EMEI_ACTION_DISCRETE_I64;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if constexpr (sizeof(R) == 4) {  // emei_charged_ball_rollout_f32's instantiations
    const ChargedBallF32Consts k = make_cb_f32_consts(pk);
    const PlanChargedBallF32State s = {on_circle, circle, free_state};
#define EMEI_GO(FRV)                                                                                                               \
  do {                                                                                                                             \
    if (disc) launch_policy_eval<PlanChargedBallF32<FRV, true>, true>(s, params, returns, actions_out, C, E, H, c, k, st);         \
    else launch_policy_eval<PlanChargedBallF32<FRV, false>, false>(s, params, returns, actions_out, C, E, H, c, k, st);            \
  } while (0)
    if (p->freq_rate == 1) EMEI_GO(1); else EMEI_GO(0);
#undef EMEI_GO
  } else {
    const ChargedBallConsts<R> k = make_cb_consts<R>(pk);
    const typename RefChargedBall<R>::Buffers s = {const_cast<uint8_t*>(on_circle), const_cast<R*>(circle), const_cast<R*>(free_state)};
    if (disc)
      launch_policy_eval<PlanRef<RefChargedBall<R>, true>, true>(s, params, returns, actions_out, C, E, H, c, k, st);
    else
      launch_policy_eval<PlanRef<RefChargedBall<R>, false>, false>(s, params, returns, actions_out, C, E, H, c, k, st);
  }
  return launch_status();
}

// The perturbation and the update act on float64 parameters in both precisions: they are compiled once, in the translation
// unit that defines EMEI_POLICY_ARS (emei_f64.cu).
#ifdef EMEI_POLICY_ARS
// ---------------------------------------------------------------------------------------------
// perturb: one thread per (direction, Philox block)
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kBlock)
    policy_perturb_kernel(const double* __restrict__ theta, double* __restrict__ params, int N, int P, unsigned long long seed, double nu) {
  const int nblk = (P + 1) >> 1;
  const int i = blockIdx.x * kBlock + threadIdx.x;
  if (i >= N * nblk) return;
  const int k = i / nblk, j = i - k * nblk;
  double d[2];
  policy_delta_pair(seed, k, j, d[0], d[1]);
#pragma unroll
  for (int h = 0; h < 2; ++h) {
    const int p = 2 * j + h;
    if (p >= P) break;
    const double th = theta[p], step = __dmul_rn(nu, d[h]);
    params[static_cast<int64_t>(2 * k) * P + p] = __dadd_rn(th, step);
    params[static_cast<int64_t>(2 * k + 1) * P + p] = __dsub_rn(th, step);
  }
}

inline int check_policy_dims(int64_t N, int64_t P) {
  if (N < 1 || N > kPolicyMaxDirections || P < 1 || P > kPolicyMaxParams) return EMEI_ERR_BAD_SIZE;
  return EMEI_OK;
}

inline int policy_perturb(const double* theta, double* params, int64_t N, int64_t P, const emei_policy_params* q, emei_stream_t stream) {
  if (const int e = check_policy_dims(N, P)) return e;
  EMEI_CHECK_PTR(q);
  if (!(q->noise >= 0.0 && std::isfinite(q->noise))) return EMEI_ERR_BAD_PARAM;
  EMEI_CHECK_PTR(theta);
  EMEI_CHECK_PTR(params);
  const int threads = static_cast<int>(N * ((P + 1) / 2));
  policy_perturb_kernel<<<grid_for(threads, kBlock), kBlock, 0, static_cast<cudaStream_t>(stream)>>>(
      theta, params, static_cast<int>(N), static_cast<int>(P), q->seed, q->noise);
  return launch_status();
}

// ---------------------------------------------------------------------------------------------
// update: one CTA
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double policy_row_mean(const double* r, int64_t row, int64_t E) {
  const double* x = r + row * E;
  double s = 0.0;
  for (int64_t e = 0; e < E; ++e) s = __dadd_rn(s, x[e]);
  return __ddiv_rn(s, static_cast<double>(E));
}

__global__ void __launch_bounds__(kBlock)
    policy_update_kernel(const double* __restrict__ returns, double* __restrict__ theta, double* __restrict__ stats, int N, int64_t E,
                         int P, int Np, unsigned long long seed, double alpha, int top) {
  __shared__ union {
    unsigned long long key[kPolicyMaxDirections];  // the order keys, then
    double diff[kPolicyMaxDirections];             // r_k+ - r_k- of the chosen directions in rank order
  } s_kd;
  __shared__ uint16_t s_idx[kPolicyMaxDirections];
  __shared__ double s_red[kBlock / 32];
  __shared__ double s_best;
  const int tid = threadIdx.x;
  // ---- pass 1: the directions' mean returns -> order keys (not eligible: key 0, after every eligible direction)
  double fin_sum = 0.0, fin_cnt = 0.0, elig = 0.0;
  for (int k = tid; k < Np; k += kBlock) {
    unsigned long long key = 0ull;
    if (k < N) {
      const double rp = policy_row_mean(returns, 2 * k, E), rm = policy_row_mean(returns, 2 * k + 1, E);
      if (isfinite(rp)) fin_sum = __dadd_rn(fin_sum, rp), fin_cnt += 1.0;
      if (isfinite(rm)) fin_sum = __dadd_rn(fin_sum, rm), fin_cnt += 1.0;
      if (isfinite(rp) && isfinite(rm)) {
        key = plan_order_key(rp > rm ? rp : rm);  // finite: key > plan_order_key(-inf) > 0
        elig += 1.0;
      }
    }
    s_kd.key[k] = key;
    s_idx[k] = static_cast<uint16_t>(k < N ? k : 0xffff);
  }
  fin_sum = block_sum_double(fin_sum, s_red);
  fin_cnt = block_sum_double(fin_cnt, s_red);  // counts: exact in double
  elig = block_sum_double(elig, s_red);
  plan_sort(s_kd.key, s_idx, Np);  // (max return desc, k asc); begins after block_sum_double's barriers, ends on one
  const int bp = static_cast<int>(elig < static_cast<double>(top) ? elig : static_cast<double>(top));
  // ---- pass 2: the chosen directions' returns again -> their mean, r_k+ - r_k- in rank order
  double part = 0.0;
  for (int j = tid; j < bp; j += kBlock) {
    const int k = s_idx[j];
    const double rp = policy_row_mean(returns, 2 * k, E), rm = policy_row_mean(returns, 2 * k + 1, E);
    part = __dadd_rn(part, __dadd_rn(rp, rm));
    s_kd.diff[j] = __dsub_rn(rp, rm);  // s_kd.key[j] was last read before plan_sort's final barrier
    if (j == 0) s_best = rp > rm ? rp : rm;
  }
  const double n2 = 2.0 * static_cast<double>(bp);
  const double mu = __ddiv_rn(block_sum_double(part, s_red), n2);
  // ---- pass 3: the population std of the 2b' returns (two passes: one-pass variance cancels on near-equal returns)
  double dev = 0.0;
  for (int j = tid; j < bp; j += kBlock) {
    const int k = s_idx[j];
    const double dp = __dsub_rn(policy_row_mean(returns, 2 * k, E), mu), dm = __dsub_rn(policy_row_mean(returns, 2 * k + 1, E), mu);
    dev = __dadd_rn(dev, __dadd_rn(__dmul_rn(dp, dp), __dmul_rn(dm, dm)));
  }
  const double sigma = sqrt(__ddiv_rn(block_sum_double(dev, s_red), n2));  // every thread holds the same bits
  // ---- pass 4: sum_j (r+ - r-) delta_{k_j}, the directions regenerated; one fixed-order block sum per coordinate
  double acc[kPolicyMaxParams];
#pragma unroll
  for (int p = 0; p < kPolicyMaxParams; ++p) acc[p] = 0.0;
  const bool step = bp > 0 && sigma > 0.0 && isfinite(sigma);  // uniform: bp and sigma are the same in every thread
  if (step) {
    for (int j = tid; j < bp; j += kBlock) {
      const int k = s_idx[j];
      const double w = s_kd.diff[j];
#pragma unroll
      for (int jb = 0; jb < kPolicyMaxParams / 2; ++jb) {
        if (2 * jb >= P) break;
        double d0, d1;
        policy_delta_pair(seed, k, jb, d0, d1);
        acc[2 * jb] = __dadd_rn(acc[2 * jb], __dmul_rn(w, d0));
        acc[2 * jb + 1] = __dadd_rn(acc[2 * jb + 1], __dmul_rn(w, d1));
      }
    }
    const double scale = __ddiv_rn(alpha, __dmul_rn(static_cast<double>(bp), sigma));
#pragma unroll
    for (int p = 0; p < kPolicyMaxParams; ++p) {
      if (p >= P) break;
      const double tot = block_sum_double(acc[p], s_red);
      if (tid == 0) theta[p] = __dadd_rn(theta[p], __dmul_rn(scale, tot));
    }
  }
  if (stats != nullptr && tid == 0) {
    const double nan = __longlong_as_double(0x7ff8000000000000ll);
    stats[0] = static_cast<double>(bp);
    stats[1] = bp > 0 ? sigma : nan;
    stats[2] = bp > 0 ? s_best : nan;
    stats[3] = fin_cnt > 0.0 ? __ddiv_rn(fin_sum, fin_cnt) : nan;
  }
}

inline int policy_update(const double* returns, double* theta_io, double* stats, int64_t N, int64_t E, int64_t P, const emei_policy_params* q,
                         emei_stream_t stream) {
  if (const int e = check_policy_dims(N, P)) return e;
  if (E < 1 || E > (int64_t(1) << 31)) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(q);
  if (q->top < 1 || q->top > N || !std::isfinite(q->step_size)) return EMEI_ERR_BAD_PARAM;
  EMEI_CHECK_PTR(returns);
  EMEI_CHECK_PTR(theta_io);
  int Np = 1;
  while (Np < N) Np <<= 1;
  policy_update_kernel<<<1, kBlock, 0, static_cast<cudaStream_t>(stream)>>>(returns, theta_io, stats, static_cast<int>(N), E,
                                                                           static_cast<int>(P), Np, q->seed, q->step_size, q->top);
  return launch_status();
}

#endif  // EMEI_POLICY_ARS

}  // namespace emei
