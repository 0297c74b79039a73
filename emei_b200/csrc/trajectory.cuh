// Differentiable open-loop trajectories: T steps of emei_cartpole_step_* (cart-pole + EMEI_IP_* variants) / emei_i2p_step_*
// from caller rows in ONE launch, and their vector-Jacobian product in ONE reverse-sweep launch; both precisions.
//
// Forward = the open-loop composition of T stateless steps (no noise, no resets, no statistics): step t's state, observation,
// reward and done are bit-equal to the t-th of T chained step calls, because every step calls the step's own device function
//   * float32 cart-pole / IP: cartpole_step_one<IP, FR> with action_to_f_mt -- the lean arithmetic of the TMA and small-batch
//     step kernels (FR 1 / 4 / 0 as their dispatch instantiates it);
//   * float64 cart-pole / IP: cartpole_env_step<double, IP> with the noise off -- the generic step kernel's;
//   * I2P: i2p_env_step<R> with the noise off.
// One env per thread, persistent grid-stride loop; the state stays in registers for all T steps and every array is time-major
// ([T(+1), n, ...]: a warp stores 32 consecutive rows).  Step t+1's action is requested before step t's math.
//
// Reverse sweep = the VJP of that composition under the model of derivs.cuh (float64 cart-pole: the float64 Euler step; the
// clamp passes inclusively; the I2P observation's angles have slope pi).  One env per thread walks t = T-1 .. 0: it reloads
// states[t] and actions[t], rebuilds the step's tangent T_t = d y_{t+1} / d (y_t, a_t) with the derivative kernels' own
// functions, forms
//   w = carry + g_states[t+1] + slope * g_obs[t] + g_rewards[t] * d reward_t / d y_{t+1}
// (the term order of cartpole_deriv_kernel / i2p_deriv_kernel, where carry is autograd's g_state_out), writes
// g_actions[t] = w^T T_t[:, D] and carries w^T T_t[:, :D]; g_state0 = carry + g_states[0].  The cotangent is never written to
// memory between steps, and step t-1's row and action are requested before step t's tangent math.
#pragma once
#include <type_traits>

#include "derivs.cuh"

namespace emei {

// The chained step's arithmetic for one cart-pole / IP env on registers, per precision.
template <typename R, bool IP, int FR>
struct CartPoleTrajStep;

template <bool IP, int FR>
struct CartPoleTrajStep<float, IP, FR> {  // the lean float32 step of cartpole_step_f32_tma_dispatch
  using Consts = CartPoleF32Consts;
  using Row = float4;
  static Consts make(const emei_cartpole_params& p) { return make_cartpole_f32_consts(p); }
  __device__ __forceinline__ static Row load(const float* p, int64_t r) { return reinterpret_cast<const float4*>(p)[r]; }
  __device__ __forceinline__ static void store(float* p, int64_t r, const Row& y) { reinterpret_cast<float4*>(p)[r] = y; }
  // force / m_total of element e of the action array, as the step kernels decode it
  template <int AK>
  __device__ __forceinline__ static float drive(const void* a, int64_t e, const Consts& k) {
    return action_to_f_mt<IP, AK>(load_action_f32<AK>(a, e), k);
  }
  __device__ __forceinline__ static void step(Row& y, float f_mt, const Consts& k, float& rew, bool& notdone, Row& obs) {
    cartpole_step_one<IP, FR>(y, f_mt, ip_flip(IP, k.variant), k, rew, notdone, obs);
  }
};

template <bool IP, int FR>
struct CartPoleTrajStep<double, IP, FR> {  // the reference-arithmetic step of cartpole_step_kernel
  using Consts = CartPoleConsts<double>;
  using Row = Vec4<double>;
  static Consts make(const emei_cartpole_params& p) { return make_cartpole_consts<double>(p); }
  __device__ __forceinline__ static Row load(const double* p, int64_t r) { return Row::load(p + 4 * r); }
  __device__ __forceinline__ static void store(double* p, int64_t r, const Row& y) { y.store(p + 4 * r); }
  template <int AK>
  __device__ __forceinline__ static double drive(const void* a, int64_t e, const Consts& k) {
    return IP ? load_ctrl<double>(a, e, AK) : load_force<double>(a, e, AK, k.force_mag);
  }
  __device__ __forceinline__ static void step(Row& y, double drv, const Consts& k, double& rew, bool& notdone, Row& obs) {
    const NoiseConsts z = {};
    cartpole_env_step<double, IP>(y, drv, k, z, 0ull, 0ull, rew, notdone, obs);
  }
};

// The action kind as a compile-time constant (the step kernels' dispatch): each step's action is one typed load, and the
// forward kernels keep no per-step kind switch (with a run-time kind the float32 I2P forward kept the decoded action in a
// stack slot across the step).
template <typename F>
inline void with_action_kind(int ak, F&& f) {
  switch (ak) {
    case EMEI_ACTION_DISCRETE_U8: f(std::integral_constant<int, EMEI_ACTION_DISCRETE_U8>{}); break;
    case EMEI_ACTION_DISCRETE_I32: f(std::integral_constant<int, EMEI_ACTION_DISCRETE_I32>{}); break;
    case EMEI_ACTION_DISCRETE_I64: f(std::integral_constant<int, EMEI_ACTION_DISCRETE_I64>{}); break;
    case EMEI_ACTION_CONTINUOUS_F32: f(std::integral_constant<int, EMEI_ACTION_CONTINUOUS_F32>{}); break;
    default: f(std::integral_constant<int, EMEI_ACTION_CONTINUOUS_F64>{}); break;
  }
}

// states[0] = state0; then per step t: states[t+1], obs[t] (nullable), rewards[t], dones[t] (nullable)
template <typename R, bool IP, int FR, int AK>
__global__ void __launch_bounds__(kBlock)
    cartpole_trajectory_kernel(const R* __restrict__ state0, const void* __restrict__ actions, R* __restrict__ states,
                               R* __restrict__ obs, R* __restrict__ rewards, uint8_t* __restrict__ dones, int64_t n, int64_t horizon,
                               const typename CartPoleTrajStep<R, IP, FR>::Consts k) {
  using S = CartPoleTrajStep<R, IP, FR>;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * kBlock;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x; i < n; i += stride) {
    typename S::Row y = S::load(state0, i);
    S::store(states, i, y);
    R drv = S::template drive<AK>(actions, i, k);
    for (int64_t t = 0, e = i; t < horizon; ++t, e += n) {  // e = t * n + i: element (t, i) of a [horizon, n] array
      const R drv_next = t + 1 < horizon ? S::template drive<AK>(actions, e + n, k) : R(0);
      typename S::Row o;
      R rew;
      bool notdone;
      S::step(y, drv, k, rew, notdone, o);
      S::store(states, e + n, y);
      if (obs != nullptr) S::store(obs, e, o);
      rewards[e] = rew;
      if (dones != nullptr) dones[e] = notdone ? 0 : 1;
      drv = drv_next;
    }
  }
}

template <typename R, bool IP>
__global__ void __launch_bounds__(kBlock)
    cartpole_trajectory_vjp_kernel(const R* __restrict__ states, const void* __restrict__ actions, const R* __restrict__ g_states,
                                   const R* __restrict__ g_obs, const R* __restrict__ g_rewards, R* __restrict__ g_state0,
                                   R* __restrict__ g_actions, int64_t n, int64_t horizon, const CartPoleConsts<R> k) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * kBlock;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x; i < n; i += stride) {
    R carry[4] = {R(0), R(0), R(0), R(0)};
    int64_t e = (horizon - 1) * n + i;
    Vec4<R> row = Vec4<R>::load(states + 4 * e);
    R force, dforce;
    cartpole_force_and_slope<R, IP>(actions, e, k, force, dforce);
    for (int64_t t = horizon - 1; t >= 0; --t, e -= n) {
      Vec4<R> row_prev = row;  // step t-1's inputs, requested before step t's tangent math
      R force_prev = R(0), dforce_prev = R(0);
      if (t > 0) {
        row_prev = Vec4<R>::load(states + 4 * (e - n));
        cartpole_force_and_slope<R, IP>(actions, e - n, k, force_prev, dforce_prev);
      }
      R y[4] = {row.x, row.y, row.z, row.w}, T[4][5], wr[4];
      cartpole_tangent<R, IP>(y, T, force, dforce, k);
      cartpole_reward_slope<R, IP>(y, k, wr);
      Vec4<R> gs = {R(0), R(0), R(0), R(0)}, go = gs;
      if (g_states != nullptr) gs = Vec4<R>::load(g_states + 4 * (e + n));
      if (g_obs != nullptr) go = Vec4<R>::load(g_obs + 4 * e);
      const R gr = g_rewards != nullptr ? g_rewards[e] : R(0);
      const R w[4] = {carry[0] + gs.x + go.x + gr * wr[0], carry[1] + gs.y + go.y + gr * wr[1], carry[2] + gs.z + go.z + gr * wr[2],
                      carry[3] + gs.w + go.w + gr * wr[3]};
      R g[5];
#pragma unroll
      for (int c = 0; c < 5; ++c) g[c] = w[0] * T[0][c] + w[1] * T[1][c] + w[2] * T[2][c] + w[3] * T[3][c];
      if (g_actions != nullptr) g_actions[e] = g[4];
#pragma unroll
      for (int c = 0; c < 4; ++c) carry[c] = g[c];
      row = row_prev, force = force_prev, dforce = dforce_prev;
    }
    Vec4<R> g0 = {carry[0], carry[1], carry[2], carry[3]};
    if (g_states != nullptr) {
      const Vec4<R> gs = Vec4<R>::load(g_states + 4 * i);
      g0 = {g0.x + gs.x, g0.y + gs.y, g0.z + gs.z, g0.w + gs.w};
    }
    g0.store(g_state0 + 4 * i);
  }
}

template <bool IP, int FR, typename R>
inline void launch_cartpole_trajectory(const R* state0, const void* actions, R* states, R* obs, R* rewards, uint8_t* dones, int64_t n,
                                       int64_t horizon, const emei_cartpole_params& p, cudaStream_t s) {
  const auto k = CartPoleTrajStep<R, IP, FR>::make(p);
  with_action_kind(p.action_kind, [&](auto ak) {
    constexpr int AK = decltype(ak)::value;
    cartpole_trajectory_kernel<R, IP, FR, AK><<<resident_grid(cartpole_trajectory_kernel<R, IP, FR, AK>, n), kBlock, 0, s>>>(
        state0, actions, states, obs, rewards, dones, n, horizon, k);
  });
}

template <typename R>
int cartpole_trajectory(const R* state0, const void* actions, R* states, R* obs, R* rewards, uint8_t* dones, int64_t n, int64_t horizon,
                        const emei_cartpole_params* p, emei_stream_t stream) {
  if (n < 0 || horizon < 0) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(p);
  if (const int e = check_cartpole_params(*p)) return e;
  if (n == 0 || horizon == 0) return EMEI_OK;
  EMEI_CHECK_PTR(state0);
  EMEI_CHECK_PTR(actions);
  EMEI_CHECK_PTR(states);
  EMEI_CHECK_PTR(rewards);
  EMEI_CHECK_ALIGN16(state0);
  EMEI_CHECK_ALIGN16(states);
  if (obs) EMEI_CHECK_ALIGN16(obs);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const bool ip = p->variant >= EMEI_IP_REBOUND_BALANCING;
#define EMEI_GO(IPV, FRV) launch_cartpole_trajectory<IPV, FRV, R>(state0, actions, states, obs, rewards, dones, n, horizon, *p, s)
  if constexpr (sizeof(R) == 4) {  // the float32 step's instantiations (cartpole_step_f32_tma_dispatch)
    if (!ip) {
      if (p->freq_rate == 1) EMEI_GO(false, 1);
      else if (p->freq_rate == 4) EMEI_GO(false, 4);
      else EMEI_GO(false, 0);
    } else {
      if (p->freq_rate == 1) EMEI_GO(true, 1);
      else if (p->freq_rate == 4) EMEI_GO(true, 4);
      else EMEI_GO(true, 0);
    }
  } else {
    if (!ip) EMEI_GO(false, 0); else EMEI_GO(true, 0);
  }
#undef EMEI_GO
  return launch_status();
}

template <typename R>
int cartpole_trajectory_vjp(const R* states, const void* actions, const R* g_states, const R* g_obs, const R* g_rewards, R* g_state0,
                            R* g_actions, int64_t n, int64_t horizon, const emei_cartpole_params* p, emei_stream_t stream) {
  if (n < 0 || horizon < 0) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(p);
  if (const int e = check_cartpole_params(*p)) return e;
  if (g_actions != nullptr && p->action_kind < EMEI_ACTION_CONTINUOUS_F32) return EMEI_ERR_BAD_ACTION_KIND;
  if (n == 0 || horizon == 0) return EMEI_OK;
  EMEI_CHECK_PTR(states);
  EMEI_CHECK_PTR(actions);
  EMEI_CHECK_PTR(g_state0);
  EMEI_CHECK_ALIGN16(states);
  EMEI_CHECK_ALIGN16(g_state0);
  if (g_states) EMEI_CHECK_ALIGN16(g_states);
  if (g_obs) EMEI_CHECK_ALIGN16(g_obs);
  const CartPoleConsts<R> k = make_cartpole_consts<R>(*p);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
#define EMEI_LAUNCH(IPV)                                                                                                     \
  cartpole_trajectory_vjp_kernel<R, IPV><<<resident_grid(cartpole_trajectory_vjp_kernel<R, IPV>, n), kBlock, 0, s>>>(        \
      states, actions, g_states, g_obs, g_rewards, g_state0, g_actions, n, horizon, k)
  if (p->variant >= EMEI_IP_REBOUND_BALANCING) EMEI_LAUNCH(true); else EMEI_LAUNCH(false);
#undef EMEI_LAUNCH
  return launch_status();
}

// ---------------------------------------------------------------------------------------------
// inverted double pendulum
// ---------------------------------------------------------------------------------------------
template <typename R, int AK>
__global__ void __launch_bounds__(kBlock)
    i2p_trajectory_kernel(const R* __restrict__ state0, const void* __restrict__ actions, R* __restrict__ states, R* __restrict__ obs,
                          R* __restrict__ rewards, uint8_t* __restrict__ dones, int64_t n, int64_t horizon, bool vec2,
                          const I2PConsts<R> k) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * kBlock;
  const NoiseConsts z = {};
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x; i < n; i += stride) {
    R y[6];
    i2p_load_row<R>(state0, i, vec2, y);
    i2p_store_row<R>(states, i, vec2, y);
    R ctrl = load_ctrl<R>(actions, i, AK);
    for (int64_t t = 0, e = i; t < horizon; ++t, e += n) {
      const R ctrl_next = t + 1 < horizon ? load_ctrl<R>(actions, e + n, AK) : R(0);
      R o[6], rew;
      bool notdone;
      i2p_env_step<R>(y, ctrl, k, z, 0ull, 0ull, o, rew, notdone);
      i2p_store_row<R>(states, e + n, vec2, y);
      if (obs != nullptr) i2p_store_row<R>(obs, e, vec2, o);
      rewards[e] = rew;
      if (dones != nullptr) dones[e] = notdone ? 0 : 1;
      ctrl = ctrl_next;
    }
  }
}

template <typename R>
__global__ void __launch_bounds__(kBlock)
    i2p_trajectory_vjp_kernel(const R* __restrict__ states, const void* __restrict__ actions, const R* __restrict__ g_states,
                              const R* __restrict__ g_obs, const R* __restrict__ g_rewards, R* __restrict__ g_state0,
                              R* __restrict__ g_actions, int64_t n, int64_t horizon, bool vec2, const I2PConsts<R> k) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * kBlock;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x; i < n; i += stride) {
    R carry[6] = {R(0), R(0), R(0), R(0), R(0), R(0)};
    int64_t e = (horizon - 1) * n + i;
    R row[6], F, dF;
    i2p_load_row<R>(states, e, vec2, row);
    i2p_force_and_slope<R>(actions, e, k, F, dF);
    for (int64_t t = horizon - 1; t >= 0; --t, e -= n) {
      R y[6], T[6][7], wr[6], F_prev = R(0), dF_prev = R(0);
#pragma unroll
      for (int r = 0; r < 6; ++r) y[r] = row[r];
      if (t > 0) {  // step t-1's inputs, requested before step t's tangent math
        i2p_load_row<R>(states, e - n, vec2, row);
        i2p_force_and_slope<R>(actions, e - n, k, F_prev, dF_prev);
      }
      i2p_tangent<R>(y, T, F, dF, k);
      i2p_reward_slope<R>(y, k, wr);
      R w[6], gs[6], go[6];
      if (g_states != nullptr) i2p_load_row<R>(g_states, e + n, vec2, gs);
      if (g_obs != nullptr) i2p_load_row<R>(g_obs, e, vec2, go);
      const R gr = g_rewards != nullptr ? g_rewards[e] : R(0);
#pragma unroll
      for (int r = 0; r < 6; ++r) {
        const R slope = (r == 1 || r == 2) ? k.pi : R(1);
        w[r] = carry[r] + (g_states != nullptr ? gs[r] : R(0)) + (g_obs != nullptr ? slope * go[r] : R(0)) + gr * wr[r];
      }
      R ga = R(0);
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        R acc = R(0);
#pragma unroll
        for (int r = 0; r < 6; ++r) acc += w[r] * T[r][c];
        carry[c] = acc;
      }
#pragma unroll
      for (int r = 0; r < 6; ++r) ga += w[r] * T[r][6];
      if (g_actions != nullptr) g_actions[e] = ga;
      F = F_prev, dF = dF_prev;
    }
    if (g_states != nullptr) {
      R gs[6];
      i2p_load_row<R>(g_states, i, vec2, gs);
#pragma unroll
      for (int r = 0; r < 6; ++r) carry[r] = carry[r] + gs[r];
    }
    i2p_store_row<R>(g_state0, i, vec2, carry);
  }
}

inline bool rows_vec2(uintptr_t amask, const void* a, const void* b, const void* c, const void* d) {
  return ((reinterpret_cast<uintptr_t>(a) | reinterpret_cast<uintptr_t>(b) | reinterpret_cast<uintptr_t>(c) |
           reinterpret_cast<uintptr_t>(d)) & amask) == 0;
}

template <typename R>
int i2p_trajectory(const R* state0, const void* actions, R* states, R* obs, R* rewards, uint8_t* dones, int64_t n, int64_t horizon,
                   const emei_i2p_params* p, emei_stream_t stream) {
  if (n < 0 || horizon < 0) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(p);
  if (const int e = check_i2p_params(*p)) return e;
  if (n == 0 || horizon == 0) return EMEI_OK;
  EMEI_CHECK_PTR(state0);
  EMEI_CHECK_PTR(actions);
  EMEI_CHECK_PTR(states);
  EMEI_CHECK_PTR(rewards);
  const bool vec2 = rows_vec2(2 * sizeof(R) - 1, state0, states, obs, nullptr);  // every row array 2-element aligned
  const I2PConsts<R> k = make_i2p_consts<R>(*p);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  with_action_kind(p->action_kind, [&](auto ak) {
    constexpr int AK = decltype(ak)::value;
    i2p_trajectory_kernel<R, AK><<<resident_grid(i2p_trajectory_kernel<R, AK>, n), kBlock, 0, s>>>(state0, actions, states, obs, rewards,
                                                                                                  dones, n, horizon, vec2, k);
  });
  return launch_status();
}

template <typename R>
int i2p_trajectory_vjp(const R* states, const void* actions, const R* g_states, const R* g_obs, const R* g_rewards, R* g_state0,
                       R* g_actions, int64_t n, int64_t horizon, const emei_i2p_params* p, emei_stream_t stream) {
  if (n < 0 || horizon < 0) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(p);
  if (const int e = check_i2p_params(*p)) return e;
  if (g_actions != nullptr && p->action_kind < EMEI_ACTION_CONTINUOUS_F32) return EMEI_ERR_BAD_ACTION_KIND;
  if (n == 0 || horizon == 0) return EMEI_OK;
  EMEI_CHECK_PTR(states);
  EMEI_CHECK_PTR(actions);
  EMEI_CHECK_PTR(g_state0);
  const bool vec2 = rows_vec2(2 * sizeof(R) - 1, states, g_states, g_obs, g_state0);
  const I2PConsts<R> k = make_i2p_consts<R>(*p);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  i2p_trajectory_vjp_kernel<R><<<resident_grid(i2p_trajectory_vjp_kernel<R>, n), kBlock, 0, s>>>(
      states, actions, g_states, g_obs, g_rewards, g_state0, g_actions, n, horizon, vec2, k);
  return launch_status();
}

}  // namespace emei
