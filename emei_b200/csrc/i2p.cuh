// Analytic inverted double pendulum step (SURVEY 8f rank 3), both precisions.
//
// The reference's I2P accelerations come from MuJoCo's mj_step (third-party).  What is implemented is the
// reference's own Lagrangian model of classic_control/auxiliary/lagrange_eqs.py:12-60 cartpole(2) (cart + two
// thin rods, relative hinge angles, inertia 1/3 m l^2 about the COM) with the COMPLETE potential energy -- the
// script omits the height of pole 1's hinge for n >= 2 (lagrange_eqs.py:45; see oracle/gen_golden_i2p.py) --
// the XML's constants (inverted_double_pendulum.xml:25,31,32,35,38,45), the forward-Euler rule of
// mujoco_env.py:91-97, the observation of inverted_double_pendulum.py:56-60 (precedence quirk replicated) and the
// reward / terminal of :84-90,114-122,150-157,185-196 on that observation, fused into the same kernel.
//
// A(q) a = b(q, qd, F), symmetric 3x3, solved by LDL^T in the operation order of oracle/emei_oracle.py:i2p_accel
// (float64 is compiled with -fmad=false: same bits as the oracle up to the 1-ulp difference of CUDA's sin/cos).
// One env per thread, persistent grid-stride; state [n,6] = [x, th0, th1, v, w0, w1] (qpos||qvel).
#pragma once
#include "common.cuh"
#include "f32math.cuh"

namespace emei {

template <typename R>
struct I2PConsts {
  R k_a, k_b, k_c, k_d, k_e, k_g1, g, l0, a00, gear, ctrl_low, ctrl_high, dt, pi, x_left, x_right;
  int freq_rate, swingup, action_kind, variant;
};

template <typename R>
inline I2PConsts<R> make_i2p_consts(const emei_i2p_params& p) {
  I2PConsts<R> k;
  const R M = static_cast<R>(p.mass_cart), m0 = static_cast<R>(p.mass_pole0), m1 = static_cast<R>(p.mass_pole1);
  const R l0 = static_cast<R>(p.length0), l1 = static_cast<R>(p.length1), g = static_cast<R>(p.gravity);
  // the same expressions, in the same order, as the oracle (evaluated in R on the host: IEEE, no contraction)
  k.k_a = (m0 + R(2) * m1) * l0;
  k.k_b = m1 * l1;
  k.k_c = R(2) * m1 * l0 * l1;
  k.k_d = static_cast<R>(4.0 / 3.0) * m1 * l1 * l1;
  k.k_e = static_cast<R>(4.0 / 3.0) * m0 * l0 * l0 + R(4) * m1 * l0 * l0 + k.k_d;
  k.k_g1 = g * l0 * (m0 + R(2) * m1);
  k.g = g;
  k.l0 = l0;
  k.a00 = M + m0 + m1;
  k.gear = static_cast<R>(p.gear);
  k.ctrl_low = static_cast<R>(p.ctrl_low);
  k.ctrl_high = static_cast<R>(p.ctrl_high);
  k.dt = static_cast<R>(p.dt);
  k.pi = static_cast<R>(3.141592653589793238462643383279502884);
  k.freq_rate = p.freq_rate;
  k.swingup = (p.variant == EMEI_I2P_REBOUND_SWINGUP || p.variant == EMEI_I2P_BOUNDARY_SWINGUP) ? 1 : 0;
  k.action_kind = p.action_kind;
  k.x_left = static_cast<R>(p.x_left);
  k.x_right = static_cast<R>(p.x_right);
  k.variant = p.variant;
  return k;
}

// sin / cos of th0, th1 and th0 + th1.  float32: the lean kernels of f32math.cuh for th0 and th1 and the
// angle-addition formulas for the sum (two sincos instead of three; libm when an angle is beyond their range);
// float64: libm, in the oracle's order.
template <typename R>
__device__ __forceinline__ void i2p_sincos3(R th0, R th1, R& s0, R& c0, R& s1, R& c1, R& s01, R& c01) {
  if constexpr (sizeof(R) == 4) {
    if (fabsf(th0) <= f32::kSinCosFastMax && fabsf(th1) <= f32::kSinCosFastMax) {
      f32::sincos_core(th0, &s0, &c0);
      f32::sincos_core(th1, &s1, &c1);
      s01 = fmaf(s0, c1, c0 * s1);
      c01 = fmaf(c0, c1, -(s0 * s1));
      return;
    }
  }
  sincos_r(th0, &s0, &c0);
  sincos_r(th1, &s1, &c1);
  sincos_r(th0 + th1, &s01, &c01);
}
// one 6-element row (24 / 48 bytes) as three 2-element vectors when the array allows it (vec2: base 8- / 16-byte aligned)
template <typename R>
struct Vec2T;
template <>
struct Vec2T<float> {
  using type = float2;
};
template <>
struct Vec2T<double> {
  using type = double2;
};
template <typename R>
__device__ __forceinline__ void i2p_load_row(const R* __restrict__ p, int64_t i, bool vec2, R (&y)[6]) {
  if (vec2) {
    using V = typename Vec2T<R>::type;
    const V* q = reinterpret_cast<const V*>(p) + 3 * i;
    const V a = q[0], b = q[1], c = q[2];
    y[0] = a.x, y[1] = a.y, y[2] = b.x, y[3] = b.y, y[4] = c.x, y[5] = c.y;
  } else {
#pragma unroll
    for (int j = 0; j < 6; ++j) y[j] = p[6 * i + j];
  }
}
template <typename R>
__device__ __forceinline__ void i2p_store_row(R* __restrict__ p, int64_t i, bool vec2, const R (&y)[6]) {
  if (vec2) {
    using V = typename Vec2T<R>::type;
    V* q = reinterpret_cast<V*>(p) + 3 * i;
    V a, b, c;
    a.x = y[0], a.y = y[1], b.x = y[2], b.y = y[3], c.x = y[4], c.y = y[5];
    q[0] = a, q[1] = b, q[2] = c;
  } else {
#pragma unroll
    for (int j = 0; j < 6; ++j) p[6 * i + j] = y[j];
  }
}
// a / b: float32 = one MUFU.RCP (<= 1 ulp) and a multiply; float64 = IEEE division (the oracle's)
template <typename R>
__device__ __forceinline__ R i2p_div(R a, R b) {
  if constexpr (sizeof(R) == 4)
    return a * f32::rcp_fast(b);
  else
    return a / b;
}

// One env step on registers (shared by the step kernel and the rollout kernel of rollout_ref.cuh: same bits):
// dynamics + optional state noise, the observation o and the variant's reward / not-done flag on it.
template <typename R>
__device__ __forceinline__ void i2p_env_step(R (&y)[6], R ctrl, const I2PConsts<R>& k, const NoiseConsts& z, unsigned long long env,
                                             unsigned long long substep0, R (&o)[6], R& rew, bool& notdone) {
  const R sign = k.swingup ? R(-1) : R(1);
  ctrl = ctrl < k.ctrl_low ? k.ctrl_low : (ctrl > k.ctrl_high ? k.ctrl_high : ctrl);  // mj_step clamps ctrl
  const R F = k.gear * ctrl;
  for (int sub = 0; sub < k.freq_rate; ++sub) {
    const R th0 = y[1], th1 = y[2], w0 = y[4], w1 = y[5];
    R s0, c0, s1, c1, s01, c01;
    i2p_sincos3<R>(th0, th1, s0, c0, s1, c1, s01, c01);
    s0 = sign * s0, c0 = sign * c0, s01 = sign * s01, c01 = sign * c01;
    const R a01 = k.k_a * c0 + k.k_b * c01;
    const R a02 = k.k_b * c01;
    const R a11 = k.k_e + R(2) * k.k_c * c1;
    const R a12 = k.k_c * c1 + k.k_d;
    const R a22 = k.k_d;
    const R ws = w0 + w1;
    const R b0 = F + k.k_a * s0 * (w0 * w0) + k.k_b * s01 * (ws * ws);
    const R b1 = k.k_g1 * s0 + k.g * k.k_b * s01 + k.k_c * s1 * (w1 * (R(2) * w0 + w1));
    const R b2 = k.k_b * (k.g * s01 - R(2) * k.l0 * s1 * (w0 * w0));
    const R l10 = i2p_div(a01, k.a00);
    const R l20 = i2p_div(a02, k.a00);
    const R d1 = a11 - l10 * a01;
    const R t12 = a12 - l10 * a02;
    const R l21 = i2p_div(t12, d1);
    const R d2 = a22 - l20 * a02 - l21 * t12;
    const R y1 = b1 - l10 * b0;
    const R y2 = b2 - l20 * b0 - l21 * y1;
    const R z2 = i2p_div(y2, d2);
    const R z1 = i2p_div(y1, d1) - l21 * z2;
    const R z0 = i2p_div(b0, k.a00) - l10 * z1 - l20 * z2;
    // mujoco_env.py:91-97: (q, v) <- (q + v h, v + a h)
    const R q0 = y[0] + y[3] * k.dt, q1 = y[1] + y[4] * k.dt, q2 = y[2] + y[5] * k.dt;
    const R v0 = y[3] + z0 * k.dt, v1 = y[4] + z1 * k.dt, v2 = y[5] + z2 * k.dt;
    y[0] = q0, y[1] = q1, y[2] = q2, y[3] = v0, y[4] = v1, y[5] = v2;
    if (z.on)  // mujoco_env.py:98-104: Gaussian state noise after every sub-step
      add_state_noise<R, 6>(y, z, env, substep0 + static_cast<unsigned long long>(sub));
  }
  // inverted_double_pendulum.py:56-60: (theta + pi) % 2 * pi - pi   (sic)
  o[0] = y[0];
  o[1] = py_mod2(y[1] + k.pi) * k.pi - k.pi;
  o[2] = py_mod2(y[2] + k.pi) * k.pi - k.pi;
  o[3] = y[3], o[4] = y[4], o[5] = y[5];
  // get_batch_reward / get_batch_terminal of the variant on that observation, fused (the expressions of
  // reward_terminal_kernel's I2P families: inverted_double_pendulum.py:84-90,114-122,150-157,185-196)
  bool finite = true;
#pragma unroll
  for (int j = 0; j < 6; ++j) finite = finite && is_finite(o[j]);
  const R yy = cos_obs(o[1]) + cos_obs(o[1] + o[2]);
  const bool in_rail = (k.x_left < o[0]) && (o[0] < k.x_right);
  switch (k.variant) {
    case EMEI_I2P_REBOUND_BALANCING:
      rew = R(1);
      notdone = (yy >= R(1.5)) && finite;
      break;
    case EMEI_I2P_BOUNDARY_BALANCING:
      rew = R(1);
      notdone = (yy >= R(0)) && in_rail && finite;
      break;
    case EMEI_I2P_REBOUND_SWINGUP:
      rew = (R(2) - yy) / R(4);
      notdone = finite;
      break;
    default: {  // EMEI_I2P_BOUNDARY_SWINGUP
      const R vel_penalty = R(5e-3) * (o[4] * o[4]) + R(1e-4) * (o[5] * o[5]);
      rew = (R(2) - yy) / R(4) - vel_penalty;
      notdone = in_rail && finite;
    } break;
  }
}

template <typename R>
__global__ void __launch_bounds__(kBlock)  // (capping float32 at 64 registers for a 4th CTA per SM measured 25 us against 22.3)
    i2p_step_kernel(const R* __restrict__ state_in, R* __restrict__ state_out, R* __restrict__ obs_out,
                    const void* __restrict__ action, R* __restrict__ reward, uint8_t* __restrict__ done, double* stats,
                    int64_t n, const I2PConsts<R> k, const NoiseConsts z) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * kBlock;
  double r_acc = 0.0;
  unsigned d_cnt = 0;
  const uintptr_t amask = 2 * sizeof(R) - 1;  // grid-uniform: all three row arrays aligned for 2-element vectors
  const bool vec2 = ((reinterpret_cast<uintptr_t>(state_in) | reinterpret_cast<uintptr_t>(state_out) | reinterpret_cast<uintptr_t>(obs_out)) & amask) == 0;
  pdl_trigger();
  pdl_wait();
  // The row of the NEXT iteration is requested before this iteration's math: at 76 registers only 768 threads are resident
  // per SM, and one 28-byte row per thread (21 KB per SM) cannot cover the HBM latency; two do.
  int64_t i = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x;
  R y[6], ctrl = R(0);
  if (i < n) {
    i2p_load_row<R>(state_in, i, vec2, y);
    ctrl = load_ctrl<R>(action, i, k.action_kind);
  }
  while (i < n) {
    const int64_t i_next = i + stride;
    R yn[6], ctrl_n = R(0), o[6];
    if (i_next < n) {
      i2p_load_row<R>(state_in, i_next, vec2, yn);
      ctrl_n = load_ctrl<R>(action, i_next, k.action_kind);
    }
    R rew;
    bool notdone;
    i2p_env_step<R>(y, ctrl, k, z, z.env_offset + static_cast<unsigned long long>(i), z.substep0, o, rew, notdone);
    i2p_store_row<R>(state_out, i, vec2, y);
    i2p_store_row<R>(obs_out, i, vec2, o);
    reward[i] = rew;
    done[i] = notdone ? 0 : 1;
    r_acc += static_cast<double>(rew);
    d_cnt += notdone ? 0u : 1u;
#pragma unroll
    for (int c = 0; c < 6; ++c) y[c] = yn[c];
    ctrl = ctrl_n;
    i = i_next;
  }
  block_stats_accumulate_counts(stats, r_acc, d_cnt);
}

// (included at the end of kernels.cuh: reward_terminal<R>() is defined above)
template <typename R>
int i2p_step(const R* state_in, R* state_out, R* obs_out, const void* action, R* reward, uint8_t* done, double* stats,
             int64_t n, const emei_i2p_params* p, emei_stream_t stream, const emei_noise_params* noise = nullptr) {
  if (n < 0) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(p);
  if (const int e = check_i2p_params(*p)) return e;
  if (const int e = check_noise_params(noise, 6)) return e;
  if (n == 0) return EMEI_OK;
  EMEI_CHECK_PTR(state_in);
  EMEI_CHECK_PTR(state_out);
  EMEI_CHECK_PTR(obs_out);
  EMEI_CHECK_PTR(action);
  EMEI_CHECK_PTR(reward);
  EMEI_CHECK_PTR(done);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const I2PConsts<R> k = make_i2p_consts<R>(*p);
  launch_pdl(i2p_step_kernel<R>, resident_grid(i2p_step_kernel<R>, n), kBlock, s, state_in, state_out, obs_out, action, reward,
             done, stats, n, k, make_noise_consts(noise, p->freq_rate));
  return launch_status();
}

}  // namespace emei
