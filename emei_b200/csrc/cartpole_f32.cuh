// float32 (tolerance-mode) cart-pole / analytic inverted-pendulum step: pieces shared by the step kernels
// (cartpole_tma.cuh: TMA-staged, two envs per thread in packed f32x2 registers; the scalar small-batch kernel) and the
// fused rollout kernel (rollout_f32.cuh: two envs per thread, packed) -- constants, action decoding, the scalar
// form of the step, and the reward / terminal / observation of one env.
//
// Replaces BaseControlEnv.step (base_control.py:61-83), ODE_approximation's forward-Euler loop
// (base_control.py:160-164), BaseCartPoleEnv._dsdt (cartpole.py:48-60) and the reward/terminal of
// cartpole.py:124-129,145-151 / inverted_pendulum.py:73-79,103-111,139-146,174-183 for a batch.
// freq_rate 1 and 4 are compiled unrolled; other values use a run-time loop.  The 4-scalar state lives in
// registers across all freq_rate sub-steps: HBM sees one 128-bit load, one 128-bit store (+ action 4 B,
// reward 4 B, done 1 B) per env step = 41 bytes.
#pragma once
#include "common.cuh"
#include "f32math.cuh"

namespace emei {

struct CartPoleF32Consts {
  f32::CartPoleK k;
  float force_mag, x_thr, th_thr, x_left, x_right, ctrl_low, ctrl_high;
  int freq_rate, variant;
};

inline CartPoleF32Consts make_cartpole_f32_consts(const emei_cartpole_params& p) {
  CartPoleF32Consts c;
  c.k.g = static_cast<float>(p.gravity);
  c.k.kpm = static_cast<float>(p.pole_mass_length / p.total_mass);
  c.k.inv_mt = static_cast<float>(1.0 / p.total_mass);
  c.k.den0 = static_cast<float>(p.length * (4.0 / 3.0));
  c.k.den1 = static_cast<float>(p.length * p.mass_pole / p.total_mass);
  c.k.dt = static_cast<float>(p.dt);
  c.force_mag = static_cast<float>(p.force_mag);
  c.x_thr = static_cast<float>(p.x_threshold);
  c.th_thr = static_cast<float>(p.theta_threshold);
  c.x_left = static_cast<float>(p.x_left);
  c.x_right = static_cast<float>(p.x_right);
  c.ctrl_low = static_cast<float>(p.ctrl_low);
  c.ctrl_high = static_cast<float>(p.ctrl_high);
  c.freq_rate = p.freq_rate;
  c.variant = p.variant;
  return c;
}

// raw action value as float (discrete kinds: the integer itself; only an exact 1 means "push right")
template <int AK>
__device__ __forceinline__ float load_action_f32(const void* __restrict__ action, int64_t i) {
  if constexpr (AK == EMEI_ACTION_DISCRETE_U8)
    return static_cast<float>(__ldg(static_cast<const uint8_t*>(action) + i));
  else if constexpr (AK == EMEI_ACTION_DISCRETE_I32)
    return static_cast<float>(__ldg(static_cast<const int32_t*>(action) + i));
  else if constexpr (AK == EMEI_ACTION_DISCRETE_I64)
    return static_cast<float>(__ldg(static_cast<const long long*>(action) + i));
  else if constexpr (AK == EMEI_ACTION_CONTINUOUS_F32)
    return __ldg(static_cast<const float*>(action) + i);
  else
    return static_cast<float>(__ldg(static_cast<const double*>(action) + i));
}

// One env step for the state in registers, scalar form (rollout kernel, small-batch kernel, the cold redo of
// the packed kernel).  FR > 0: compile-time sub-step count (unrolled); FR == 0: run-time k.freq_rate.
// flip = 0x80000000 for the inverted pendulum's swing-up models (pole hangs down at theta = 0).
//
// integrate_fast: f32::cartpole_integrate (one sincos + angle addition).  Returns false when its guard trips
// (|theta| > kSinCosSaneMax, a sub-step increment beyond pi/4, Inf): the caller then restores the state and calls
// integrate_libm (same structure, range-reduced evaluations).  cos_cp = cos of the final cart-pole angle.
template <bool IP, int FR>
__device__ __forceinline__ bool integrate_fast(float4& y, float f_mt, uint32_t flip, const CartPoleF32Consts& k, float& cos_cp) {
  f32::LaneMax<float> dmax;
  const float th0 = fabsf(IP ? y.y : y.z);
  if constexpr (!IP)
    cos_cp = f32::cartpole_integrate<float, FR>(y.x, y.y, y.z, y.w, -f_mt, 0u, k.k, k.freq_rate, dmax);  // [x, x_dot, theta, theta_dot]
  else
    cos_cp = f32::cartpole_integrate<float, FR>(y.x, y.z, y.y, y.w, -f_mt, flip, k.k, k.freq_rate, dmax);  // [x, theta, v, omega]
  return th0 <= f32::kSinCosSaneMax && dmax.m <= f32::kDeltaMax;
}
// The cold path of an env whose guard tripped (a sub-step increment beyond pi/4, i.e. |theta_dot| > 39 rad/s at
// dt = 0.02, or an absurd / non-finite angle).  Same structure as the fast path -- ONE sincos of the stored angle,
// then (sin, cos) ROTATED by each sub-step's increment -- with range-reduced evaluations: libm for theta_0 (any
// magnitude, NaN, Inf), the reduced kernels (libm beyond 1e5) for the increments.  Re-evaluating sincosf of the
// float32 theta at every sub-step instead (the first version of this path) re-rounds theta to float32 between
// sub-steps: at theta = 400 rad that is 1.5e-5 rad per sub-step, which the accelerations (hundreds of rad/s^2 per
// radian for a fast pole) turn into 1e-4 of velocity error per step -- 100 x the absolute envelope.  The rotation
// tracks theta_0 + sum(d) like the reference's float64 angle does.  cos_cp = cos of the final cart-pole angle.
template <bool IP, int FR>
__device__ __noinline__ float4 integrate_libm(float4 y, float f_mt, uint32_t flip, const f32::CartPoleK k, int freq_rate, float* cos_cp) {
  const int fr = FR > 0 ? FR : freq_rate;
  float &x = y.x, &xd = IP ? y.z : y.y, &th = IP ? y.y : y.z, &w = y.w;
  float s, c;
  f32::sincos_libm(th, &s, &c);
  s = f32::u2f(f32::f2u(s) ^ flip);
  c = f32::u2f(f32::f2u(c) ^ flip);
  for (int sub = 0; sub < fr; ++sub) {
    const float d = f32::vmul(w, k.dt);
    f32::cartpole_euler<float>(x, xd, th, w, s, c, -f_mt, k);
    float sd, cd;
    f32::sincos_fast(d, &sd, &cd);
    const float s_next = f32::vfma(s, cd, f32::vmul(c, sd));
    c = f32::vfma(c, cd, f32::vneg(f32::vmul(s, sd)));
    s = s_next;
  }
  *cos_cp = c;
  return y;
}

__device__ __forceinline__ uint32_t ip_flip(bool ip, int variant) {
  return (ip && (variant == EMEI_IP_REBOUND_SWINGUP || variant == EMEI_IP_BOUNDARY_SWINGUP)) ? 0x80000000u : 0u;
}

// force / m_total from the raw action value (cartpole.py:121-122,142-143; continuous: force_mag * action[0];
// IP: gear * clamp(ctrl), mj_step clamps ctrl to ctrlrange)
template <bool IP, int AK>
__device__ __forceinline__ float action_to_f_mt(float a, const CartPoleF32Consts& k) {
  if constexpr (!IP) {
    float force;
    if constexpr (AK <= EMEI_ACTION_DISCRETE_I64)
      force = a == 1.0f ? k.force_mag : -k.force_mag;
    else
      force = k.force_mag * a;
    return force * k.k.inv_mt;
  } else {
    float ctrl = a;
    ctrl = ctrl < k.ctrl_low ? k.ctrl_low : (ctrl > k.ctrl_high ? k.ctrl_high : ctrl);
    return (k.force_mag * ctrl) * k.k.inv_mt;
  }
}

// reward, not-done flag and observation of one env after its step (cartpole.py:124-129,145-151;
// inverted_pendulum.py:45-49,73-79,103-111,139-146,174-183).  cy = cos of the reward angle from the integrator
// (cart-pole: theta; IP: the IP's own theta, i.e. the integrator's value with the flip undone).
template <bool IP>
__device__ __forceinline__ void cartpole_outcome(const float4& y, float cy, const CartPoleF32Consts& k, float& rew, bool& notdone,
                                                 float4& obs) {
  obs = y;
  if constexpr (!IP) {
    if (k.variant == EMEI_CARTPOLE_SWINGUP) {
      rew = fmaf(cy, 0.5f, 0.5f);      // cartpole.py:149-151
      notdone = fabsf(y.x) < k.x_thr;  // cartpole.py:145-147
    } else {
      rew = 1.0f;                                                     // cartpole.py:128-129
      notdone = (fabsf(y.z) < k.th_thr) && (fabsf(y.x) < k.x_thr);  // cartpole.py:124-126
    }
  } else {
    const float th_obs = wrap_pi_f32(y.y);  // observation: theta wrapped to [-pi, pi) (inverted_pendulum.py:45-49)
    obs.y = th_obs;
    const bool finite = isfinite(y.x) && isfinite(th_obs) && isfinite(y.z) && isfinite(y.w);
    const bool in_rail = (k.x_left < y.x) && (y.x < k.x_right);
    switch (k.variant) {
      case EMEI_IP_REBOUND_BALANCING:  // inverted_pendulum.py:73-79
        rew = 1.0f;
        notdone = (cy >= 0.9f) && finite;
        break;
      case EMEI_IP_BOUNDARY_BALANCING:  // :103-111
        rew = 1.0f;
        notdone = (cy >= 0.0f) && in_rail && finite;
        break;
      case EMEI_IP_REBOUND_SWINGUP:  // :139-146
        rew = fmaf(cy, -0.5f, 0.5f);
        notdone = finite;
        break;
      default:  // EMEI_IP_BOUNDARY_SWINGUP :174-183
        rew = fmaf(cy, -0.5f, 0.5f);
        notdone = in_rail && finite;
        break;
    }
  }
}

// the whole step of ONE env in scalar form: same bits as a lane of the packed step kernel
template <bool IP, int FR>
__device__ __forceinline__ void cartpole_step_one(float4& y, float f_mt, uint32_t flip, const CartPoleF32Consts& k, float& rew,
                                                  bool& notdone, float4& obs) {
  const float4 y0 = y;
  float c;
  const bool ok = integrate_fast<IP, FR>(y, f_mt, flip, k, c);
  if (!ok) {
    y = integrate_libm<IP, FR>(y0, f_mt, flip, k.k, k.freq_rate, &c);
  }
  cartpole_outcome<IP>(y, IP ? f32::u2f(f32::f2u(c) ^ flip) : c, k, rew, notdone, obs);
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

template <int AK>
struct ActionStorage {  // element type of the action array
  using type = float;
};
template <> struct ActionStorage<EMEI_ACTION_DISCRETE_U8> { using type = uint8_t; };
template <> struct ActionStorage<EMEI_ACTION_DISCRETE_I32> { using type = int32_t; };
template <> struct ActionStorage<EMEI_ACTION_DISCRETE_I64> { using type = long long; };
template <> struct ActionStorage<EMEI_ACTION_CONTINUOUS_F64> { using type = double; };

constexpr int64_t kCartPoleMaxLaunch = (1ll << 31) - (1ll << 20);  // envs per launch (32-bit index)

inline int action_kind_bytes(int ak) {
  switch (ak) {
    case EMEI_ACTION_DISCRETE_U8: return 1;
    case EMEI_ACTION_DISCRETE_I32: return 4;
    case EMEI_ACTION_DISCRETE_I64: return 8;
    case EMEI_ACTION_CONTINUOUS_F32: return 4;
    default: return 8;
  }
}

}  // namespace emei
