// Templated device code shared by the float32 and float64 translation units.
//
// emei_f32.cu instantiates everything with R=float (FMA contraction allowed: tolerance mode).
// emei_f64.cu instantiates everything with R=double and is compiled with -fmad=false so that the
// evaluation order written here IS the arithmetic that executes (reference-exact mode): the
// expressions below follow the reference's python line by line (file:line cited at each block).
#pragma once
#include "common.cuh"
#include "f32math.cuh"
#include "cartpole_tma.cuh"
#include "charged_ball_f32.cuh"

namespace emei {

// =============================================================================================
// cart-pole / analytic inverted pendulum step
// =============================================================================================
template <typename R>
struct CartPoleConsts {
  R gravity, mass_pole, total_mass, length, pml, four_thirds, force_mag;
  R x_thr, th_thr, x_left, x_right, ctrl_low, ctrl_high;
  R dt;        // sub-step seconds in R
  float dt32;  // float32(dt): the reference multiplies float32 derivatives by a weak python float
  R pi, two_pi;
  int freq_rate, variant, action_kind;
};

template <typename R>
inline CartPoleConsts<R> make_cartpole_consts(const emei_cartpole_params& p) {
  CartPoleConsts<R> k;
  k.gravity = static_cast<R>(p.gravity);
  k.mass_pole = static_cast<R>(p.mass_pole);
  k.total_mass = static_cast<R>(p.total_mass);
  k.length = static_cast<R>(p.length);
  k.pml = static_cast<R>(p.pole_mass_length);
  k.four_thirds = static_cast<R>(4.0 / 3.0);
  k.force_mag = static_cast<R>(p.force_mag);
  k.x_thr = static_cast<R>(p.x_threshold);
  k.th_thr = static_cast<R>(p.theta_threshold);
  k.x_left = static_cast<R>(p.x_left);
  k.x_right = static_cast<R>(p.x_right);
  k.ctrl_low = static_cast<R>(p.ctrl_low);
  k.ctrl_high = static_cast<R>(p.ctrl_high);
  k.dt = static_cast<R>(p.dt);
  k.dt32 = static_cast<float>(p.dt);
  k.pi = static_cast<R>(3.141592653589793238462643383279502884);
  k.two_pi = static_cast<R>(2.0 * 3.141592653589793238462643383279502884);
  k.freq_rate = p.freq_rate;
  k.variant = p.variant;
  k.action_kind = p.action_kind;
  return k;
}

// cartpole.py:51-58, same evaluation order.
template <typename R>
__device__ __forceinline__ void cartpole_accel(R theta_dot, R force, R s, R c, const CartPoleConsts<R>& k, R& x_acc,
                                               R& theta_acc) {
  const R temp = (force + k.pml * (theta_dot * theta_dot) * s) / k.total_mass;
  theta_acc = (k.gravity * s - c * temp) / (k.length * (k.four_thirds - k.mass_pole * (c * c) / k.total_mass));
  x_acc = temp - k.pml * theta_acc * c / k.total_mass;
}

// Euler increment.  float: y + d*dt.  double, cart-pole family: the reference's mixed rule
// y64 += float64(float32(d) * float32(dt))  (cartpole.py:60 + base_control.py:164).
__device__ __forceinline__ float euler_cp(float y, float d, const CartPoleConsts<float>& k) { return y + d * k.dt; }
__device__ __forceinline__ double euler_cp(double y, double d, const CartPoleConsts<double>& k) {
  return y + static_cast<double>(__fmul_rn(static_cast<float>(d), k.dt32));
}

// ---------------------------------------------------------------------------------------------
// Per-sub-step Gaussian state noise ("obs_noise_params": mujoco_env.py:98-104 adds
// additive_gaussian_noise(qpos, qvel) to the simulator state after EVERY sub-step; :197-249 draws one
// N(0, sigma_pos) / N(0, sigma_vel) per hinge/slide joint coordinate).  The reference's stream is numpy's
// global Mersenne Twister; here coordinates 2*pr, 2*pr+1 of env e at global sub-step g are the Box-Muller
// pair of Philox block (g * 4 + pr) keyed by (seed, e) -- same arithmetic as init_gaussian_kernel
// (mirror: oracle/philox.py obs_noise).  on == 0: no noise, no cost beyond one uniform branch.
// ---------------------------------------------------------------------------------------------

// Box-Muller: the standard-normal pair (rad cs, rad sn) of one Philox block (numpy-style 53-bit uniforms, float64
// arithmetic), returned as its three factors so that a caller forms only the products it stores.  The one normal sampler
// of the library: state noise, init_gaussian_kernel and the resets of both rollout kernels.
__device__ __forceinline__ void philox_normal_pair(uint64_t seed, uint64_t env, uint32_t block, uint32_t purpose, double& rad,
                                                   double& cs, double& sn) {
  uint32_t w[4];
  Philox::generate(seed, env, block, purpose, w);
  const double u1 = 1.0 - u01_from_bits(w[0], w[1]);  // (0,1]
  const double u2 = u01_from_bits(w[2], w[3]);
  rad = sqrt(-2.0 * log(u1));
  sincospi(2.0 * u2, &sn, &cs);
}

// Columns 2 pr, 2 pr + 1 of a Gaussian initial state (mujoco_env.py:137-140): mean + sigma * N(0,1), the arithmetic of
// init_gaussian_kernel.  The resets of both rollout kernels.
template <typename T>
__device__ __forceinline__ void gaussian_initial_pair(const double* mean, const double* sigma, uint64_t seed, uint64_t env, int pr, T& v0,
                                                      T& v1) {
  double rad, cs, sn;
  philox_normal_pair(seed, env, static_cast<uint32_t>(pr), kPurposeGaussian, rad, cs, sn);
  v0 = static_cast<T>(__dadd_rn(mean[2 * pr], __dmul_rn(sigma[2 * pr], __dmul_rn(rad, cs))));
  v1 = static_cast<T>(__dadd_rn(mean[2 * pr + 1], __dmul_rn(sigma[2 * pr + 1], __dmul_rn(rad, sn))));
}

struct NoiseConsts {
  double sigma[6];
  unsigned long long seed, env_offset, substep0;  // substep0 = step * freq_rate: global index of this call's first sub-step
  int on;
};
inline NoiseConsts make_noise_consts(const emei_noise_params* z, int freq_rate) {
  NoiseConsts c = {};
  if (z != nullptr) {
    for (int j = 0; j < 6; ++j) c.sigma[j] = z->sigma[j];
    c.seed = z->seed;
    c.env_offset = z->env_offset;
    c.substep0 = z->step * static_cast<unsigned long long>(freq_rate);
    c.on = 1;
  }
  return c;
}
// y[c] += sigma[c] * N(0,1) for c < DIM (DIM even)
template <typename R, int DIM>
__device__ __forceinline__ void add_state_noise(R (&y)[DIM], const NoiseConsts& z, unsigned long long env, unsigned long long g) {
#pragma unroll
  for (int pr = 0; pr < DIM / 2; ++pr) {
    const unsigned long long blk = g * 4ull + static_cast<unsigned long long>(pr);
    double rad, cs, sn;
    philox_normal_pair(z.seed, env, static_cast<uint32_t>(blk), kPurposeObsNoise | (static_cast<uint32_t>(blk >> 32) << 8), rad, cs, sn);
    y[2 * pr] = static_cast<R>(__dadd_rn(static_cast<double>(y[2 * pr]), __dmul_rn(z.sigma[2 * pr], __dmul_rn(rad, cs))));
    y[2 * pr + 1] = static_cast<R>(__dadd_rn(static_cast<double>(y[2 * pr + 1]), __dmul_rn(z.sigma[2 * pr + 1], __dmul_rn(rad, sn))));
  }
}

// cos of an observation angle in the double pendulum's scores (the fused step of i2p.cuh and the I2P scoring families share it,
// so get_batch_reward(obs) equals the step's own reward bit for bit): float32 = the lean kernel of f32math.cuh (|error| <= 7e-8 up to
// |x| = 1e5, libm beyond and for NaN / Inf), float64 = libm like the oracle.
template <typename R>
__device__ __forceinline__ R cos_obs(R x) {
  if constexpr (sizeof(R) == 4)
    return f32::cos_fast(x);
  else
    return cos(x);
}

// One env step on registers: the whole of BaseControlEnv.step for one env (shared by the step kernel and the
// reference-arithmetic rollout kernel of rollout_ref.cuh: same bits).  drive = the force (cart-pole family,
// cartpole.py:121-122,142-143) or the raw control value (IP: clamped to ctrlrange like mj_step, then x gear).
//
// Both precisions take the float64 constants.  The float32 instantiation (the noisy inverted-pendulum step and the
// reference-arithmetic float32 rollouts) runs the float64 step on the widened state and rounds once.  A float32 angle held
// between sub-steps and re-evaluated by sincosf is re-rounded at every sub-step (1.5e-5 rad at |theta| = 300), which the
// accelerations of a fast pole turn into 100+ envelopes of velocity error at freq_rate 4 (DESIGN.md 2).  So the state, the
// reward and the flags are those of the float64 step (the reference's own precision) rounded to float32, and the
// observation's angle is the wrap of the stored float32 angle: the value RefCartPole::observation gives for that state.
template <typename R, bool IP>
__device__ __forceinline__ void cartpole_env_step(Vec4<R>& y, R drive, const CartPoleConsts<double>& k, const NoiseConsts& z,
                                                  unsigned long long env, unsigned long long substep0, R& rew, bool& notdone,
                                                  Vec4<R>& obs) {
  if constexpr (sizeof(R) == 4) {
    Vec4<double> yd = {y.x, y.y, y.z, y.w}, od;
    double rd;
    cartpole_env_step<double, IP>(yd, static_cast<double>(drive), k, z, env, substep0, rd, notdone, od);
    y = {static_cast<float>(yd.x), static_cast<float>(yd.y), static_cast<float>(yd.z), static_cast<float>(yd.w)};
    obs = y;
    if constexpr (IP) obs.y = static_cast<float>(py_mod(static_cast<double>(y.y) + k.pi, k.two_pi) - k.pi);
    rew = static_cast<float>(rd);
  } else if constexpr (!IP) {
    // state = [x, x_dot, theta, theta_dot]; base_control.py:71-74
    const R force = drive;
    for (int sub = 0; sub < k.freq_rate; ++sub) {
      R s, c, x_acc, th_acc;
      sincos_r(y.z, &s, &c);
      cartpole_accel<R>(y.w, force, s, c, k, x_acc, th_acc);
      const R nx = euler_cp(y.x, y.y, k), nxd = euler_cp(y.y, x_acc, k);
      const R nth = euler_cp(y.z, y.w, k), nthd = euler_cp(y.w, th_acc, k);
      y.x = nx, y.y = nxd, y.z = nth, y.w = nthd;
    }
    obs = y;
    if (k.variant == EMEI_CARTPOLE_SWINGUP) {
      rew = (cos_r(y.z) + R(1)) / R(2);     // cartpole.py:149-151
      notdone = abs_r(y.x) < k.x_thr;       // cartpole.py:145-147
    } else {
      rew = R(1);                                                     // cartpole.py:128-129
      notdone = (abs_r(y.z) < k.th_thr) && (abs_r(y.x) < k.x_thr);  // cartpole.py:124-126
    }
  } else {
    // state = [x, theta, v, omega] (qpos||qvel); mujoco_env.py:91-97 forward Euler on the analytic
    // acceleration; SwingUp models hang the pole down at theta=0 -> theta_cartpole = theta + pi.
    const bool swingup = (k.variant == EMEI_IP_REBOUND_SWINGUP) || (k.variant == EMEI_IP_BOUNDARY_SWINGUP);
    const R sign = swingup ? R(-1) : R(1);
    R ctrl = drive;
    ctrl = ctrl < k.ctrl_low ? k.ctrl_low : (ctrl > k.ctrl_high ? k.ctrl_high : ctrl);  // mj_step clamps ctrl
    const R force = k.force_mag * ctrl;  // gear * ctrl (inverted_pendulum.xml:23)
    for (int sub = 0; sub < k.freq_rate; ++sub) {
      R s, c, x_acc, th_acc;
      sincos_r(y.y, &s, &c);
      s = sign * s;
      c = sign * c;
      cartpole_accel<R>(y.w, force, s, c, k, x_acc, th_acc);
      const R nx = y.x + y.z * k.dt, nth = y.y + y.w * k.dt;
      const R nv = y.z + x_acc * k.dt, nw = y.w + th_acc * k.dt;
      y.x = nx, y.y = nth, y.z = nv, y.w = nw;
      if (z.on) {  // mujoco_env.py:98-104
        R q[4] = {y.x, y.y, y.z, y.w};
        add_state_noise<R, 4>(q, z, env, substep0 + static_cast<unsigned long long>(sub));
        y.x = q[0], y.y = q[1], y.z = q[2], y.w = q[3];
      }
    }
    // observation: theta wrapped, inverted_pendulum.py:45-49
    const R th_obs = py_mod(y.y + k.pi, k.two_pi) - k.pi;
    obs = y;
    obs.y = th_obs;
    const bool finite = is_finite(y.x) && is_finite(th_obs) && is_finite(y.z) && is_finite(y.w);
    const R cy = cos_r(th_obs);
    const bool in_rail = (k.x_left < y.x) && (y.x < k.x_right);
    switch (k.variant) {
      case EMEI_IP_REBOUND_BALANCING:  // inverted_pendulum.py:73-79
        rew = R(1);
        notdone = (cy >= R(0.9)) && finite;
        break;
      case EMEI_IP_BOUNDARY_BALANCING:  // :103-111
        rew = R(1);
        notdone = (cy >= R(0)) && in_rail && finite;
        break;
      case EMEI_IP_REBOUND_SWINGUP:  // :139-146
        rew = (R(1) - cy) / R(2);
        notdone = finite;
        break;
      default:  // EMEI_IP_BOUNDARY_SWINGUP :174-183
        rew = (R(1) - cy) / R(2);
        notdone = in_rail && finite;
        break;
    }
  }
}

template <typename R, bool IP>
__global__ void __launch_bounds__(kBlock)
    cartpole_step_kernel(const R* state_in, R* state_out, R* obs_out, const void* __restrict__ action,
                         R* __restrict__ reward, uint8_t* __restrict__ done, double* stats, int64_t n,
                         const CartPoleConsts<double> k, const NoiseConsts z) {
  // persistent grid-stride loop; reward / done partials stay in registers and are reduced once per
  // thread (a per-env shuffle reduction makes streaming kernels MIO-bound, profiles/r01_ncu_full_c4)
  const int64_t stride = static_cast<int64_t>(gridDim.x) * kBlock;
  double r_acc = 0.0;
  unsigned d_cnt = 0;
  pdl_trigger();  // programmatic dependent launch (common.cuh): the next step's CTAs are staged while this grid's tail drains
  pdl_wait();
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x; i < n; i += stride) {
    Vec4<R> y = Vec4<R>::load(state_in + 4 * i), obs;
    const R drive = IP ? load_ctrl<R>(action, i, k.action_kind) : load_force<R>(action, i, k.action_kind, static_cast<R>(k.force_mag));
    R rew;
    bool notdone;
    cartpole_env_step<R, IP>(y, drive, k, z, z.env_offset + static_cast<unsigned long long>(i), z.substep0, rew, notdone, obs);
    y.store(state_out + 4 * i);
    if (obs_out != nullptr) obs.store(obs_out + 4 * i);
    reward[i] = rew;
    done[i] = notdone ? 0 : 1;
    r_acc += static_cast<double>(rew);
    d_cnt += notdone ? 0u : 1u;
  }
  block_stats_accumulate_counts(stats, r_acc, d_cnt);
}

template <typename R>
int cartpole_step(const R* state_in, R* state_out, R* obs_out, const void* action, R* reward, uint8_t* done,
                  double* stats, int64_t n, const emei_cartpole_params* p, emei_stream_t stream,
                  const emei_noise_params* noise = nullptr) {
  if (n < 0) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(p);
  if (const int e = check_cartpole_params(*p)) return e;
  // the noisy step exists for the MuJoCo-shell family only (mujoco_env.py:98-104)
  if (noise != nullptr && p->variant < EMEI_IP_REBOUND_BALANCING) return EMEI_ERR_BAD_VARIANT;
  if (const int e = check_noise_params(noise, 4)) return e;
  if (n == 0) return EMEI_OK;
  EMEI_CHECK_PTR(state_in);
  EMEI_CHECK_PTR(state_out);
  EMEI_CHECK_PTR(action);
  EMEI_CHECK_PTR(reward);
  EMEI_CHECK_PTR(done);
  EMEI_CHECK_ALIGN16(state_in);
  EMEI_CHECK_ALIGN16(state_out);
  if (obs_out) EMEI_CHECK_ALIGN16(obs_out);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if constexpr (sizeof(R) == 4) {  // lean float32 kernel: TMA-staged, packed f32x2 (cartpole_tma.cuh)
    if (noise == nullptr) {        // (the noisy step takes the generic kernel below: Philox + double Box-Muller dominate it)
      cartpole_step_f32_tma_dispatch<R>(state_in, state_out, obs_out, action, reward, done, stats, n, *p, s);
      return launch_status();
    }
  }
  const CartPoleConsts<double> k = make_cartpole_consts<double>(*p);
  const NoiseConsts z = make_noise_consts(noise, p->freq_rate);
  if (p->variant <= EMEI_CARTPOLE_SWINGUP)
    launch_pdl(cartpole_step_kernel<R, false>, resident_grid(cartpole_step_kernel<R, false>, n), kBlock, s, state_in, state_out, obs_out,
               action, reward, done, stats, n, k, z);
  else
    launch_pdl(cartpole_step_kernel<R, true>, resident_grid(cartpole_step_kernel<R, true>, n), kBlock, s, state_in, state_out, obs_out,
               action, reward, done, stats, n, k, z);
  return launch_status();
}

// =============================================================================================
// charged ball step  (charged_ball.py:25-82)
// =============================================================================================
template <typename R>
struct ChargedBallConsts {
  R g, m, r, charge, h, pi, two_pi, eps, land_thr;  // land_thr = r*r + 0.001 (charged_ball.py:64)
  int freq_rate, action_kind;
};

template <typename R>
inline ChargedBallConsts<R> make_cb_consts(const emei_charged_ball_params& p) {
  ChargedBallConsts<R> k;
  k.g = static_cast<R>(p.gravity_acc);
  k.m = static_cast<R>(p.mass_ball);
  k.r = static_cast<R>(p.radius);
  k.charge = static_cast<R>(p.charge);
  k.h = static_cast<R>(p.time_step / p.freq_rate);  // charged_ball.py:58,63
  k.pi = static_cast<R>(3.141592653589793238462643383279502884);
  k.two_pi = static_cast<R>(2.0 * 3.141592653589793238462643383279502884);
  k.eps = static_cast<R>(1e-8);
  k.land_thr = k.r * k.r + static_cast<R>(0.001);
  k.freq_rate = p.freq_rate;
  k.action_kind = p.action_kind;
  return k;
}

// charged_ball.py:30-36.  float32: the cancellation-free form of the lean kernel (charged_ball_f32.cuh).  asin of the float32
// quotient loses half its digits as |x| -> scale, and `scale * r + 1e-8f` rounds to scale * r near r = 1, which puts a landing
// at y = 0 at +-pi/2 instead of 1.4e-4 rad away from it.
template <typename R>
__device__ __forceinline__ R cb_get_angle(R x, R y, const ChargedBallConsts<R>& k) {
  if constexpr (sizeof(R) == 4) return cb_get_angle_f32(x, y, k.r, k.eps, fmaf(k.r, k.r, -1.0f), 2.0f * k.eps * k.r);
  const R scale = sqrt_r(x * x + y * y);
  const R a = asin_r(x / (scale * k.r + k.eps));
  const R angle = (y > R(0)) ? a : (k.pi - a);
  return py_mod(angle, k.two_pi);
}

// F32FORCE (double only): the reference's continuous variant under numpy>=2 evaluates every
// `python_float (op) np.float32` of _get_update_info in float32 (see oracle/emei_oracle.py).
// One env step on registers (shared by the step kernel and the reference-arithmetic rollout kernel); returns the reward.
template <typename R, bool F32FORCE>
__device__ __forceinline__ R charged_ball_env_step(bool& on, R& theta, R& omega, Vec4<R>& f, R E, const ChargedBallConsts<R>& k) {
  [[maybe_unused]] const float E32 = static_cast<float>(E);
  const R gravity = k.m * k.g;
  for (int sub = 0; sub < k.freq_rate; ++sub) {
    if (on) {
      // _get_update_info :72-78 + update_state :56-61 + circle_to_free :25-28
      R s, c;
      sincos_r(theta, &s, &c);
      const R centrifugal = k.m * (omega * omega) * k.r;
      R theta_acc;
      bool flag;
      if constexpr (F32FORCE) {
        const float t = __fadd_rn(static_cast<float>(s * gravity), __fmul_rn(static_cast<float>(c), E32));
        theta_acc = static_cast<R>(__fdiv_rn(t, static_cast<float>(k.m * k.r)));
        flag = centrifugal + static_cast<R>(__fmul_rn(static_cast<float>(s), E32)) < c * gravity;
      } else {
        theta_acc = (s * gravity + c * E) / (k.m * k.r);
        flag = centrifugal + s * E < c * gravity;
      }
      const R theta_n = theta + omega * k.h;
      const R omega_n = omega + theta_acc * k.h;
      theta = theta_n, omega = omega_n;
      R sn, cn;
      sincos_r(theta, &sn, &cn);
      f.x = sn * k.r;
      f.y = cn * k.r;
      f.z = omega * f.y;
      f.w = -omega * f.x;
      if (flag) on = false;
    } else {
      // _get_update_info :79-82 + update_state :62-66 + free_to_circle :44-52
      R acc_x;
      if constexpr (F32FORCE)
        acc_x = static_cast<R>(__fdiv_rn(E32, static_cast<float>(k.m)));
      else
        acc_x = E / k.m;
      const R nx = f.x + f.z * k.h, ny = f.y + f.w * k.h;
      const R nvx = f.z + acc_x * k.h, nvy = f.w + (-k.g) * k.h;
      f.x = nx, f.y = ny, f.z = nvx, f.w = nvy;
      if (f.x * f.x + f.y * f.y > k.land_thr) {
        on = true;
        theta = cb_get_angle<R>(f.x, f.y, k);
        const R v_angle = cb_get_angle<R>(f.z, f.w, k);
        const bool greater = (abs_r(v_angle - theta) < k.pi) ? (v_angle > theta) : (v_angle < theta);  // :38-42
        const R speed = sqrt_r(f.z * f.z + f.w * f.w) / k.r;
        omega = greater ? speed : -speed;
      }
    }
  }
  return R(1) - sqrt_r(f.x * f.x + f.y * f.y) / k.r;  // charged_ball.py:158-160
}

template <typename R, bool F32FORCE>
__global__ void __launch_bounds__(kBlock)
    charged_ball_step_kernel(uint8_t* on_circle, R* circle, R* free_state, const void* __restrict__ action,
                             R* __restrict__ reward, uint8_t* __restrict__ done, double* stats, int64_t n,
                             const ChargedBallConsts<R> k) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * kBlock;
  double r_acc = 0.0;
  // one env ahead: the next iteration's state is requested before this iteration's math (the float64 mode moves 108 B per
  // env and is bound by bytes in flight x memory latency, like the float32 kernel before it took four envs per thread)
  auto load_env = [&](int64_t j, uint8_t& on_u8, R& th, R& om, Vec4<R>& ff, R& EE) {
    on_u8 = on_circle[j];
    if constexpr (sizeof(R) == 4) {
      const float2 c2 = reinterpret_cast<const float2*>(circle)[j];
      th = c2.x, om = c2.y;
    } else {
      const double2 c2 = reinterpret_cast<const double2*>(circle)[j];
      th = c2.x, om = c2.y;
    }
    ff = Vec4<R>::load(free_state + 4 * j);                       // x, y, vx, vy
    EE = load_force<R>(action, j, k.action_kind, k.charge);      // charged_ball.py:155-156,169-170
  };
  int64_t i = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x;
  uint8_t on_u8 = 0, on_n = 0;
  R theta = R(0), omega = R(0), E = R(0), theta_n = R(0), omega_n = R(0), E_n = R(0);
  Vec4<R> f = {R(0), R(0), R(0), R(0)}, f_n = f;
  if (i < n) load_env(i, on_u8, theta, omega, f, E);
  for (; i < n; i += stride) {
    const int64_t i_next = i + stride;
    if (i_next < n) load_env(i_next, on_n, theta_n, omega_n, f_n, E_n);
    bool on = on_u8 != 0;
    const R rew = charged_ball_env_step<R, F32FORCE>(on, theta, omega, f, E, k);
    on_circle[i] = on ? 1 : 0;
    if constexpr (sizeof(R) == 4)
      reinterpret_cast<float2*>(circle)[i] = make_float2(theta, omega);
    else
      reinterpret_cast<double2*>(circle)[i] = make_double2(theta, omega);
    f.store(free_state + 4 * i);
    reward[i] = rew;
    done[i] = 0;  // charged_ball.py:110-111
    r_acc += static_cast<double>(rew);
    on_u8 = on_n, theta = theta_n, omega = omega_n, f = f_n, E = E_n;
  }
  block_stats_accumulate_counts(stats, r_acc, 0u);
}

template <typename R>
int charged_ball_step(uint8_t* on_circle, R* circle, R* free_state, const void* action, R* reward, uint8_t* done,
                      double* stats, int64_t n, const emei_charged_ball_params* p, emei_stream_t stream) {
  if (n < 0) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(p);
  if (const int e = check_charged_ball_params(*p)) return e;
  if (n == 0) return EMEI_OK;
  EMEI_CHECK_PTR(on_circle);
  EMEI_CHECK_PTR(circle);
  EMEI_CHECK_PTR(free_state);
  EMEI_CHECK_PTR(action);
  EMEI_CHECK_PTR(reward);
  EMEI_CHECK_PTR(done);
  EMEI_CHECK_ALIGN16(circle);
  EMEI_CHECK_ALIGN16(free_state);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if constexpr (sizeof(R) == 4) {  // lean float32 kernel (charged_ball_f32.cuh)
    charged_ball_step_f32_dispatch<R>(on_circle, circle, free_state, action, reward, done, stats, n, *p, s);
  } else {
    const ChargedBallConsts<R> k = make_cb_consts<R>(*p);
    if (p->action_kind >= EMEI_ACTION_CONTINUOUS_F32)
      charged_ball_step_kernel<R, true><<<resident_grid(charged_ball_step_kernel<R, true>, n), kBlock, 0, s>>>(
          on_circle, circle, free_state, action, reward, done, stats, n, k);
    else
      charged_ball_step_kernel<R, false><<<resident_grid(charged_ball_step_kernel<R, false>, n), kBlock, 0, s>>>(
          on_circle, circle, free_state, action, reward, done, stats, n, k);
  }
  return launch_status();
}

// =============================================================================================
// scoring: get_batch_reward + get_batch_terminal fused, one row per thread
// =============================================================================================
template <typename R>
struct ScoringConsts {
  int family, terminate_when_unhealthy;
  R fwd_w, ctrl_w, healthy_reward, hs_lo, hs_hi, hz_lo, hz_hi, dt, x_thr, th_thr, x_left, x_right, radius;
};

template <typename R>
inline ScoringConsts<R> make_scoring_consts(const emei_scoring_params& p) {
  ScoringConsts<R> k;
  k.family = p.family;
  k.terminate_when_unhealthy = p.terminate_when_unhealthy;
  k.fwd_w = static_cast<R>(p.forward_reward_weight);
  k.ctrl_w = static_cast<R>(p.ctrl_cost_weight);
  k.healthy_reward = static_cast<R>(p.healthy_reward);
  k.hs_lo = static_cast<R>(p.healthy_state_lo);
  k.hs_hi = static_cast<R>(p.healthy_state_hi);
  k.hz_lo = static_cast<R>(p.healthy_z_lo);
  k.hz_hi = static_cast<R>(p.healthy_z_hi);
  k.dt = static_cast<R>(p.dt);
  k.x_thr = static_cast<R>(p.x_threshold);
  k.th_thr = static_cast<R>(p.theta_threshold);
  k.x_left = static_cast<R>(p.x_left);
  k.x_right = static_cast<R>(p.x_right);
  k.radius = static_cast<R>(p.radius);
  return k;
}

// row loader: widest vector access the row stride allows (16 B when D*sizeof(R) % 16 == 0, else 8 B)
template <typename R, int D>
__device__ __forceinline__ void load_row(const R* __restrict__ base, int64_t row, R (&v)[D]) {
  constexpr int kBytes = D * sizeof(R);
  const char* p = reinterpret_cast<const char*>(base) + row * kBytes;
  if constexpr (kBytes % 16 == 0) {
#pragma unroll
    for (int j = 0; j < kBytes / 16; ++j) {
      const uint4 q = __ldg(reinterpret_cast<const uint4*>(p) + j);
      reinterpret_cast<uint4*>(v)[j] = q;
    }
  } else {
    static_assert(kBytes % 8 == 0, "row stride must be a multiple of 8 bytes");
#pragma unroll
    for (int j = 0; j < kBytes / 8; ++j) {
      const uint2 q = __ldg(reinterpret_cast<const uint2*>(p) + j);
      reinterpret_cast<uint2*>(v)[j] = q;
    }
  }
}

template <typename R, int D>
__device__ __forceinline__ bool row_finite(const R (&o)[D]) {
  bool f = true;
#pragma unroll
  for (int j = 0; j < D; ++j) f = f && is_finite(o[j]);
  return f;
}

template <typename R, int FAMILY>
struct FamilyDim {
  static constexpr int value = (FAMILY == EMEI_HOPPER)        ? 12
                               : (FAMILY == EMEI_HALFCHEETAH) ? 18
                               : (FAMILY >= EMEI_I2P_REBOUND_BALANCING && FAMILY <= EMEI_I2P_BOUNDARY_SWINGUP) ? 6
                                                                                                                : 4;
};

// reward and not-done flag of ONE transition row (o = obs row, p0 = pre_obs[:, 0] for Hopper / HalfCheetah,
// ctrl_cost = ctrl_cost_weight * sum over the WHOLE batch of action^2)
template <typename R, int FAMILY, int D>
__device__ __forceinline__ void score_row(const R (&o)[D], R p0, R ctrl_cost, const ScoringConsts<R>& k, R& rew, bool& notdone) {
  if constexpr (FAMILY == EMEI_CARTPOLE_BALANCING) {  // cartpole.py:124-129
    rew = R(1);
    notdone = (abs_r(o[2]) < k.th_thr) && (abs_r(o[0]) < k.x_thr);
  } else if constexpr (FAMILY == EMEI_CARTPOLE_SWINGUP) {  // cartpole.py:145-151
    rew = (cos_r(o[2]) + R(1)) / R(2);
    notdone = abs_r(o[0]) < k.x_thr;
  } else if constexpr (FAMILY >= EMEI_IP_REBOUND_BALANCING && FAMILY <= EMEI_IP_BOUNDARY_SWINGUP) {
    const bool finite = row_finite<R, D>(o);
    const R cy = cos_r(o[1]);
    const bool in_rail = (k.x_left < o[0]) && (o[0] < k.x_right);
    if constexpr (FAMILY == EMEI_IP_REBOUND_BALANCING) {  // inverted_pendulum.py:73-79
      rew = R(1);
      notdone = (cy >= R(0.9)) && finite;
    } else if constexpr (FAMILY == EMEI_IP_BOUNDARY_BALANCING) {  // :103-111
      rew = R(1);
      notdone = (cy >= R(0)) && in_rail && finite;
    } else if constexpr (FAMILY == EMEI_IP_REBOUND_SWINGUP) {  // :139-146
      rew = (R(1) - cy) / R(2);
      notdone = finite;
    } else {  // :174-183
      rew = (R(1) - cy) / R(2);
      notdone = in_rail && finite;
    }
  } else if constexpr (FAMILY >= EMEI_I2P_REBOUND_BALANCING && FAMILY <= EMEI_I2P_BOUNDARY_SWINGUP) {
    const bool finite = row_finite<R, D>(o);
    const R y = cos_obs(o[1]) + cos_obs(o[1] + o[2]);  // inverted_double_pendulum.py:88 (the fused step's expression: same bits)
    const bool in_rail = (k.x_left < o[0]) && (o[0] < k.x_right);
    if constexpr (FAMILY == EMEI_I2P_REBOUND_BALANCING) {  // :84-90
      rew = R(1);
      notdone = (y >= R(1.5)) && finite;
    } else if constexpr (FAMILY == EMEI_I2P_BOUNDARY_BALANCING) {  // :114-122
      rew = R(1);
      notdone = (y >= R(0)) && in_rail && finite;
    } else if constexpr (FAMILY == EMEI_I2P_REBOUND_SWINGUP) {  // :150-157
      rew = (R(2) - y) / R(4);
      notdone = finite;
    } else {  // :185-196
      const R vel_penalty = R(5e-3) * (o[4] * o[4]) + R(1e-4) * (o[5] * o[5]);
      rew = (R(2) - y) / R(4) - vel_penalty;
      notdone = in_rail && finite;
    }
  } else if constexpr (FAMILY == EMEI_HOPPER) {
    // hopper.py:79-106.  healthy_angle is computed and discarded by the reference (np.logical_and's
    // third positional argument is out=, hopper.py:91) -- replicated: only state and z count.
    bool healthy = (k.hz_lo < o[1]) && (o[1] < k.hz_hi);
#pragma unroll
    for (int j = 2; j < D; ++j) healthy = healthy && (k.hs_lo < o[j]) && (o[j] < k.hs_hi);
    const bool alive = healthy || (k.terminate_when_unhealthy != 0);
    const R x_velocity = (o[0] - p0) / k.dt;
    const R control_cost = ctrl_cost;
    const R healthy_reward = alive ? k.healthy_reward : R(0) * k.healthy_reward;
    rew = healthy_reward + k.fwd_w * x_velocity - control_cost;
    notdone = alive;
  } else if constexpr (FAMILY == EMEI_HALFCHEETAH) {  // half_cheetah.py:59-67
    const R control_cost = ctrl_cost;
    rew = k.fwd_w * (o[0] - p0) / k.dt - control_cost;
    notdone = row_finite<R, D>(o);
  } else {  // EMEI_CHARGED_BALL charged_ball.py:110-111,158-160
    rew = R(1) - sqrt_r(o[0] * o[0] + o[1] * o[1]) / k.radius;
    notdone = true;
  }
}

// 1 / x rounded to nearest, without the division subroutine (whose call made the float64 trajectory VJP spill)
__device__ __forceinline__ float rcp_rn(float x) { return __frcp_rn(x); }
__device__ __forceinline__ double rcp_rn(double x) { return __drcp_rn(x); }

// Does the reward gradient of the family read the observation row?  Constant rewards do not, nor do Hopper / HalfCheetah,
// whose reward is affine in obs[:, 0] and pre_obs[:, 0].
template <int FAMILY>
__host__ __device__ constexpr bool score_grad_reads_obs() {
  return FAMILY == EMEI_CARTPOLE_SWINGUP || FAMILY == EMEI_IP_REBOUND_SWINGUP || FAMILY == EMEI_IP_BOUNDARY_SWINGUP ||
         FAMILY == EMEI_I2P_REBOUND_SWINGUP || FAMILY == EMEI_I2P_BOUNDARY_SWINGUP || FAMILY == EMEI_CHARGED_BALL;
}

// The derivative of score_row's reward, the one place it is written (the row and the trajectory VJP kernels call it, so the
// two layouts give the same bits): go = g * d rew / d o (every column written), gp0 = g * d rew / d p0.  The batch-wide
// control cost's derivative is the action's (ctrl_cost_vjp_kernel); `notdone` and the healthy term are piecewise constant.
template <typename R, int FAMILY, int D>
__device__ __forceinline__ void score_row_grad(const R (&o)[D], R g, const ScoringConsts<R>& k, R (&go)[D], R& gp0) {
#pragma unroll
  for (int c = 0; c < D; ++c) go[c] = R(0);
  gp0 = R(0);
  if constexpr (FAMILY == EMEI_CARTPOLE_SWINGUP) {  // (cos o2 + 1) / 2
    go[2] = -sin_r(o[2]) / R(2) * g;
  } else if constexpr (FAMILY == EMEI_IP_REBOUND_SWINGUP || FAMILY == EMEI_IP_BOUNDARY_SWINGUP) {  // (1 - cos o1) / 2
    go[1] = sin_r(o[1]) / R(2) * g;
  } else if constexpr (FAMILY == EMEI_I2P_REBOUND_SWINGUP || FAMILY == EMEI_I2P_BOUNDARY_SWINGUP) {
    // (2 - cos o1 - cos(o1 + o2)) / 4 [- 5e-3 o4^2 - 1e-4 o5^2]
    const R s12 = sin_r(o[1] + o[2]) / R(4);
    go[1] = (sin_r(o[1]) / R(4) + s12) * g;
    go[2] = s12 * g;
    if constexpr (FAMILY == EMEI_I2P_BOUNDARY_SWINGUP) {
      go[4] = R(-1e-2) * o[4] * g;
      go[5] = R(-2e-4) * o[5] * g;
    }
  } else if constexpr (FAMILY == EMEI_HOPPER || FAMILY == EMEI_HALFCHEETAH) {  // fwd_w (o0 - p0) / dt
    const R v = k.fwd_w * rcp_rn(k.dt) * g;
    go[0] = v;
    gp0 = -v;
  } else if constexpr (FAMILY == EMEI_CHARGED_BALL) {  // 1 - rho / radius; 0 at rho = 0
    const R rho = sqrt_r(o[0] * o[0] + o[1] * o[1]);
    const R s = rho == R(0) ? R(0) : -g / (k.radius * rho);
    go[0] = s * o[0];
    go[1] = s * o[1];
  }
}

template <typename R, int FAMILY>
__global__ void __launch_bounds__(kBlock)
    reward_terminal_kernel(const R* __restrict__ obs, const R* __restrict__ pre_obs, R* __restrict__ reward,
                           uint8_t* __restrict__ done, double* stats, const double* __restrict__ sumsq, int64_t n,
                           const ScoringConsts<R> k) {
  constexpr int D = FamilyDim<R, FAMILY>::value;
  constexpr bool kNeedsPre = FAMILY == EMEI_HOPPER || FAMILY == EMEI_HALFCHEETAH;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * kBlock;
  double r_acc = 0.0;
  unsigned d_cnt = 0;
  [[maybe_unused]] R ctrl_cost = R(0);
  if constexpr (kNeedsPre) ctrl_cost = k.ctrl_w * static_cast<R>(*sumsq);
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x; i < n; i += stride) {
    alignas(16) R o[D];
    load_row<R, D>(obs, i, o);
    R p0 = R(0);
    if constexpr (kNeedsPre) p0 = __ldg(pre_obs + i * D);
    R rew;
    bool notdone;
    score_row<R, FAMILY, D>(o, p0, ctrl_cost, k, rew, notdone);
    reward[i] = rew;
    done[i] = notdone ? 0 : 1;
    r_acc += static_cast<double>(rew);
    d_cnt += notdone ? 0u : 1u;
  }
  block_stats_accumulate_counts(stats, r_acc, d_cnt);
}

// ---------------------------------------------------------------------------------------------
// Trajectory ("sequence") scoring for Hopper / HalfCheetah: rows whose pre_obs IS the observation one time step
// earlier.  An imagined rollout is a tensor obs_seq[T+1, k, D]; its transitions are obs = obs_seq[1:], pre_obs =
// obs_seq[:-1], i.e. pre_obs + k*D == obs: transition row i = t*k + j reads pre_obs[i] == obs[i - k].  Reading
// `pre_obs[:, 0]` as a separate strided column costs the WHOLE pre_obs array in DRAM traffic (a 4-byte column of
// 48 / 72-byte rows touches every 64-byte DRAM atom: ncu measured 1.46x / 1.42x the algorithmic bytes, profiles/
// r01_ncu_full_c3_*.txt), so here a thread owns env column j and walks t, carrying obs[t-1][0] in a register:
// every obs row is read exactly once (65 / 101 B per transition instead of 113 / 173 B of DRAM traffic).
// A thread handles a segment of `seg_len` consecutive time steps (grid.y = segments), reading the one strided
// pre_obs value of its first row; the next row's loads are issued before the current row is scored.
// ---------------------------------------------------------------------------------------------
template <typename R, int FAMILY>
__global__ void __launch_bounds__(kBlock)
    reward_terminal_seq_kernel(const R* __restrict__ obs, const R* __restrict__ pre_obs, R* __restrict__ reward,
                               uint8_t* __restrict__ done, double* stats, const double* __restrict__ sumsq, int64_t n,
                               int64_t k_envs, int64_t seg_len, const ScoringConsts<R> k) {
  constexpr int D = FamilyDim<R, FAMILY>::value;
  const int64_t j = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x;  // env column
  const int64_t t0 = static_cast<int64_t>(blockIdx.y) * seg_len;
  double r_acc = 0.0;
  unsigned d_cnt = 0;
  const R ctrl_cost = k.ctrl_w * static_cast<R>(*sumsq);
  int64_t i = t0 * k_envs + j;  // first transition row of this thread
  if (j < k_envs && i < n) {
    alignas(16) R o[D], nx[D];
    R p0 = __ldg(pre_obs + i * D);
    load_row<R, D>(obs, i, o);
    for (int64_t s = 0; s < seg_len && i < n; ++s) {
      const int64_t i_next = i + k_envs;
      const bool more = s + 1 < seg_len && i_next < n;
      if (more) load_row<R, D>(obs, i_next, nx);
      R rew;
      bool notdone;
      score_row<R, FAMILY, D>(o, p0, ctrl_cost, k, rew, notdone);
      reward[i] = rew;
      done[i] = notdone ? 0 : 1;
      r_acc += static_cast<double>(rew);
      d_cnt += notdone ? 0u : 1u;
      p0 = o[0];
#pragma unroll
      for (int c = 0; c < D; ++c) o[c] = nx[c];
      i = i_next;
    }
  }
  block_stats_accumulate_counts(stats, r_acc, d_cnt);
}

// rows are scored by the sequence kernel when pre_obs + k*D == obs for a column count k that keeps the walk
// coalesced; the address identity alone makes pre_obs[i] and obs[i - k] the same memory, whatever the allocation
constexpr int64_t kSeqMinEnvs = 256;
template <typename R>
inline int64_t scoring_alias_columns(const R* obs, const R* pre_obs, int dim, int64_t n) {
  if (pre_obs == nullptr || obs <= pre_obs) return 0;
  const int64_t diff = obs - pre_obs;  // elements
  if (diff % dim != 0) return 0;
  const int64_t k = diff / dim;
  return (k >= kSeqMinEnvs && k < n) ? k : 0;
}

template <typename R, int FAMILY>
void launch_reward_terminal(const R* obs, const R* pre_obs, R* reward, uint8_t* done, double* stats, const double* sumsq,
                            int64_t n, const ScoringConsts<R>& k, cudaStream_t s) {
  if constexpr (FAMILY == EMEI_HOPPER || FAMILY == EMEI_HALFCHEETAH) {
    const int64_t cols = scoring_alias_columns<R>(obs, pre_obs, FamilyDim<R, FAMILY>::value, n);
    if (cols > 0) {
      const int64_t T = (n + cols - 1) / cols;
      // enough segments for ~2^20 threads in flight, at least 8 time steps each (one strided pre_obs read per segment)
      int64_t segs = ((int64_t{1} << 20) + cols - 1) / cols;
      const int64_t max_segs = (T + 7) / 8;
      if (segs > max_segs) segs = max_segs;
      if (segs < 1) segs = 1;
      if (segs > 65535) segs = 65535;
      const int64_t seg_len = (T + segs - 1) / segs;
      segs = (T + seg_len - 1) / seg_len;
      const dim3 grid(static_cast<unsigned>(grid_for(cols, kBlock)), static_cast<unsigned>(segs), 1);
      reward_terminal_seq_kernel<R, FAMILY><<<grid, kBlock, 0, s>>>(obs, pre_obs, reward, done, stats, sumsq, n, cols, seg_len, k);
      return;
    }
  }
  // without statistics: one row per thread over a full grid (measured 9 % faster than the persistent
  // loop for these load-dominated rows); with statistics: one resident wave, partials in registers
  const int grid = stats == nullptr ? grid_for(n, kBlock) : resident_grid(reward_terminal_kernel<R, FAMILY>, n);
  reward_terminal_kernel<R, FAMILY><<<grid, kBlock, 0, s>>>(obs, pre_obs, reward, done, stats, sumsq, n, k);
}

template <typename R>
int reward_terminal(const R* obs, const R* pre_obs, R* reward, uint8_t* done, double* stats, const double* sumsq,
                    int64_t n, const emei_scoring_params* p, emei_stream_t stream) {
  if (n < 0) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(p);
  if (p->family < 0 || p->family >= EMEI_NUM_FAMILIES) return EMEI_ERR_BAD_VARIANT;
  const bool mj = (p->family == EMEI_HOPPER || p->family == EMEI_HALFCHEETAH);
  if (mj && !(p->dt > 0.0)) return EMEI_ERR_BAD_PARAM;
  if (n == 0) return EMEI_OK;
  EMEI_CHECK_PTR(obs);
  EMEI_CHECK_PTR(reward);
  EMEI_CHECK_PTR(done);
  if (mj) {
    EMEI_CHECK_PTR(pre_obs);
    EMEI_CHECK_PTR(sumsq);
  }
  EMEI_CHECK_ALIGN16(obs);
  const ScoringConsts<R> k = make_scoring_consts<R>(*p);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  switch (p->family) {
#define EMEI_CASE(F)                                                                  \
  case F:                                                                             \
    launch_reward_terminal<R, F>(obs, pre_obs, reward, done, stats, sumsq, n, k, s); \
    break;
    EMEI_CASE(EMEI_CARTPOLE_BALANCING)
    EMEI_CASE(EMEI_CARTPOLE_SWINGUP)
    EMEI_CASE(EMEI_IP_REBOUND_BALANCING)
    EMEI_CASE(EMEI_IP_BOUNDARY_BALANCING)
    EMEI_CASE(EMEI_IP_REBOUND_SWINGUP)
    EMEI_CASE(EMEI_IP_BOUNDARY_SWINGUP)
    EMEI_CASE(EMEI_I2P_REBOUND_BALANCING)
    EMEI_CASE(EMEI_I2P_BOUNDARY_BALANCING)
    EMEI_CASE(EMEI_I2P_REBOUND_SWINGUP)
    EMEI_CASE(EMEI_I2P_BOUNDARY_SWINGUP)
    EMEI_CASE(EMEI_HOPPER)
    EMEI_CASE(EMEI_HALFCHEETAH)
    EMEI_CASE(EMEI_CHARGED_BALL)
#undef EMEI_CASE
  }
  return launch_status();
}

// trajectory form: obs_seq [horizon + 1, n_envs, D]; transition (t, j) has obs = obs_seq[t + 1, j], pre_obs = obs_seq[t, j]
template <typename R>
int reward_terminal_seq(const R* obs_seq, R* reward, uint8_t* done, double* stats, const double* sumsq, int64_t n_envs,
                        int64_t horizon, const emei_scoring_params* p, emei_stream_t stream) {
  if (n_envs < 0 || horizon < 0) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(p);
  if (p->family < 0 || p->family >= EMEI_NUM_FAMILIES) return EMEI_ERR_BAD_VARIANT;
  if (n_envs == 0 || horizon == 0) return EMEI_OK;
  EMEI_CHECK_PTR(obs_seq);
  const int dim = emei_family_obs_dim(p->family);
  // the rows of t >= 1 must keep the 16-byte alignment of the row loader
  if ((static_cast<uint64_t>(n_envs) * dim * sizeof(R)) % 16 != 0) return EMEI_ERR_MISALIGNED;
  return reward_terminal<R>(obs_seq + n_envs * dim, obs_seq, reward, done, stats, sumsq, n_envs * horizon, p, stream);
}

// =============================================================================================
// sum of squares (batch-wide control cost, hopper.py:98 / half_cheetah.py:61)
// =============================================================================================
constexpr int kSumsqMaxBlocks = kNumSMs * 8;

// Deterministic (bit-reproducible run to run) single-launch reduction: every CTA writes its partial
// to workspace[1 + blockIdx]; the last CTA to arrive (ticket counter in workspace[0], left at zero
// again for the next call) adds the partials in index order.  No floating-point atomics: the result
// does not depend on CTA scheduling, so get_batch_reward and get_batch_reward_terminal agree bitwise.
// SQUARE: the sum of squares (sumsq_kernel) or the plain sum (sum_kernel: the batch-wide sum of the reward cotangents that the
// control cost's derivative needs).
template <typename R, bool SQUARE>
__device__ __forceinline__ void batch_sum(const R* __restrict__ x, int64_t n, double* out, double* workspace) {
  // grid-stride, 128-bit loads on the aligned body; double accumulation
  constexpr int V = 16 / sizeof(R);
  auto term = [](double t) { return SQUARE ? t * t : t; };
  const int64_t nvec = n / V;
  double acc = 0.0;
  const int64_t stride = static_cast<int64_t>(gridDim.x) * kBlock;
  // four independent 128-bit loads in flight per thread (a single dependent load per iteration left this pass at
  // 5 TB/s); the summation order per thread is fixed, so the result stays bit-reproducible
  int64_t j = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x;
  for (; j + 3 * stride < nvec; j += 4 * stride) {
    uint4 q[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) q[u] = __ldg(reinterpret_cast<const uint4*>(x) + j + u * stride);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const R* v = reinterpret_cast<const R*>(&q[u]);
#pragma unroll
      for (int e = 0; e < V; ++e) acc += term(static_cast<double>(v[e]));
    }
  }
  for (; j < nvec; j += stride) {
    const uint4 q = __ldg(reinterpret_cast<const uint4*>(x) + j);
    const R* v = reinterpret_cast<const R*>(&q);
#pragma unroll
    for (int e = 0; e < V; ++e) acc += term(static_cast<double>(v[e]));
  }
  if (blockIdx.x == 0 && threadIdx.x < n - nvec * V) {
    acc += term(static_cast<double>(x[nvec * V + threadIdx.x]));
  }
  __shared__ double s_acc[kBlock / 32];
  __shared__ bool s_last;
  acc = warp_sum(acc);
  if ((threadIdx.x & 31) == 0) s_acc[threadIdx.x >> 5] = acc;
  __syncthreads();
  if (threadIdx.x < 32) {
    double t = threadIdx.x < kBlock / 32 ? s_acc[threadIdx.x] : 0.0;
    t = warp_sum(t);
    if (threadIdx.x == 0) {
      workspace[1 + blockIdx.x] = t;
      __threadfence();
      unsigned long long* ticket = reinterpret_cast<unsigned long long*>(workspace);
      s_last = atomicAdd(ticket, 1ull) == gridDim.x - 1;
    }
  }
  __syncthreads();
  if (s_last) {
    __threadfence();
    double t = 0.0;
    for (int j = threadIdx.x; j < static_cast<int>(gridDim.x); j += kBlock) t += __ldcg(workspace + 1 + j);
    t = warp_sum(t);
    if ((threadIdx.x & 31) == 0) s_acc[threadIdx.x >> 5] = t;
    __syncthreads();
    if (threadIdx.x < 32) {
      double u = threadIdx.x < kBlock / 32 ? s_acc[threadIdx.x] : 0.0;
      u = warp_sum(u);
      if (threadIdx.x == 0) {
        *out = u;
        *reinterpret_cast<unsigned long long*>(workspace) = 0ull;  // ready for the next call
      }
    }
  }
}

template <typename R>
__global__ void __launch_bounds__(kBlock) sumsq_kernel(const R* __restrict__ x, int64_t n, double* out, double* workspace) {
  batch_sum<R, true>(x, n, out, workspace);
}

template <typename R>
__global__ void __launch_bounds__(kBlock) sum_kernel(const R* __restrict__ x, int64_t n, double* out, double* workspace) {
  batch_sum<R, false>(x, n, out, workspace);
}

template <typename R, bool SQUARE>
int batch_sum_launch(const R* x, int64_t n_elems, double* out, double* workspace, emei_stream_t stream) {
  if (n_elems < 0) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(out);
  EMEI_CHECK_PTR(workspace);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (n_elems == 0) {
    cudaError_t e = cudaMemsetAsync(out, 0, sizeof(double), s);
    return e == cudaSuccess ? EMEI_OK : static_cast<int>(e);
  }
  EMEI_CHECK_PTR(x);
  EMEI_CHECK_ALIGN16(x);
  constexpr int V = 16 / sizeof(R);
  int64_t want = (n_elems / V + kBlock - 1) / kBlock;
  int grid = static_cast<int>(want < 1 ? 1 : (want > kSumsqMaxBlocks ? kSumsqMaxBlocks : want));
  if constexpr (SQUARE)
    sumsq_kernel<R><<<grid, kBlock, 0, s>>>(x, n_elems, out, workspace);
  else
    sum_kernel<R><<<grid, kBlock, 0, s>>>(x, n_elems, out, workspace);
  return launch_status();
}

template <typename R>
int sumsq(const R* x, int64_t n_elems, double* out, double* workspace, emei_stream_t stream) {
  return batch_sum_launch<R, true>(x, n_elems, out, workspace, stream);
}

template <typename R>
int sum(const R* x, int64_t n_elems, double* out, double* workspace, emei_stream_t stream) {
  return batch_sum_launch<R, false>(x, n_elems, out, workspace, stream);
}

// =============================================================================================
// scoring VJP: d reward / d (obs, pre_obs, action) contracted with the reward cotangent g
// =============================================================================================
// row store: the widest vector access the row stride allows (the mirror of load_row)
template <typename R, int D>
__device__ __forceinline__ void store_row(R* __restrict__ base, int64_t row, const R (&v)[D]) {
  constexpr int kBytes = D * sizeof(R);
  char* p = reinterpret_cast<char*>(base) + row * kBytes;
  if constexpr (kBytes % 16 == 0) {
#pragma unroll
    for (int j = 0; j < kBytes / 16; ++j) reinterpret_cast<uint4*>(p)[j] = reinterpret_cast<const uint4*>(v)[j];
  } else {
    static_assert(kBytes % 8 == 0, "row stride must be a multiple of 8 bytes");
#pragma unroll
    for (int j = 0; j < kBytes / 8; ++j) reinterpret_cast<uint2*>(p)[j] = reinterpret_cast<const uint2*>(v)[j];
  }
}

// Gradient row store of the VJP kernels.  Hopper / HalfCheetah rows are 48-144 bytes: one row per lane spreads each of a warp's
// store instructions over 3-9x the sectors of one contiguous access, and measured 0.21-0.84 of the copy peak.  STAGE: a full
// warp's 32 consecutive rows (one contiguous run, 16-byte aligned) go through the warp's slice of shared memory and leave as
// 16-byte stores at consecutive addresses.  `warp_full` must be uniform across the warp; other warps store row by row.
template <typename R, int D, bool STAGE>
__device__ __forceinline__ void store_grad_row(R* __restrict__ base, int64_t row, const R (&v)[D], R* __restrict__ s_warp,
                                               bool warp_full) {
  if (!STAGE || !warp_full) {
    store_row<R, D>(base, row, v);
    return;
  }
  const int lane = threadIdx.x & 31;
  __syncwarp();  // the previous row's chunks have left s_warp
  store_row<R, D>(s_warp, lane, v);
  __syncwarp();
  constexpr int kChunks = 2 * D * static_cast<int>(sizeof(R));  // 32 rows of D * sizeof(R) bytes in 16-byte chunks
  const uint4* src = reinterpret_cast<const uint4*>(s_warp);
  uint4* dst = reinterpret_cast<uint4*>(base + (row - lane) * D);
#pragma unroll
  for (int q = 0; q < (kChunks + 31) / 32; ++q) {
    const int c = q * 32 + lane;
    if (c < kChunks) dst[c] = src[c];
  }
}

template <int FAMILY>
__host__ __device__ constexpr bool score_grad_stages_rows() {
  return FAMILY == EMEI_HOPPER || FAMILY == EMEI_HALFCHEETAH;
}

// one transition row per thread: g_obs[i] = g[i] d rew / d obs[i], g_pre_obs[i] = g[i] d rew / d pre_obs[i] (dense rows,
// each nullable); the obs row is loaded only where the family's derivative reads it
template <typename R, int FAMILY>
__global__ void __launch_bounds__(kBlock)
    reward_vjp_kernel(const R* __restrict__ obs, const R* __restrict__ g_reward, R* __restrict__ g_obs, R* __restrict__ g_pre_obs,
                      int64_t n, const ScoringConsts<R> k) {
  constexpr int D = FamilyDim<R, FAMILY>::value;
  constexpr bool kStage = score_grad_stages_rows<FAMILY>();
  __shared__ alignas(16) R s_stage[kStage ? kBlock * D : 1];
  R* s_warp = s_stage + (kStage ? (threadIdx.x >> 5) * 32 * D : 0);
  const int64_t i = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x;
  const bool warp_full = static_cast<int64_t>(blockIdx.x) * kBlock + (threadIdx.x | 31) < n;
  if (i >= n) return;  // in the last, partial warp only
  alignas(16) R o[D] = {};
  if constexpr (score_grad_reads_obs<FAMILY>()) load_row<R, D>(obs, i, o);
  alignas(16) R go[D];
  R gp0;
  score_row_grad<R, FAMILY, D>(o, __ldg(g_reward + i), k, go, gp0);
  if (g_obs != nullptr) store_grad_row<R, D, kStage>(g_obs, i, go, s_warp, warp_full);
  if (g_pre_obs != nullptr) {
    alignas(16) R gp[D] = {};
    gp[0] = gp0;
    store_grad_row<R, D, kStage>(g_pre_obs, i, gp, s_warp, warp_full);
  }
}

// Trajectory layout: g_obs_seq[r] = g[r-1] d rew_{r-1} / d obs + g[r] d rew_r / d pre_obs for the T + 1 rows r of obs_seq
// (the first term exists for r >= 1, the second for r < T).  One thread per env column walks a segment of rows (grid.y =
// segments) and carries g[r] to the next row as its g[r-1]: every g_obs_seq row is written once, every cotangent read once,
// plus one boundary neighbour per segment; the next row's loads are issued before the current row's math.
template <typename R, int FAMILY>
__global__ void __launch_bounds__(kBlock)
    reward_seq_vjp_kernel(const R* __restrict__ obs_seq, const R* __restrict__ g_reward, R* __restrict__ g_obs_seq, int64_t n_envs,
                          int64_t horizon, int64_t seg_len, const ScoringConsts<R> k) {
  constexpr int D = FamilyDim<R, FAMILY>::value;
  constexpr bool kReadsObs = score_grad_reads_obs<FAMILY>();
  constexpr bool kStage = score_grad_stages_rows<FAMILY>();
  __shared__ alignas(16) R s_stage[kStage ? kBlock * D : 1];
  R* s_warp = s_stage + (kStage ? (threadIdx.x >> 5) * 32 * D : 0);
  const int64_t j = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x;  // env column
  const int64_t r0 = static_cast<int64_t>(blockIdx.y) * seg_len;
  // a full warp's 32 columns are 32 consecutive rows at every r, and its lanes walk the same rows
  const bool warp_full = static_cast<int64_t>(blockIdx.x) * kBlock + (threadIdx.x | 31) < n_envs;
  if (j >= n_envs || r0 > horizon) return;
  const int64_t r1 = r0 + seg_len < horizon + 1 ? r0 + seg_len : horizon + 1;
  R g_prev = r0 > 0 ? __ldg(g_reward + (r0 - 1) * n_envs + j) : R(0);
  R g_cur = r0 < horizon ? __ldg(g_reward + r0 * n_envs + j) : R(0);
  alignas(16) R o[D] = {}, nx[D] = {};
  if constexpr (kReadsObs) load_row<R, D>(obs_seq, r0 * n_envs + j, o);
  for (int64_t r = r0; r < r1; ++r) {
    const bool more = r + 1 < r1;
    R g_next = R(0);
    if (more) {
      if constexpr (kReadsObs) load_row<R, D>(obs_seq, (r + 1) * n_envs + j, nx);
      if (r + 1 < horizon) g_next = __ldg(g_reward + (r + 1) * n_envs + j);
    }
    alignas(16) R go[D], unused[D];
    R gp0, unused0;
    score_row_grad<R, FAMILY, D>(o, g_prev, k, go, unused0);  // transition r - 1, whose obs is this row
    if (r == 0) {
#pragma unroll
      for (int c = 0; c < D; ++c) go[c] = R(0);
    }
    if (r < horizon) {
      score_row_grad<R, FAMILY, D>(o, g_cur, k, unused, gp0);  // transition r, whose pre_obs is this row
      // one rounded add of the two rounded terms (no FMA contraction): the bits of the one-shot layout's two rows summed
      if constexpr (sizeof(R) == 4)
        go[0] = __fadd_rn(go[0], gp0);
      else
        go[0] = __dadd_rn(go[0], gp0);
    }
    store_grad_row<R, D, kStage>(g_obs_seq, r * n_envs + j, go, s_warp, warp_full);
    g_prev = g_cur;
    g_cur = g_next;
#pragma unroll
    for (int c = 0; c < D; ++c) o[c] = nx[c];
  }
}

// g_action = -2 ctrl_w G action, G = the batch-wide sum of the reward cotangents: one scalar times the whole action tensor,
// streamed flat with 128-bit accesses whatever the row width (12 / 24-byte float32 action rows)
template <typename R>
__global__ void __launch_bounds__(kBlock)
    ctrl_cost_vjp_kernel(const R* __restrict__ action, const double* __restrict__ g_sum, R* __restrict__ g_action, int64_t n_elems,
                         double ctrl_w) {
  constexpr int V = 16 / sizeof(R);
  const R c = static_cast<R>(-2.0 * ctrl_w * *g_sum);
  const int64_t nvec = n_elems / V;
  const int64_t j = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x;
  if (j < nvec) {
    uint4 q = __ldg(reinterpret_cast<const uint4*>(action) + j);
    R* v = reinterpret_cast<R*>(&q);
#pragma unroll
    for (int e = 0; e < V; ++e) v[e] = c * v[e];
    reinterpret_cast<uint4*>(g_action)[j] = q;
  }
  if (blockIdx.x == 0 && threadIdx.x < n_elems - nvec * V) {
    const int64_t t = nvec * V + threadIdx.x;
    g_action[t] = c * action[t];
  }
}

// argument checks shared by both VJP entry points (after the size checks): the order and codes of reward_terminal
template <typename R>
int check_reward_vjp(const R* obs, const R* action, const R* g_reward, const double* g_reward_sum, const R* g_action,
                     const emei_scoring_params* p) {
  const bool mj = p->family == EMEI_HOPPER || p->family == EMEI_HALFCHEETAH;
  const bool reads_obs = !mj && p->family != EMEI_CARTPOLE_BALANCING && p->family != EMEI_IP_REBOUND_BALANCING &&
                         p->family != EMEI_IP_BOUNDARY_BALANCING && p->family != EMEI_I2P_REBOUND_BALANCING &&
                         p->family != EMEI_I2P_BOUNDARY_BALANCING;
  if (reads_obs) EMEI_CHECK_PTR(obs);
  EMEI_CHECK_PTR(g_reward);
  if (g_action != nullptr) {
    if (!mj) return EMEI_ERR_BAD_PARAM;  // no other family's reward reads the action
    EMEI_CHECK_PTR(action);
    EMEI_CHECK_PTR(g_reward_sum);
  }
  if (reads_obs) EMEI_CHECK_ALIGN16(obs);
  if (g_action != nullptr) {
    EMEI_CHECK_ALIGN16(action);
    EMEI_CHECK_ALIGN16(g_action);
  }
  return EMEI_OK;
}

template <typename R>
void launch_ctrl_cost_vjp(const R* action, const double* g_reward_sum, R* g_action, int64_t n_elems, const ScoringConsts<R>& k,
                          cudaStream_t s) {
  constexpr int V = 16 / sizeof(R);
  const int64_t nvec = n_elems / V;
  const int grid = nvec > 0 ? grid_for(nvec, kBlock) : 1;
  ctrl_cost_vjp_kernel<R><<<grid, kBlock, 0, s>>>(action, g_reward_sum, g_action, n_elems, static_cast<double>(k.ctrl_w));
}

#define EMEI_SCORING_FAMILIES(X)                                                                                          \
  X(EMEI_CARTPOLE_BALANCING) X(EMEI_CARTPOLE_SWINGUP) X(EMEI_IP_REBOUND_BALANCING) X(EMEI_IP_BOUNDARY_BALANCING)         \
  X(EMEI_IP_REBOUND_SWINGUP) X(EMEI_IP_BOUNDARY_SWINGUP) X(EMEI_I2P_REBOUND_BALANCING) X(EMEI_I2P_BOUNDARY_BALANCING)    \
  X(EMEI_I2P_REBOUND_SWINGUP) X(EMEI_I2P_BOUNDARY_SWINGUP) X(EMEI_HOPPER) X(EMEI_HALFCHEETAH) X(EMEI_CHARGED_BALL)

template <typename R>
int reward_vjp(const R* obs, const R* action, const R* g_reward, const double* g_reward_sum, R* g_obs, R* g_pre_obs, R* g_action,
               int64_t n, const emei_scoring_params* p, emei_stream_t stream) {
  if (n < 0) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(p);
  if (p->family < 0 || p->family >= EMEI_NUM_FAMILIES) return EMEI_ERR_BAD_VARIANT;
  if ((p->family == EMEI_HOPPER || p->family == EMEI_HALFCHEETAH) && !(p->dt > 0.0)) return EMEI_ERR_BAD_PARAM;
  if (n == 0) return EMEI_OK;
  if (const int e = check_reward_vjp<R>(obs, action, g_reward, g_reward_sum, g_action, p)) return e;
  if (g_obs != nullptr) EMEI_CHECK_ALIGN16(g_obs);
  if (g_pre_obs != nullptr) EMEI_CHECK_ALIGN16(g_pre_obs);
  const ScoringConsts<R> k = make_scoring_consts<R>(*p);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (g_obs != nullptr || g_pre_obs != nullptr) {
    switch (p->family) {
#define EMEI_CASE(F)                                                                                            \
  case F:                                                                                                       \
    reward_vjp_kernel<R, F><<<grid_for(n, kBlock), kBlock, 0, s>>>(obs, g_reward, g_obs, g_pre_obs, n, k); \
    break;
      EMEI_SCORING_FAMILIES(EMEI_CASE)
#undef EMEI_CASE
    }
  }
  if (g_action != nullptr) launch_ctrl_cost_vjp<R>(action, g_reward_sum, g_action, n * emei_family_action_dim(p->family), k, s);
  return launch_status();
}

template <typename R>
int reward_seq_vjp(const R* obs_seq, const R* action, const R* g_reward, const double* g_reward_sum, R* g_obs_seq, R* g_action,
                   int64_t n_envs, int64_t horizon, const emei_scoring_params* p, emei_stream_t stream) {
  if (n_envs < 0 || horizon < 0) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(p);
  if (p->family < 0 || p->family >= EMEI_NUM_FAMILIES) return EMEI_ERR_BAD_VARIANT;
  if ((p->family == EMEI_HOPPER || p->family == EMEI_HALFCHEETAH) && !(p->dt > 0.0)) return EMEI_ERR_BAD_PARAM;
  if (n_envs == 0 || horizon == 0) return EMEI_OK;
  EMEI_CHECK_PTR(g_obs_seq);
  if (const int e = check_reward_vjp<R>(obs_seq, action, g_reward, g_reward_sum, g_action, p)) return e;
  const int dim = emei_family_obs_dim(p->family);
  // the rows of t >= 1 must keep the 16-byte alignment of the row accesses (as emei_reward_terminal_seq_*)
  if ((static_cast<uint64_t>(n_envs) * dim * sizeof(R)) % 16 != 0) return EMEI_ERR_MISALIGNED;
  EMEI_CHECK_ALIGN16(g_obs_seq);
  const ScoringConsts<R> k = make_scoring_consts<R>(*p);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // segments as the forward's walk: ~2^20 threads in flight, at least 8 rows each
  const int64_t rows = horizon + 1;
  int64_t segs = ((int64_t{1} << 20) + n_envs - 1) / n_envs;
  const int64_t max_segs = (rows + 7) / 8;
  if (segs > max_segs) segs = max_segs;
  if (segs < 1) segs = 1;
  if (segs > 65535) segs = 65535;
  const int64_t seg_len = (rows + segs - 1) / segs;
  segs = (rows + seg_len - 1) / seg_len;
  const dim3 grid(static_cast<unsigned>(grid_for(n_envs, kBlock)), static_cast<unsigned>(segs), 1);
  switch (p->family) {
#define EMEI_CASE(F)                                                                                                      \
  case F:                                                                                                                 \
    reward_seq_vjp_kernel<R, F><<<grid, kBlock, 0, s>>>(obs_seq, g_reward, g_obs_seq, n_envs, horizon, seg_len, k); \
    break;
    EMEI_SCORING_FAMILIES(EMEI_CASE)
#undef EMEI_CASE
  }
  if (g_action != nullptr)
    launch_ctrl_cost_vjp<R>(action, g_reward_sum, g_action, horizon * n_envs * emei_family_action_dim(p->family), k, s);
  return launch_status();
}
#undef EMEI_SCORING_FAMILIES

// =============================================================================================
// initial-state sampling (Philox4x32-10; value depends on (seed, env id, column) only)
// =============================================================================================
__host__ __device__ inline double philox_uniform(uint64_t seed, uint64_t env, int col, uint32_t purpose) {
  uint32_t w[4];
  Philox::generate(seed, env, static_cast<uint32_t>(col >> 1), purpose, w);
  return (col & 1) ? u01_from_bits(w[2], w[3]) : u01_from_bits(w[0], w[1]);
}

// Column col of a uniform initial state (cartpole.py:131-132,153-156): numpy Generator.uniform, low + (high-low)*next_double
// (no FMA), + pi on pi_column (cartpole.py:155).  init_uniform_kernel and the resets of rollout_ref.cuh.
__device__ __forceinline__ double uniform_initial_sample(uint64_t seed, uint64_t env, int col, double low, double high, int pi_column) {
  const double u = philox_uniform(seed, env, col, kPurposeUniform);
  double v = __dadd_rn(low, __dmul_rn(high - low, u));
  if (col == pi_column) v = __dadd_rn(v, 3.141592653589793238462643383279502884);
  return v;
}

// Charged-ball initial state (charged_ball.py:84-94): on the ring at theta = pi + U(-0.5, 0.5) with omega = U(-0.5, 0.5)
// (float64 like the reference, then cast to R), f = (x, y, vx, vy) of that ring point.  init_charged_ball_kernel and the
// resets of both rollout kernels.
template <typename R>
__device__ __forceinline__ void charged_ball_initial_sample(uint64_t seed, uint64_t env, R radius, R& th, R& om, R (&f)[4]) {
  const double theta = __dadd_rn(__dadd_rn(-0.5, philox_uniform(seed, env, 0, kPurposeChargedBall)),
                                 3.141592653589793238462643383279502884);
  const double omega = __dadd_rn(-0.5, philox_uniform(seed, env, 1, kPurposeChargedBall));
  th = static_cast<R>(theta);
  om = static_cast<R>(omega);
  R s, c;
  sincos_r(th, &s, &c);
  const R x = s * radius, y = c * radius;
  f[0] = x;
  f[1] = y;
  f[2] = om * y;
  f[3] = -om * x;
}

template <typename R>
__global__ void __launch_bounds__(kBlock)
    init_uniform_kernel(R* __restrict__ out, int64_t n, int dim, double low, double high, int pi_column, uint64_t seed,
                        uint64_t env_offset) {
  const int64_t idx = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x;
  if (idx >= n * dim) return;
  const int64_t row = idx / dim;
  const int col = static_cast<int>(idx - row * dim);
  out[idx] = static_cast<R>(uniform_initial_sample(seed, env_offset + static_cast<uint64_t>(row), col, low, high, pi_column));
}

struct GaussianTable {
  double mean[32];
  double sigma[32];
};

template <typename R>
__global__ void __launch_bounds__(kBlock)
    init_gaussian_kernel(R* __restrict__ out, int64_t n, int dim, const GaussianTable t, uint64_t seed,
                         uint64_t env_offset) {
  // one thread per PAIR of columns (Box-Muller produces two normals per Philox block)
  const int pairs = (dim + 1) >> 1;
  const int64_t idx = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x;
  if (idx >= n * pairs) return;
  const int64_t row = idx / pairs;
  const int pr = static_cast<int>(idx - row * pairs);
  double rad, cs, sn;
  philox_normal_pair(seed, env_offset + static_cast<uint64_t>(row), static_cast<uint32_t>(pr), kPurposeGaussian, rad, cs, sn);
  const int c0 = 2 * pr, c1 = 2 * pr + 1;
  out[row * dim + c0] = static_cast<R>(__dadd_rn(t.mean[c0], __dmul_rn(t.sigma[c0], __dmul_rn(rad, cs))));
  if (c1 < dim) out[row * dim + c1] = static_cast<R>(__dadd_rn(t.mean[c1], __dmul_rn(t.sigma[c1], __dmul_rn(rad, sn))));
}

template <typename R>
__global__ void __launch_bounds__(kBlock)
    init_charged_ball_kernel(uint8_t* __restrict__ on_circle, R* __restrict__ circle, R* __restrict__ free_state,
                             int64_t n, double radius, uint64_t seed, uint64_t env_offset) {
  const int64_t i = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x;
  if (i >= n) return;
  R th, om, f[4];
  charged_ball_initial_sample<R>(seed, env_offset + static_cast<uint64_t>(i), static_cast<R>(radius), th, om, f);
  on_circle[i] = 1;
  circle[2 * i] = th;
  circle[2 * i + 1] = om;
  Vec4<R> v = {f[0], f[1], f[2], f[3]};
  v.store(free_state + 4 * i);
}

template <typename R>
int init_uniform(R* out, int64_t n, int32_t dim, double low, double high, int32_t pi_column, uint64_t seed,
                 uint64_t env_offset, emei_stream_t stream) {
  if (n < 0 || dim < 1) return EMEI_ERR_BAD_SIZE;
  if (n == 0) return EMEI_OK;
  EMEI_CHECK_PTR(out);
  init_uniform_kernel<R><<<grid_for(n * dim, kBlock), kBlock, 0, static_cast<cudaStream_t>(stream)>>>(
      out, n, dim, low, high, pi_column, seed, env_offset);
  return launch_status();
}

template <typename R>
int init_gaussian(R* out, int64_t n, int32_t dim, const double* mean, const double* sigma, uint64_t seed,
                  uint64_t env_offset, emei_stream_t stream) {
  if (n < 0 || dim < 1 || dim > 32) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(mean);
  EMEI_CHECK_PTR(sigma);
  if (n == 0) return EMEI_OK;
  EMEI_CHECK_PTR(out);
  GaussianTable t;
  for (int j = 0; j < 32; ++j) {
    t.mean[j] = j < dim ? mean[j] : 0.0;
    t.sigma[j] = j < dim ? sigma[j] : 0.0;
  }
  const int pairs = (dim + 1) / 2;
  init_gaussian_kernel<R><<<grid_for(n * pairs, kBlock), kBlock, 0, static_cast<cudaStream_t>(stream)>>>(
      out, n, dim, t, seed, env_offset);
  return launch_status();
}

template <typename R>
int init_charged_ball(uint8_t* on_circle, R* circle, R* free_state, int64_t n, double radius, uint64_t seed,
                      uint64_t env_offset, emei_stream_t stream) {
  if (n < 0) return EMEI_ERR_BAD_SIZE;
  if (n == 0) return EMEI_OK;
  EMEI_CHECK_PTR(on_circle);
  EMEI_CHECK_PTR(circle);
  EMEI_CHECK_PTR(free_state);
  EMEI_CHECK_ALIGN16(free_state);
  init_charged_ball_kernel<R><<<grid_for(n, kBlock), kBlock, 0, static_cast<cudaStream_t>(stream)>>>(
      on_circle, circle, free_state, n, radius, seed, env_offset);
  return launch_status();
}

}  // namespace emei

#include "i2p.cuh"
