// float32 (tolerance-mode) charged-ball step: freq_rate x update_state(_get_update_info(E))
// (charged_ball.py:54-82) with circle_to_free / free_to_circle / _get_angle / _angle_greater (:25-52),
// reward (:158-160) and terminal (:110-111), in place on the three state arrays.
//
// HBM-bound (56 B/env with uint8 actions): persistent grid (148 SMs x 8 CTAs x 256 threads), grid-stride,
// every load of an env issued before any math, 2048 resident threads/SM (<= 32 registers) so ~50 KB of
// loads are in flight per SM; reward partials stay in a register and are reduced ONCE per thread (the
// per-env warp-shuffle reduction of the first version made the kernel MIO-bound: ncu short-scoreboard
// stalls 54 %, 2.8 TB/s).  The common
// branches (on the circle: two sincos; free flight: four FMAs) use the lean float32 math of
// f32math.cuh; only a landing (rare) evaluates asin / fmod / sqrt through libm.
#pragma once
#include "common.cuh"
#include "f32math.cuh"

namespace emei {

struct ChargedBallF32Consts {
  float mg /* m*g */, inv_mr /* 1/(m*r) */, m_r /* m*r */, inv_m, g, r, inv_r, charge, h, land_thr, eps;
  float r2m1 /* r*r - 1 */, two_eps_r /* 2*eps*r */;
  int freq_rate;
};

inline ChargedBallF32Consts make_cb_f32_consts(const emei_charged_ball_params& p) {
  ChargedBallF32Consts k;
  k.mg = static_cast<float>(p.mass_ball * p.gravity_acc);
  k.inv_mr = static_cast<float>(1.0 / (p.mass_ball * p.radius));
  k.m_r = static_cast<float>(p.mass_ball * p.radius);
  k.inv_m = static_cast<float>(1.0 / p.mass_ball);
  k.g = static_cast<float>(p.gravity_acc);
  k.r = static_cast<float>(p.radius);
  k.inv_r = static_cast<float>(1.0 / p.radius);
  k.charge = static_cast<float>(p.charge);
  k.h = static_cast<float>(p.time_step / p.freq_rate);  // charged_ball.py:58,63
  k.land_thr = static_cast<float>(p.radius * p.radius + 0.001);  // :64
  k.eps = 1e-8f;
  k.r2m1 = static_cast<float>(p.radius * p.radius - 1.0);
  k.two_eps_r = static_cast<float>(2.0 * 1e-8 * p.radius);
  k.freq_rate = p.freq_rate;
  return k;
}

__device__ __forceinline__ float sqrt_fast(float x) {  // sqrt.approx: max relative error 2^-23
  float r;
  asm("sqrt.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(x));
  return r;
}

// atan2(x, c) for c >= 0 (result in [-pi/2, pi/2]): octant reduction to |z| <= tan(pi/8) with ONE MUFU.RCP, then the
// classic single-precision minimax polynomial atan z = z + z^3 P(z^2) (|error| <= 1e-7 there).
__device__ __forceinline__ float cb_atan2_pos(float x, float c) {
  const float ax = fabsf(x);
  const float hi = fmaxf(ax, c), lo = fminf(ax, c);
  const bool mid = lo > 0.41421356237309503f * hi;  // atan(lo / hi) = pi/4 + atan((lo - hi) / (lo + hi))
  const float num = mid ? lo - hi : lo, den = mid ? lo + hi : hi;
  const float z = num * f32::rcp_fast(den), z2 = z * z;
  float pz = fmaf(8.05374449538e-2f, z2, -1.38776856032e-1f);
  pz = fmaf(pz, z2, 1.99777106478e-1f);
  pz = fmaf(pz, z2, -3.33329491539e-1f);
  float a = fmaf(pz * z2, z, z) + (mid ? 0.78539816339744830962f : 0.0f);
  a = ax > c ? 1.57079632679489661923f - a : a;  // the octant swap
  return copysignf(a, x);
}

// charged_ball.py:30-36, evaluated only when a ball lands (2 % of env-steps, but 43 % of warp-steps in a
// rollout, so its length matters).  The reference computes  a = asin(x / (scale * r + 1e-8)).  Evaluating asin of
// a float32 quotient loses half the digits where |x| -> scale (the derivative 1 / sqrt(1 - arg^2) is unbounded), so
// the float32 path uses the identity asin(q) = atan2(q, sqrt(1 - q^2)) with the complement formed WITHOUT
// cancellation: for q = x / D, D = scale * r + eps,
//     D^2 - x^2 = y^2 + scale^2 (r^2 - 1) + 2 eps r scale + eps^2
// (the eps term is what keeps the reference's angle 1.4e-4 rad away from +-pi/2 at y = 0: it is kept).
// Well conditioned everywhere: the landing angle meets the 1e-5 / 1e-6 envelope for every landing position.
// `% 2 pi` of an angle that is already in [-pi/2, 3 pi/2] is one select -- the same bits as fmodf there.
__device__ __forceinline__ float cb_get_angle_f32(float x, float y, float r, float eps, float r2m1, float two_eps_r) {
  const float scale = sqrt_fast(fmaf(x, x, y * y));
  const float c2 = fmaf(y, y, fmaf(scale * scale, r2m1, two_eps_r * scale));  // D^2 - x^2 >= 0 for r >= 1
  const float a = cb_atan2_pos(x, sqrt_fast(fmaxf(c2, 0.0f)));
  const float angle = (y > 0.f) ? a : (3.14159265358979323846f - a);
  (void)eps;
  return angle < 0.f ? angle + 6.28318530717958647692f : angle + 0.0f;  // python `%`: result in [0, 2 pi), +0
}

// sin/cos of the circle angle: lean path for |theta| <= 1e5, libm (Payne-Hanek) beyond / NaN
__device__ __forceinline__ void cb_sincos(float theta, float* s, float* c) {
  if (fabsf(theta) <= f32::kSinCosFastMax)
    f32::sincos_core(theta, s, c);
  else
    sincosf(theta, s, c);
}

// one env's registers.  Invariant kept by cb_env_step: while `on`, (s, c) = sin/cos(theta) -- the value computed
// for circle_to_free at the end of a sub-step is the one the next sub-step's dynamics needs (same function of
// the same float32 theta, so carrying it changes no bit).  Callers that load theta from memory establish the
// invariant with cb_prepare().
struct CBRegs {
  bool on;
  float theta, omega, s, c;
  float4 f;  // x, y, vx, vy
};

__device__ __forceinline__ void cb_prepare(CBRegs& e) {
  e.s = e.c = 0.f;
  if (e.on) cb_sincos(e.theta, &e.s, &e.c);
}

template <int AK>
__device__ __forceinline__ float cb_field(float a, const ChargedBallF32Consts& k) {
  if constexpr (AK <= EMEI_ACTION_DISCRETE_I64)
    return a == 1.0f ? k.charge : -k.charge;  // charged_ball.py:155-156
  else
    return k.charge * a;  // :169-170
}

// freq_rate x update_state(_get_update_info(E)) on one env's registers; returns the reward (:158-160).
// Shared by the step kernel and the fused rollout kernel (rollout_f32.cuh): same bits.
//
// In a rollout nearly every warp holds balls on the ring, balls in flight AND a ball that lands in this very
// step (5 % of env-steps, 85 % of warp-steps), so a warp issues all three paths: they are kept short and share
// ONE sincos site (after the branches) instead of one per path.
// FR > 0: the sub-step count is a compile-time constant (the rollout kernel's freq_rate = 1 instance has no loop at all);
// FR = 0: k.freq_rate at run time.  Same bits either way.
template <int FR = 0>
__device__ __forceinline__ float cb_env_step(CBRegs& e, float E, const ChargedBallF32Consts& k) {
  bool on = e.on;
  float theta = e.theta, omega = e.omega, s = e.s, c = e.c;
  float4 f = e.f;
  const int n_sub = FR > 0 ? FR : k.freq_rate;
#pragma unroll
  for (int sub = 0; sub < n_sub; ++sub) {
    bool on_ring = on;  // took the ring path: (x, y, vx, vy) follow from the new (theta, omega)
    if (on) {
      // _get_update_info :72-78 + update_state :56-61
      const float theta_acc = fmaf(s, k.mg, c * E) * k.inv_mr;
      const bool flag = fmaf(s, E, k.m_r * (omega * omega)) < c * k.mg;  // evaluated on the pre-update state
      theta = fmaf(omega, k.h, theta);
      omega = fmaf(theta_acc, k.h, omega);
      if (flag) on = false;
    } else {
      // _get_update_info :79-82 + update_state :62-66 + free_to_circle :44-52
      const float acc_x = E * k.inv_m;
      const float nx = fmaf(f.z, k.h, f.x), ny = fmaf(f.w, k.h, f.y);
      f.z = fmaf(acc_x, k.h, f.z);
      f.w = fmaf(-k.g, k.h, f.w);
      f.x = nx;
      f.y = ny;
      if (fmaf(f.x, f.x, f.y * f.y) > k.land_thr) {
        on = true;
        theta = cb_get_angle_f32(f.x, f.y, k.r, k.eps, k.r2m1, k.two_eps_r);
        // _angle_greater(_get_angle(vx, vy), theta) (:38-42,48-51) asks whether the velocity direction is ahead
        // of the position direction on the circle of angles, i.e. sin(v_angle - theta) > 0, i.e. the sign of
        // the cross product vx*y - vy*x: same answer as comparing the two angles (wrap rule included) except
        // on the measure-zero set where they coincide or oppose exactly, without a second asin.
        const bool greater = fmaf(f.z, f.y, -(f.w * f.x)) > 0.f;
        const float speed = sqrt_fast(fmaf(f.z, f.z, f.w * f.w)) * k.inv_r;
        omega = greater ? speed : -speed;
      }
    }
    if (on_ring || on) {  // the ONE sincos site: ring lanes (circle_to_free :25-28) and lanes that just landed
      cb_sincos(theta, &s, &c);
      if (on_ring) {
        f.x = s * k.r;
        f.y = c * k.r;
        f.z = omega * f.y;
        f.w = -omega * f.x;
      }
    }
  }
  e.on = on;
  e.theta = theta;
  e.omega = omega;
  e.s = s;
  e.c = c;
  e.f = f;
  return fmaf(-sqrt_fast(fmaf(f.x, f.x, f.y * f.y)), k.inv_r, 1.0f);  // charged_ball.py:158-160
}

// EPT envs per thread per iteration: ALL loads of the EPT envs are issued before any math, so EPT x 26 bytes per thread are in
// flight (the kernel is bound by memory latency x bytes in flight: ncu long-scoreboard stalls, 0.96 eligible warps per cycle).
template <int AK, int EPT, int MINB>
__global__ void __launch_bounds__(kBlock, MINB)
    charged_ball_step_f32_kernel(uint8_t* on_circle, float2* circle, float4* free_state, const void* __restrict__ action,
                                 float* __restrict__ reward, uint8_t* __restrict__ done, double* stats, int64_t n,
                                 const ChargedBallF32Consts k) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * kBlock;
  float r_acc = 0.f;  // <= a few hundred rewards in [-inf, 1] per thread; widened to double for the block reduction
  pdl_trigger();
  pdl_wait();
#pragma unroll 1
  for (int64_t i0 = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x; i0 < n; i0 += stride * EPT) {
    // all loads first
    uint8_t on_u8[EPT];
    float2 c2[EPT];
    float a[EPT];
    CBRegs e[EPT];
#pragma unroll
    for (int u = 0; u < EPT; ++u) {
      const int64_t i = i0 + u * stride;
      if (i < n) {
        on_u8[u] = on_circle[i];
        c2[u] = circle[i];
        e[u].f = free_state[i];
        a[u] = load_action_f32<AK>(action, i);
      }
    }
#pragma unroll
    for (int u = 0; u < EPT; ++u) {
      const int64_t i = i0 + u * stride;
      if (i < n) {
        e[u].on = on_u8[u] != 0;
        e[u].theta = c2[u].x;
        e[u].omega = c2[u].y;
        cb_prepare(e[u]);
        const float rew = cb_env_step(e[u], cb_field<AK>(a[u], k), k);
        on_circle[i] = e[u].on ? 1 : 0;
        circle[i] = make_float2(e[u].theta, e[u].omega);
        free_state[i] = e[u].f;
        reward[i] = rew;
        done[i] = 0;  // charged_ball.py:110-111
        r_acc += rew;
      }
    }
  }
  block_stats_accumulate_counts(stats, static_cast<double>(r_acc), 0u);
}

// Launch shape = <envs per thread><min blocks per SM>.  Measured on the B200 (2^26 envs, profiles/r02_c4_shapes.txt): 1 env x 8 CTAs
// (32 registers, 53 KB of loads in flight per SM) 0.687 ms = 0.835 of the copy peak; 2 x 6: 0.635; 2 x 5: 0.618; 4 x 4
// (64 registers, 106 KB in flight): 0.611 ms = 0.94; shapes that spill (4 x 5, 8 x 3) collapse.  At 2^23 envs (the 8-way
// strong-scaled shard of BASELINE configs[3]) the two ends measure the same (84 vs 86 us), so small batches keep the shape with
// the most CTAs.
// R = float.  A template, so that the translation units that see this header without calling it instantiate none of the kernels.
template <typename R>
inline void charged_ball_step_f32_dispatch(uint8_t* on_circle, R* circle, R* free_state, const void* action, R* reward,
                                           uint8_t* done, double* stats, int64_t n, const emei_charged_ball_params& p,
                                           cudaStream_t s) {
  const ChargedBallF32Consts k = make_cb_f32_consts(p);
  float2* c2 = reinterpret_cast<float2*>(circle);
  float4* f4 = reinterpret_cast<float4*>(free_state);
  const bool large = n >= (int64_t{1} << 24);
#define EMEI_CB_LAUNCH(A, EPT, MINB)                                                                                               \
  launch_pdl(charged_ball_step_f32_kernel<A, EPT, MINB>, persistent_grid((n + EPT - 1) / EPT, kBlock, MINB), kBlock, s, on_circle, c2, f4, \
             action, reward, done, stats, n, k)
  switch (p.action_kind) {
#define EMEI_AK(A)              \
  case A:                       \
    if (large)                  \
      EMEI_CB_LAUNCH(A, 4, 4);  \
    else                        \
      EMEI_CB_LAUNCH(A, 1, 8);  \
    break;
    EMEI_AK(EMEI_ACTION_DISCRETE_U8)
    EMEI_AK(EMEI_ACTION_DISCRETE_I32)
    EMEI_AK(EMEI_ACTION_DISCRETE_I64)
    EMEI_AK(EMEI_ACTION_CONTINUOUS_F32)
    EMEI_AK(EMEI_ACTION_CONTINUOUS_F64)
#undef EMEI_AK
#undef EMEI_CB_LAUNCH
  }
}

}  // namespace emei
