// Derivatives of the analytic step kernels: batched Jacobians and vector-Jacobian products (autograd's backward) of
// emei_cartpole_step_* (cart-pole family + EMEI_IP_* variants) and emei_i2p_step_*, both precisions.
//
// What is differentiated: the real-valued model the step evaluates -- freq_rate forward-Euler sub-steps of cartpole_accel /
// the I2P solve A(q) z = b(q, qd, F), then the observation, then the variant's reward -- with no state noise.
//   * float64: plain R arithmetic.  The cart-pole family's forward step rounds every Euler increment through float32
//     (euler_cp, the reference's mixed rule); that rounding is piecewise constant and has no useful derivative, so the
//     derivative kernels differentiate y + h f(y) in float64 instead (they agree with a complex-step derivative to ~1e-12;
//     the forward step keeps its reference-exact bits).
//   * float32: the generic device arithmetic (libm sincos), not the lean TMA kernel's: gradients are a tolerance product.
//   * action column: cart-pole continuous force = force_mag * a -> force_mag; IP / I2P force = gear * clamp(ctrl) ->
//     gear where ctrl_low <= ctrl <= ctrl_high (inclusive, as torch.clamp), 0 outside; discrete kinds -> 0.
//   * observation: the IP wrap (th + pi) mod 2pi - pi has slope 1; the I2P current_obs quirk ((th + pi) mod 2) * pi - pi
//     has slope pi on both angles, and the reward on that observation inherits the factor.  `done` is not differentiable.
//
// Method: one env per thread, persistent grid-stride loop.  The primal and a tangent matrix T = d y / d (y_in, a)
// (4x5 cart-pole family, 6x7 I2P) advance together in registers, T <- (I + h N_k) T per sub-step (forward mode).  For
// I2P the sub-step's LDL^T factors of A are reused for the five right-hand sides
//   dz/dth_k = A^-1 (db/dth_k - dA/dth_k z),  dz/dw_k = A^-1 db/dw_k,  dz/dF = A^-1 e0.
// The Jacobian kernel stores T (and w_rew^T T); the VJP kernel contracts T with w = g_state_out + slope * g_obs +
// g_reward * d reward / d y in registers and never writes T.
#pragma once
#include "kernels.cuh"

namespace emei {

// ---------------------------------------------------------------------------------------------
// cart-pole family: y = [x, x_dot, th, th_dot] (cart-pole) or [x, th, v, w] (IP)
// ---------------------------------------------------------------------------------------------
template <typename R, bool IP>
struct CpIdx {
  static constexpr int X = 0, XD = IP ? 2 : 1, TH = IP ? 1 : 2, W = 3;
};

// primal drive -> force and d force / d action (the step's _extract_action / mj_step clamp)
template <typename R, bool IP>
__device__ __forceinline__ void cartpole_force_and_slope(const void* action, int64_t i, const CartPoleConsts<R>& k, R& force, R& dforce) {
  const bool continuous = k.action_kind >= EMEI_ACTION_CONTINUOUS_F32;
  if constexpr (!IP) {
    force = load_force<R>(action, i, k.action_kind, k.force_mag);
    dforce = continuous ? k.force_mag : R(0);
  } else {
    const R ctrl = load_ctrl<R>(action, i, k.action_kind);
    const R cc = ctrl < k.ctrl_low ? k.ctrl_low : (ctrl > k.ctrl_high ? k.ctrl_high : ctrl);
    force = k.force_mag * cc;
    dforce = (continuous && ctrl >= k.ctrl_low && ctrl <= k.ctrl_high) ? k.force_mag : R(0);
  }
}

// freq_rate sub-steps of the primal y and its tangent T = d y / d (y_in, action)
template <typename R, bool IP>
__device__ __forceinline__ void cartpole_tangent(R (&y)[4], R (&T)[4][5], R force, R dforce, const CartPoleConsts<R>& k) {
  using I = CpIdx<R, IP>;
#pragma unroll
  for (int r = 0; r < 4; ++r)
#pragma unroll
    for (int c = 0; c < 5; ++c) T[r][c] = (r == c) ? R(1) : R(0);
  const R sign = (IP && (k.variant == EMEI_IP_REBOUND_SWINGUP || k.variant == EMEI_IP_BOUNDARY_SWINGUP)) ? R(-1) : R(1);
  const R inv_tm = R(1) / k.total_mass, pml_tm = k.pml / k.total_mass, h = k.dt;
  for (int sub = 0; sub < k.freq_rate; ++sub) {
    const R th = y[I::TH], w = y[I::W];
    R s, c;
    sincos_r(th, &s, &c);
    s = sign * s;
    c = sign * c;  // d s / d th = c, d c / d th = -s
    // cartpole_accel and its partials in (th, w, F)
    const R temp = (force + k.pml * (w * w) * s) / k.total_mass;
    const R den = k.length * (k.four_thirds - k.mass_pole * (c * c) / k.total_mass);
    const R th_acc = (k.gravity * s - c * temp) / den;
    const R x_acc = temp - k.pml * th_acc * c / k.total_mass;
    const R inv_den = R(1) / den;
    const R t_th = pml_tm * (w * w) * c, t_w = R(2) * pml_tm * w * s;
    const R den_th = k.length * k.mass_pole * R(2) * c * s * inv_tm;
    const R B_th = (k.gravity * c + s * temp - c * t_th - th_acc * den_th) * inv_den;
    const R B_w = -c * t_w * inv_den;
    const R B_F = -c * inv_tm * inv_den;
    const R A_th = t_th - pml_tm * (B_th * c - th_acc * s);
    const R A_w = t_w - pml_tm * c * B_w;
    const R A_F = inv_tm - pml_tm * c * B_F;
#pragma unroll
    for (int col = 0; col < 5; ++col) {
      const R dth = T[I::TH][col], dw = T[I::W][col], dF = col == 4 ? dforce : R(0);
      const R dxa = A_th * dth + A_w * dw + A_F * dF;
      const R dta = B_th * dth + B_w * dw + B_F * dF;
      T[I::X][col] = T[I::X][col] + h * T[I::XD][col];
      T[I::TH][col] = dth + h * dw;
      T[I::XD][col] = T[I::XD][col] + h * dxa;
      T[I::W][col] = dw + h * dta;
    }
    const R nx = y[I::X] + y[I::XD] * h, nth = th + w * h;
    const R nxd = y[I::XD] + x_acc * h, nw = w + th_acc * h;
    y[I::X] = nx, y[I::TH] = nth, y[I::XD] = nxd, y[I::W] = nw;
  }
}

// d reward / d y_out of the variant (the observation's slope, 1, folded in)
template <typename R, bool IP>
__device__ __forceinline__ void cartpole_reward_slope(const R (&y)[4], const CartPoleConsts<R>& k, R (&wr)[4]) {
  using I = CpIdx<R, IP>;
  wr[0] = wr[1] = wr[2] = wr[3] = R(0);
  if constexpr (!IP) {
    if (k.variant == EMEI_CARTPOLE_SWINGUP) wr[I::TH] = -sin(y[I::TH]) / R(2);  // (cos th + 1) / 2
  } else {
    if (k.variant == EMEI_IP_REBOUND_SWINGUP || k.variant == EMEI_IP_BOUNDARY_SWINGUP) wr[I::TH] = sin(y[I::TH]) / R(2);  // (1 - cos th) / 2
  }
}

template <typename R, bool IP, bool VJP>
__global__ void __launch_bounds__(kBlock)
    cartpole_deriv_kernel(const R* __restrict__ state_in, const void* __restrict__ action, R* __restrict__ jac, R* __restrict__ reward_grad,
                          const R* __restrict__ g_state_out, const R* __restrict__ g_obs, const R* __restrict__ g_reward,
                          R* __restrict__ g_state_in, R* __restrict__ g_action, int64_t n, const CartPoleConsts<R> k) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * kBlock;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x; i < n; i += stride) {
    const Vec4<R> v = Vec4<R>::load(state_in + 4 * i);
    R y[4] = {v.x, v.y, v.z, v.w}, T[4][5], force, dforce, wr[4];
    cartpole_force_and_slope<R, IP>(action, i, k, force, dforce);
    cartpole_tangent<R, IP>(y, T, force, dforce, k);
    cartpole_reward_slope<R, IP>(y, k, wr);
    if constexpr (!VJP) {
      R* J = jac + 20 * i;
#pragma unroll
      for (int r = 0; r < 4; ++r)
#pragma unroll
        for (int c = 0; c < 5; ++c) J[5 * r + c] = T[r][c];
      if (reward_grad != nullptr) {
#pragma unroll
        for (int c = 0; c < 5; ++c) reward_grad[5 * i + c] = wr[0] * T[0][c] + wr[1] * T[1][c] + wr[2] * T[2][c] + wr[3] * T[3][c];
      }
    } else {
      Vec4<R> gs = {R(0), R(0), R(0), R(0)}, go = gs;
      if (g_state_out != nullptr) gs = Vec4<R>::load(g_state_out + 4 * i);
      if (g_obs != nullptr) go = Vec4<R>::load(g_obs + 4 * i);
      const R gr = g_reward != nullptr ? g_reward[i] : R(0);
      const R w[4] = {gs.x + go.x + gr * wr[0], gs.y + go.y + gr * wr[1], gs.z + go.z + gr * wr[2], gs.w + go.w + gr * wr[3]};
      R g[5];
#pragma unroll
      for (int c = 0; c < 5; ++c) g[c] = w[0] * T[0][c] + w[1] * T[1][c] + w[2] * T[2][c] + w[3] * T[3][c];
      const Vec4<R> gi = {g[0], g[1], g[2], g[3]};
      gi.store(g_state_in + 4 * i);
      if (g_action != nullptr) g_action[i] = g[4];
    }
  }
}

template <typename R>
int cartpole_step_derivs(const R* state_in, const void* action, R* jac, R* reward_grad, const R* g_state_out, const R* g_obs,
                         const R* g_reward, R* g_state_in, R* g_action, int64_t n, const emei_cartpole_params* p, emei_stream_t stream,
                         bool vjp) {
  if (n < 0) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(p);
  if (const int e = check_cartpole_params(*p)) return e;
  if (vjp && g_action != nullptr && p->action_kind < EMEI_ACTION_CONTINUOUS_F32) return EMEI_ERR_BAD_ACTION_KIND;
  if (n == 0) return EMEI_OK;
  EMEI_CHECK_PTR(state_in);
  EMEI_CHECK_PTR(action);
  EMEI_CHECK_ALIGN16(state_in);
  if (vjp) {
    EMEI_CHECK_PTR(g_state_in);
    EMEI_CHECK_ALIGN16(g_state_in);
    if (g_state_out) EMEI_CHECK_ALIGN16(g_state_out);
    if (g_obs) EMEI_CHECK_ALIGN16(g_obs);
  } else {
    EMEI_CHECK_PTR(jac);
  }
  const CartPoleConsts<R> k = make_cartpole_consts<R>(*p);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const bool ip = p->variant >= EMEI_IP_REBOUND_BALANCING;
#define EMEI_LAUNCH(IPV, VJPV)                                                                                              \
  cartpole_deriv_kernel<R, IPV, VJPV><<<resident_grid(cartpole_deriv_kernel<R, IPV, VJPV>, n), kBlock, 0, s>>>(            \
      state_in, action, jac, reward_grad, g_state_out, g_obs, g_reward, g_state_in, g_action, n, k)
  if (ip) {
    if (vjp) EMEI_LAUNCH(true, true); else EMEI_LAUNCH(true, false);
  } else {
    if (vjp) EMEI_LAUNCH(false, true); else EMEI_LAUNCH(false, false);
  }
#undef EMEI_LAUNCH
  return launch_status();
}

// ---------------------------------------------------------------------------------------------
// inverted double pendulum: y = [x, th0, th1, v, w0, w1]
// ---------------------------------------------------------------------------------------------
template <typename R>
__device__ __forceinline__ void i2p_tangent(R (&y)[6], R (&T)[6][7], R F, R dF, const I2PConsts<R>& k) {
#pragma unroll
  for (int r = 0; r < 6; ++r)
#pragma unroll
    for (int c = 0; c < 7; ++c) T[r][c] = (r == c) ? R(1) : R(0);
  const R sign = k.swingup ? R(-1) : R(1), h = k.dt, inv_a00 = R(1) / k.a00;
  for (int sub = 0; sub < k.freq_rate; ++sub) {
    const R th0 = y[1], th1 = y[2], w0 = y[4], w1 = y[5];
    R s0, c0, s1, c1, s01, c01;
    sincos_r(th0, &s0, &c0);
    sincos_r(th1, &s1, &c1);
    sincos_r(th0 + th1, &s01, &c01);
    s0 = sign * s0, c0 = sign * c0, s01 = sign * s01, c01 = sign * c01;
    // the forward's A, b and LDL^T factors (i2p_env_step)
    const R a01 = k.k_a * c0 + k.k_b * c01, a02 = k.k_b * c01;
    const R a11 = k.k_e + R(2) * k.k_c * c1, a12 = k.k_c * c1 + k.k_d, a22 = k.k_d;
    const R ws = w0 + w1;
    const R b0 = F + k.k_a * s0 * (w0 * w0) + k.k_b * s01 * (ws * ws);
    const R b1 = k.k_g1 * s0 + k.g * k.k_b * s01 + k.k_c * s1 * (w1 * (R(2) * w0 + w1));
    const R b2 = k.k_b * (k.g * s01 - R(2) * k.l0 * s1 * (w0 * w0));
    const R l10 = a01 * inv_a00, l20 = a02 * inv_a00;
    const R d1 = a11 - l10 * a01, t12 = a12 - l10 * a02;
    const R inv_d1 = R(1) / d1, l21 = t12 * inv_d1;
    const R inv_d2 = R(1) / (a22 - l20 * a02 - l21 * t12);
    auto solve = [&](R r0, R r1, R r2, R& z0, R& z1, R& z2) {
      const R y1 = r1 - l10 * r0, y2 = r2 - l20 * r0 - l21 * y1;
      z2 = y2 * inv_d2;
      z1 = y1 * inv_d1 - l21 * z2;
      z0 = r0 * inv_a00 - l10 * z1 - l20 * z2;
    };
    R z0, z1, z2;
    solve(b0, b1, b2, z0, z1, z2);
    // d z / d (th0, th1, w0, w1, F)
    R D[5][3];
    {  // th0: dA = [[0, e01, e02], [e01, 0, 0], [e02, 0, 0]]
      const R e01 = -k.k_a * s0 - k.k_b * s01, e02 = -k.k_b * s01;
      solve(k.k_a * c0 * (w0 * w0) + k.k_b * c01 * (ws * ws) - (e01 * z1 + e02 * z2),
            k.k_g1 * c0 + k.g * k.k_b * c01 - e01 * z0,
            k.k_b * k.g * c01 - e02 * z0, D[0][0], D[0][1], D[0][2]);
    }
    {  // th1: dA = [[0, e, e], [e, f11, f12], [e, f12, 0]]
      const R e = -k.k_b * s01, f11 = R(-2) * k.k_c * s1, f12 = -k.k_c * s1;
      solve(k.k_b * c01 * (ws * ws) - (e * z1 + e * z2),
            k.g * k.k_b * c01 + k.k_c * c1 * (w1 * (R(2) * w0 + w1)) - (e * z0 + f11 * z1 + f12 * z2),
            k.k_b * (k.g * c01 - R(2) * k.l0 * c1 * (w0 * w0)) - (e * z0 + f12 * z1), D[1][0], D[1][1], D[1][2]);
    }
    solve(R(2) * k.k_a * s0 * w0 + R(2) * k.k_b * s01 * ws, R(2) * k.k_c * s1 * w1, R(-4) * k.k_b * k.l0 * s1 * w0, D[2][0], D[2][1],
          D[2][2]);
    solve(R(2) * k.k_b * s01 * ws, R(2) * k.k_c * s1 * ws, R(0), D[3][0], D[3][1], D[3][2]);
    solve(R(1), R(0), R(0), D[4][0], D[4][1], D[4][2]);
#pragma unroll
    for (int col = 0; col < 7; ++col) {
      const R p0 = T[1][col], p1 = T[2][col], p2 = T[4][col], p3 = T[5][col], pf = col == 6 ? dF : R(0);
#pragma unroll
      for (int j = 0; j < 3; ++j) {
        const R dz = D[0][j] * p0 + D[1][j] * p1 + D[2][j] * p2 + D[3][j] * p3 + D[4][j] * pf;
        T[j][col] = T[j][col] + h * T[3 + j][col];
        T[3 + j][col] = T[3 + j][col] + h * dz;
      }
    }
    const R q0 = y[0] + y[3] * h, q1 = y[1] + y[4] * h, q2 = y[2] + y[5] * h;
    const R v0 = y[3] + z0 * h, v1 = y[4] + z1 * h, v2 = y[5] + z2 * h;
    y[0] = q0, y[1] = q1, y[2] = q2, y[3] = v0, y[4] = v1, y[5] = v2;
  }
}

// primal control -> force gear * clamp(ctrl) and d force / d ctrl (the step's mj_step clamp, inclusive)
template <typename R>
__device__ __forceinline__ void i2p_force_and_slope(const void* action, int64_t i, const I2PConsts<R>& k, R& F, R& dF) {
  const bool continuous = k.action_kind >= EMEI_ACTION_CONTINUOUS_F32;
  const R ctrl = load_ctrl<R>(action, i, k.action_kind);
  const R cc = ctrl < k.ctrl_low ? k.ctrl_low : (ctrl > k.ctrl_high ? k.ctrl_high : ctrl);
  F = k.gear * cc;
  dF = (continuous && ctrl >= k.ctrl_low && ctrl <= k.ctrl_high) ? k.gear : R(0);
}

// d reward / d y_out of the variant, through the observation (slope pi on both angles: the current_obs quirk)
template <typename R>
__device__ __forceinline__ void i2p_reward_slope(const R (&y)[6], const I2PConsts<R>& k, R (&wr)[6]) {
#pragma unroll
  for (int j = 0; j < 6; ++j) wr[j] = R(0);
  if (k.variant == EMEI_I2P_REBOUND_SWINGUP || k.variant == EMEI_I2P_BOUNDARY_SWINGUP) {
    const R o1 = py_mod2(y[1] + k.pi) * k.pi - k.pi, o2 = py_mod2(y[2] + k.pi) * k.pi - k.pi;
    const R s12 = sin(o1 + o2);
    wr[1] = k.pi * (sin(o1) + s12) / R(4);  // (2 - cos o1 - cos(o1 + o2)) / 4
    wr[2] = k.pi * s12 / R(4);
    if (k.variant == EMEI_I2P_BOUNDARY_SWINGUP) {  // - 5e-3 w0^2 - 1e-4 w1^2
      wr[4] = R(-1e-2) * y[4];
      wr[5] = R(-2e-4) * y[5];
    }
  }
}

template <typename R, bool VJP>
__global__ void __launch_bounds__(kBlock)
    i2p_deriv_kernel(const R* __restrict__ state_in, const void* __restrict__ action, R* __restrict__ jac, R* __restrict__ reward_grad,
                     const R* __restrict__ g_state_out, const R* __restrict__ g_obs, const R* __restrict__ g_reward,
                     R* __restrict__ g_state_in, R* __restrict__ g_action, int64_t n, bool vec2, const I2PConsts<R> k) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * kBlock;
  for (int64_t i = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x; i < n; i += stride) {
    R y[6], T[6][7], wr[6], F, dF;
    i2p_load_row<R>(state_in, i, vec2, y);
    i2p_force_and_slope<R>(action, i, k, F, dF);
    i2p_tangent<R>(y, T, F, dF, k);
    i2p_reward_slope<R>(y, k, wr);
    if constexpr (!VJP) {
      R* J = jac + 42 * i;
#pragma unroll
      for (int r = 0; r < 6; ++r)
#pragma unroll
        for (int c = 0; c < 7; ++c) J[7 * r + c] = T[r][c];
      if (reward_grad != nullptr) {
#pragma unroll
        for (int c = 0; c < 7; ++c) {
          R acc = R(0);
#pragma unroll
          for (int r = 0; r < 6; ++r) acc += wr[r] * T[r][c];
          reward_grad[7 * i + c] = acc;
        }
      }
    } else {
      R w[6], gs[6], go[6];
      if (g_state_out != nullptr) i2p_load_row<R>(g_state_out, i, vec2, gs);
      if (g_obs != nullptr) i2p_load_row<R>(g_obs, i, vec2, go);
      const R gr = g_reward != nullptr ? g_reward[i] : R(0);
#pragma unroll
      for (int r = 0; r < 6; ++r) {
        const R slope = (r == 1 || r == 2) ? k.pi : R(1);
        w[r] = (g_state_out != nullptr ? gs[r] : R(0)) + (g_obs != nullptr ? slope * go[r] : R(0)) + gr * wr[r];
      }
      R g[6], ga = R(0);
#pragma unroll
      for (int c = 0; c < 6; ++c) {
        R acc = R(0);
#pragma unroll
        for (int r = 0; r < 6; ++r) acc += w[r] * T[r][c];
        g[c] = acc;
      }
#pragma unroll
      for (int r = 0; r < 6; ++r) ga += w[r] * T[r][6];
      i2p_store_row<R>(g_state_in, i, vec2, g);
      if (g_action != nullptr) g_action[i] = ga;
    }
  }
}

template <typename R>
int i2p_step_derivs(const R* state_in, const void* action, R* jac, R* reward_grad, const R* g_state_out, const R* g_obs,
                    const R* g_reward, R* g_state_in, R* g_action, int64_t n, const emei_i2p_params* p, emei_stream_t stream, bool vjp) {
  if (n < 0) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(p);
  if (const int e = check_i2p_params(*p)) return e;
  if (vjp && g_action != nullptr && p->action_kind < EMEI_ACTION_CONTINUOUS_F32) return EMEI_ERR_BAD_ACTION_KIND;
  if (n == 0) return EMEI_OK;
  EMEI_CHECK_PTR(state_in);
  EMEI_CHECK_PTR(action);
  if (vjp) {
    EMEI_CHECK_PTR(g_state_in);
  } else {
    EMEI_CHECK_PTR(jac);
  }
  const uintptr_t amask = 2 * sizeof(R) - 1;  // every row array aligned for 2-element vectors: vector row access
  const bool vec2 = ((reinterpret_cast<uintptr_t>(state_in) | reinterpret_cast<uintptr_t>(g_state_out) |
                      reinterpret_cast<uintptr_t>(g_obs) | reinterpret_cast<uintptr_t>(g_state_in)) & amask) == 0;
  const I2PConsts<R> k = make_i2p_consts<R>(*p);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (vjp)
    i2p_deriv_kernel<R, true><<<resident_grid(i2p_deriv_kernel<R, true>, n), kBlock, 0, s>>>(
        state_in, action, jac, reward_grad, g_state_out, g_obs, g_reward, g_state_in, g_action, n, vec2, k);
  else
    i2p_deriv_kernel<R, false><<<resident_grid(i2p_deriv_kernel<R, false>, n), kBlock, 0, s>>>(
        state_in, action, jac, reward_grad, g_state_out, g_obs, g_reward, g_state_in, g_action, n, vec2, k);
  return launch_status();
}

}  // namespace emei
