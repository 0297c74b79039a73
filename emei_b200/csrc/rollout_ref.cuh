// Fused T-step rollouts in the arithmetic of the step ENTRY POINTS of this translation unit (included by impl.inc, so
// it exists in both precisions): the families and modes the packed float32 rollout kernels (rollout_f32.cuh) do not
// cover --
//   * float64 reference-exact mode of the cart-pole family, the analytic inverted pendulum and the charged ball
//     (emei_f64.cu, -fmad=false: the reference's own operation order);
//   * the analytic inverted double pendulum, both precisions (6-d state and observation);
//   * obs_noise_params: Gaussian state noise after every sub-step (mujoco_env.py:98-104), inverted pendulum and
//     inverted double pendulum, both precisions -- the Philox keying of emei_ip_step_noisy_* / emei_i2p_step_noisy_*
//     with the global step counter continued inside the kernel.
// Same contract as emei_cartpole_rollout_f32 (zoo/util.py:33-93 batched: policy, step, TimeLimit, auto-reset, optional
// records in the dataset layout, six statistics).  One env per thread; per step the arithmetic is the SAME device
// function the step kernel calls (cartpole_env_step / i2p_env_step / charged_ball_env_step), so a rollout equals
// `horizon` step calls bit for bit.  In-kernel resets use the arithmetic of the emei_init_* kernels in this precision,
// keyed by (seed_reset + episode_index * 0xD1B54A32D192ED03, global env id): host mirror = oracle/philox.py init_*.
#pragma once
#include "rollout.cuh"

namespace emei {

// action value of env i at step t: teacher-forced array [T, n] in `kind`, or the counter-based random policy of
// rollout_f32.cuh (Discrete(2): one bit per step; Box: 24 bits -> [low, high), a float32 like action_space.sample())
struct RefAction {
  float value;      // random policy / continuous: the float32 action; discrete: 0 or 1
  long long index;  // teacher-forced: element index into the action array (-1: use value)
};

__device__ __forceinline__ void ref_store_action(void* rec, size_t at, int kind, const void* src, long long idx, float v) {
  switch (kind) {
    case EMEI_ACTION_DISCRETE_U8:
      static_cast<uint8_t*>(rec)[at] = idx >= 0 ? static_cast<const uint8_t*>(src)[idx] : static_cast<uint8_t>(v);
      break;
    case EMEI_ACTION_DISCRETE_I32:
      static_cast<int32_t*>(rec)[at] = idx >= 0 ? static_cast<const int32_t*>(src)[idx] : static_cast<int32_t>(v);
      break;
    case EMEI_ACTION_DISCRETE_I64:
      static_cast<long long*>(rec)[at] = idx >= 0 ? static_cast<const long long*>(src)[idx] : static_cast<long long>(v);
      break;
    case EMEI_ACTION_CONTINUOUS_F32:
      static_cast<float*>(rec)[at] = idx >= 0 ? static_cast<const float*>(src)[idx] : v;
      break;
    default:
      static_cast<double*>(rec)[at] = idx >= 0 ? static_cast<const double*>(src)[idx] : static_cast<double>(v);
      break;
  }
}

// ------------------------------------------------------------------------------------------------
// env families: Regs (one env in registers), load / store, observation, step, reset
// ------------------------------------------------------------------------------------------------
template <typename R, bool IP>
struct RefCartPole {
  using Real = R;
  using Consts = CartPoleConsts<double>;  // both precisions: cartpole_env_step takes the float64 constants
  static constexpr int kObs = 4;
  struct Buffers {
    R* state;
  };
  struct Regs {
    Vec4<R> y;
  };
  __device__ __forceinline__ static void load(Regs& e, const Buffers& b, int64_t i) { e.y = Vec4<R>::load(b.state + 4 * i); }
  __device__ __forceinline__ static void store(const Regs& e, const Buffers& b, int64_t i) { e.y.store(b.state + 4 * i); }
  __device__ __forceinline__ static void observation(const Regs& e, const Consts& k, R (&o)[kObs]) {
    o[0] = e.y.x, o[1] = e.y.y, o[2] = e.y.z, o[3] = e.y.w;
    if constexpr (IP) o[1] = static_cast<R>(py_mod(static_cast<double>(e.y.y) + k.pi, k.two_pi) - k.pi);  // inverted_pendulum.py:45-49
  }
  __device__ __forceinline__ static R drive(const Consts& k, const void* actions, const RefAction& a, int kind) {
    if (a.index >= 0) return IP ? load_ctrl<R>(actions, a.index, kind) : load_force<R>(actions, a.index, kind, static_cast<R>(k.force_mag));
    if constexpr (IP) return static_cast<R>(a.value);
    if (kind <= EMEI_ACTION_DISCRETE_I64) return static_cast<R>(a.value == 1.0f ? k.force_mag : -k.force_mag);
    return static_cast<R>(__fmul_rn(static_cast<float>(k.force_mag), a.value));  // load_force's float32 product
  }
  __device__ __forceinline__ static void step(Regs& e, R drv, const Consts& k, const NoiseConsts& z, unsigned long long env,
                                              unsigned long long substep0, R& rew, bool& terminated, R (&o)[kObs]) {
    Vec4<R> obs;
    bool notdone;
    cartpole_env_step<R, IP>(e.y, drv, k, z, env, substep0, rew, notdone, obs);
    terminated = !notdone;
    o[0] = obs.x, o[1] = obs.y, o[2] = obs.z, o[3] = obs.w;
  }
  __device__ static void reset(Regs& e, const RolloutConsts<6>& r, const Consts&, unsigned long long env, unsigned long long seed) {
    R v[4];
    if constexpr (!IP) {  // init_uniform_kernel
#pragma unroll
      for (int c = 0; c < 4; ++c) v[c] = static_cast<R>(uniform_initial_sample(seed, env, c, r.init_low, r.init_high, r.init_pi_column));
    } else {  // init_gaussian_kernel
#pragma unroll
      for (int pr = 0; pr < 2; ++pr) gaussian_initial_pair<R>(r.mean, r.sigma, seed, env, pr, v[2 * pr], v[2 * pr + 1]);
    }
    e.y = {v[0], v[1], v[2], v[3]};
  }
};

template <typename R>
struct RefI2P {
  using Real = R;
  using Consts = I2PConsts<R>;
  static constexpr int kObs = 6;
  struct Buffers {
    R* state;
  };
  struct Regs {
    R y[6];
  };
  __device__ __forceinline__ static void load(Regs& e, const Buffers& b, int64_t i) { i2p_load_row<R>(b.state, i, true, e.y); }
  __device__ __forceinline__ static void store(const Regs& e, const Buffers& b, int64_t i) { i2p_store_row<R>(b.state, i, true, e.y); }
  __device__ __forceinline__ static void observation(const Regs& e, const Consts& k, R (&o)[kObs]) {
    o[0] = e.y[0];
    o[1] = py_mod2(e.y[1] + k.pi) * k.pi - k.pi;  // inverted_double_pendulum.py:56-60 (sic)
    o[2] = py_mod2(e.y[2] + k.pi) * k.pi - k.pi;
    o[3] = e.y[3], o[4] = e.y[4], o[5] = e.y[5];
  }
  __device__ __forceinline__ static R drive(const Consts&, const void* actions, const RefAction& a, int kind) {
    return a.index >= 0 ? load_ctrl<R>(actions, a.index, kind) : static_cast<R>(a.value);
  }
  __device__ __forceinline__ static void step(Regs& e, R drv, const Consts& k, const NoiseConsts& z, unsigned long long env,
                                              unsigned long long substep0, R& rew, bool& terminated, R (&o)[kObs]) {
    bool notdone;
    i2p_env_step<R>(e.y, drv, k, z, env, substep0, o, rew, notdone);
    terminated = !notdone;
  }
  __device__ static void reset(Regs& e, const RolloutConsts<6>& r, const Consts&, unsigned long long env, unsigned long long seed) {
#pragma unroll
    for (int pr = 0; pr < 3; ++pr) gaussian_initial_pair<R>(r.mean, r.sigma, seed, env, pr, e.y[2 * pr], e.y[2 * pr + 1]);
  }
};

template <typename R>
struct RefChargedBall {
  using Real = R;
  using Consts = ChargedBallConsts<R>;
  static constexpr int kObs = 4;
  struct Buffers {
    uint8_t* on_circle;
    R* circle;
    R* free_state;
  };
  struct Regs {
    bool on;
    R theta, omega;
    Vec4<R> f;
  };
  __device__ __forceinline__ static void load(Regs& e, const Buffers& b, int64_t i) {
    e.on = b.on_circle[i] != 0;
    e.theta = b.circle[2 * i];
    e.omega = b.circle[2 * i + 1];
    e.f = Vec4<R>::load(b.free_state + 4 * i);
  }
  __device__ __forceinline__ static void store(const Regs& e, const Buffers& b, int64_t i) {
    b.on_circle[i] = e.on ? 1 : 0;
    b.circle[2 * i] = e.theta;
    b.circle[2 * i + 1] = e.omega;
    e.f.store(b.free_state + 4 * i);
  }
  __device__ __forceinline__ static void observation(const Regs& e, const Consts&, R (&o)[kObs]) {
    o[0] = e.f.x, o[1] = e.f.y, o[2] = e.f.z, o[3] = e.f.w;  // charged_ball.py:96-97
  }
  __device__ __forceinline__ static R drive(const Consts& k, const void* actions, const RefAction& a, int kind) {
    if (a.index >= 0) return load_force<R>(actions, a.index, kind, k.charge);
    if (kind <= EMEI_ACTION_DISCRETE_I64) return a.value == 1.0f ? k.charge : -k.charge;
    return static_cast<R>(__fmul_rn(static_cast<float>(k.charge), a.value));
  }
  __device__ __forceinline__ static void step(Regs& e, R drv, const Consts& k, const NoiseConsts&, unsigned long long, unsigned long long,
                                              R& rew, bool& terminated, R (&o)[kObs]) {
    // the continuous variant evaluates the field terms in float32 (NEP 50: see charged_ball_step_kernel); double only
    if (sizeof(R) == 8 && k.action_kind >= EMEI_ACTION_CONTINUOUS_F32)
      rew = charged_ball_env_step<R, (sizeof(R) == 8)>(e.on, e.theta, e.omega, e.f, drv, k);
    else
      rew = charged_ball_env_step<R, false>(e.on, e.theta, e.omega, e.f, drv, k);
    terminated = false;  // charged_ball.py:110-111
    o[0] = e.f.x, o[1] = e.f.y, o[2] = e.f.z, o[3] = e.f.w;
  }
  __device__ static void reset(Regs& e, const RolloutConsts<6>&, const Consts& k, unsigned long long env, unsigned long long seed) {
    R f[4];
    charged_ball_initial_sample<R>(seed, env, k.r, e.theta, e.omega, f);  // init_charged_ball_kernel
    e.on = true;
    e.f = {f[0], f[1], f[2], f[3]};
  }
};

// ------------------------------------------------------------------------------------------------
// the kernel
// ------------------------------------------------------------------------------------------------
template <class Fam>
__global__ void __launch_bounds__(kBlock)
    rollout_ref_kernel(const typename Fam::Buffers b, const RolloutIO<typename Fam::Real> io, int64_t n, const typename Fam::Consts k,
                       const RolloutConsts<6> r, const NoiseConsts z, int freq_rate) {
  using R = typename Fam::Real;
  constexpr int D = Fam::kObs;
  const int64_t i = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x;
  double r_sum = 0.0, fin_ret = 0.0;
  unsigned n_term = 0, n_trunc = 0, n_fin = 0, fin_len = 0;
  if (i < n) {
    typename Fam::Regs e;
    Fam::load(e, b, i);
    int ep_step = io.ep_step[i], ep_idx = io.ep_index[i];
    R ep_ret = io.ep_return[i];
    const unsigned long long env = r.env_offset + static_cast<unsigned long long>(i);
    const bool discrete = k.action_kind <= EMEI_ACTION_DISCRETE_I64;
    uint32_t w[4] = {0u, 0u, 0u, 0u};
    for (int t = 0; t < r.horizon; ++t) {
      // ---- policy
      RefAction a;
      a.value = 0.f;
      a.index = -1;
      const unsigned long long tg = r.t0 + static_cast<unsigned long long>(t);
      if (r.random_policy) {  // the stream of rollout_f32_kernel; a copy of its own (DESIGN.md 4.6)
        if (discrete) {
          if (t == 0 || (tg & 127ull) == 0) Philox::generate(r.seed_action, env, static_cast<uint32_t>(tg >> 7), kPurposeRolloutAction, w);
          const unsigned j = static_cast<unsigned>(tg >> 5) & 3u;
          const uint32_t word = j == 0 ? w[0] : (j == 1 ? w[1] : (j == 2 ? w[2] : w[3]));
          a.value = static_cast<float>((word >> (static_cast<unsigned>(tg) & 31u)) & 1u);
        } else {
          if (t == 0 || (tg & 3ull) == 0) Philox::generate(r.seed_action, env, static_cast<uint32_t>(tg >> 2), kPurposeRolloutAction, w);
          const unsigned j = static_cast<unsigned>(tg) & 3u;
          const uint32_t word = j == 0 ? w[0] : (j == 1 ? w[1] : (j == 2 ? w[2] : w[3]));
          a.value = fmaf(r.act_high - r.act_low, static_cast<float>(word >> 8) * (1.0f / 16777216.0f), r.act_low);
        }
      } else {
        a.index = static_cast<long long>(t) * n + i;
      }
      const size_t rec = static_cast<size_t>(t) * n + i;
      if (io.rec_obs != nullptr) {
        R o[D];
        Fam::observation(e, k, o);
#pragma unroll
        for (int c = 0; c < D; ++c) io.rec_obs[rec * D + c] = o[c];
        ref_store_action(io.rec_act, rec, k.action_kind, io.actions, a.index, a.value);
      }
      // ---- dynamics + reward + terminal: the step entry point's device function
      R rew, o[D];
      bool terminated;
      // noise: z.substep0 holds the env-step counter of this call's first step (emei_noise_params.step)
      Fam::step(e, Fam::drive(k, io.actions, a, k.action_kind), k, z, env,
                (z.substep0 + static_cast<unsigned long long>(t)) * static_cast<unsigned long long>(freq_rate), rew, terminated, o);
      // ---- TimeLimit + bookkeeping (zoo/util.py:58-73; gym TimeLimit: truncated = elapsed >= max)
      ep_step += 1;
      ep_ret += rew;
      const bool truncated = r.max_episode_steps > 0 && ep_step >= r.max_episode_steps;
      const bool done = terminated || truncated;
      if (io.rec_obs != nullptr) {
#pragma unroll
        for (int c = 0; c < D; ++c) io.rec_next[rec * D + c] = o[c];
        io.rec_rew[rec] = rew;
        io.rec_done[rec] = done ? 1 : 0;
        io.rec_timeout[rec] = truncated ? 1 : 0;
      }
      r_sum += static_cast<double>(rew);
      n_term += terminated ? 1u : 0u;
      n_trunc += truncated ? 1u : 0u;
      if (done && r.auto_reset) {
        n_fin += 1u;
        fin_ret += static_cast<double>(ep_ret);
        fin_len += static_cast<unsigned>(ep_step);
        ep_idx += 1;
        Fam::reset(e, r, k, env, reset_seed(r.seed_reset, ep_idx));
        ep_step = 0;
        ep_ret = R(0);
      }
    }
    Fam::store(e, b, i);
    io.ep_step[i] = ep_step;
    io.ep_return[i] = ep_ret;
    io.ep_index[i] = ep_idx;
  }
  if (io.stats != nullptr) {  // uniform across the grid
    __shared__ double s_red[kBlock / 32];
    const double vals[6] = {r_sum, static_cast<double>(n_term), static_cast<double>(n_trunc),
                            static_cast<double>(n_fin), fin_ret, static_cast<double>(fin_len)};
#pragma unroll
    for (int j = 0; j < 6; ++j) {
      const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
      double v = warp_sum(vals[j]);
      __syncthreads();
      if (lane == 0) s_red[warp] = v;
      __syncthreads();
      v = warp_sum(lane < kBlock / 32 ? s_red[lane] : 0.0);
      if (threadIdx.x == 0) atomicAdd(&io.stats[j], v);
    }
  }
}

template <class Fam>
inline void launch_ref_rollout(const typename Fam::Buffers& b, const RolloutIO<typename Fam::Real>& io, int64_t n, const typename Fam::Consts& k,
                               const RolloutConsts<6>& rc, const NoiseConsts& z, int freq_rate, cudaStream_t s) {
  rollout_ref_kernel<Fam><<<grid_for(n, kBlock), kBlock, 0, s>>>(b, io, n, k, rc, z, freq_rate);
}

template <typename R>
int cartpole_rollout_ref(R* state_io, int32_t* ep_step, R* ep_return, int32_t* ep_index, const void* actions, R* rec_obs, R* rec_next,
                         void* rec_act, R* rec_rew, uint8_t* rec_done, uint8_t* rec_timeout, double* stats, int64_t n,
                         const emei_cartpole_params* p, const emei_rollout_params* r, const emei_noise_params* noise, emei_stream_t stream) {
  if (n < 0) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(p);
  EMEI_CHECK_PTR(r);
  if (const int e = check_cartpole_params(*p)) return e;
  const bool ip = p->variant > EMEI_CARTPOLE_SWINGUP;
  if (noise != nullptr && !ip) return EMEI_ERR_BAD_VARIANT;  // the noisy step exists for the MuJoCo-shell family only (mujoco_env.py:98-104)
  if (const int e = check_noise_params(noise, 4)) return e;
  const RolloutIO<R> io = {ep_step, ep_return, ep_index, actions, rec_obs, rec_next, rec_act, rec_rew, rec_done, rec_timeout, stats};
  RolloutConsts<6> rc;
  if (const int e = make_rollout(r, io, false, nullptr, nullptr, rc)) return e;
  if (n == 0 || r->horizon == 0) return EMEI_OK;
  EMEI_CHECK_PTR(state_io);
  EMEI_CHECK_ALIGN16(state_io);
  const CartPoleConsts<double> k = make_cartpole_consts<double>(*p);
  const NoiseConsts z = make_noise_consts(noise, 1);  // substep0 = the env-step counter; the kernel scales by freq_rate
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (ip) {
    typename RefCartPole<R, true>::Buffers b = {state_io};
    launch_ref_rollout<RefCartPole<R, true>>(b, io, n, k, rc, z, p->freq_rate, s);
  } else {
    typename RefCartPole<R, false>::Buffers b = {state_io};
    launch_ref_rollout<RefCartPole<R, false>>(b, io, n, k, rc, z, p->freq_rate, s);
  }
  return launch_status();
}

template <typename R>
int i2p_rollout(R* state_io, int32_t* ep_step, R* ep_return, int32_t* ep_index, const void* actions, R* rec_obs, R* rec_next, void* rec_act,
                R* rec_rew, uint8_t* rec_done, uint8_t* rec_timeout, double* stats, int64_t n, const emei_i2p_params* p,
                const emei_rollout_params* r, const double* init_mean, const double* init_sigma, const emei_noise_params* noise,
                emei_stream_t stream) {
  if (n < 0) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(p);
  EMEI_CHECK_PTR(r);
  EMEI_CHECK_PTR(init_mean);
  EMEI_CHECK_PTR(init_sigma);
  if (const int e = check_i2p_params(*p)) return e;
  if (const int e = check_noise_params(noise, 6)) return e;
  const RolloutIO<R> io = {ep_step, ep_return, ep_index, actions, rec_obs, rec_next, rec_act, rec_rew, rec_done, rec_timeout, stats};
  RolloutConsts<6> rc;
  if (const int e = make_rollout(r, io, false, init_mean, init_sigma, rc)) return e;
  if (n == 0 || r->horizon == 0) return EMEI_OK;
  EMEI_CHECK_PTR(state_io);
  EMEI_CHECK_ALIGN16(state_io);
  typename RefI2P<R>::Buffers b = {state_io};
  launch_ref_rollout<RefI2P<R>>(b, io, n, make_i2p_consts<R>(*p), rc, make_noise_consts(noise, 1), p->freq_rate, static_cast<cudaStream_t>(stream));
  return launch_status();
}

template <typename R>
int charged_ball_rollout_ref(uint8_t* on_circle_io, R* circle_io, R* free_state_io, int32_t* ep_step, R* ep_return, int32_t* ep_index,
                             const void* actions, R* rec_obs, R* rec_next, void* rec_act, R* rec_rew, uint8_t* rec_done, uint8_t* rec_timeout,
                             double* stats, int64_t n, const emei_charged_ball_params* p, const emei_rollout_params* r, emei_stream_t stream) {
  if (n < 0) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(p);
  EMEI_CHECK_PTR(r);
  if (const int e = check_charged_ball_params(*p)) return e;
  const RolloutIO<R> io = {ep_step, ep_return, ep_index, actions, rec_obs, rec_next, rec_act, rec_rew, rec_done, rec_timeout, stats};
  RolloutConsts<6> rc;
  if (const int e = make_rollout(r, io, false, nullptr, nullptr, rc)) return e;
  if (n == 0 || r->horizon == 0) return EMEI_OK;
  EMEI_CHECK_PTR(on_circle_io);
  EMEI_CHECK_PTR(circle_io);
  EMEI_CHECK_PTR(free_state_io);
  EMEI_CHECK_ALIGN16(circle_io);
  EMEI_CHECK_ALIGN16(free_state_io);
  typename RefChargedBall<R>::Buffers b = {on_circle_io, circle_io, free_state_io};
  launch_ref_rollout<RefChargedBall<R>>(b, io, n, make_cb_consts<R>(*p), rc, NoiseConsts{}, p->freq_rate, static_cast<cudaStream_t>(stream));
  return launch_status();
}

}  // namespace emei
