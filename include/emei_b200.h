/*
 * emei_b200 -- C ABI of the B200-native batched environment engine for polixir/emei's hot path.
 *
 * The reference (pure Python/numpy) has no FFI; its boundary for this path is the EmeiEnv class
 * contract (emei/core.py:131-193).  This header is what a ctypes binding inside that contract
 * calls (INTEGRATION.md shows the stub).  Each entry point cites the reference code it replaces
 * (paths relative to the reference tree).
 *
 * Conventions (all functions):
 *   - plain pointers + element counts + POD parameter structs; NO torch / C++ types;
 *   - every data pointer is a DEVICE pointer owned by the caller; nothing is allocated;
 *   - asynchronous on `stream` (a cudaStream_t passed as void*; NULL = legacy default stream);
 *   - no global state: re-entrant and thread-safe;
 *   - returns 0 on success, a positive cudaError_t if the launch failed, or a negative
 *     EMEI_ERR_* code if an argument is invalid (see emei_error_string); never aborts/throws;
 *   - n == 0 is a valid no-op.
 *   - `stats` (nullable) is double[2] on the device: {sum of rewards, number of done flags};
 *     kernels ACCUMULATE into it (warp-shuffle + one atomic per block); zero it with
 *     emei_stats_reset before a rollout.
 *   - layouts are row-major [n, dim]; rows of float4/double2 alignment: state/obs base pointers
 *     must be 16-byte aligned.
 */
#ifndef EMEI_B200_H
#define EMEI_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define EMEI_B200_VERSION 100 /* 0.1.0 */

typedef void* emei_stream_t; /* cudaStream_t */

/* ---- error codes (negative = argument errors; positive = cudaError_t) ---------------------- */
#define EMEI_OK 0
#define EMEI_ERR_NULL_POINTER (-1)
#define EMEI_ERR_BAD_VARIANT (-2)
#define EMEI_ERR_BAD_ACTION_KIND (-3)
#define EMEI_ERR_BAD_SIZE (-4)
#define EMEI_ERR_MISALIGNED (-5)
#define EMEI_ERR_BAD_PARAM (-6)

/* ---- action encodings ----------------------------------------------------------------------
 * discrete: force = +mag if action == 1 else -mag  (cartpole.py:121-122,142-143;
 *           charged_ball.py:155-156).  continuous: force = mag * action[0]
 *           (charged_ball.py:169-170), one value per env. */
#define EMEI_ACTION_DISCRETE_U8 0
#define EMEI_ACTION_DISCRETE_I32 1
#define EMEI_ACTION_DISCRETE_I64 2
#define EMEI_ACTION_CONTINUOUS_F32 3
#define EMEI_ACTION_CONTINUOUS_F64 4

/* ---- env families / variants (also the `family` of emei_reward_terminal_*) ------------------ */
#define EMEI_CARTPOLE_BALANCING 0    /* cartpole.py:115-132  obs [x, x', th, th']            */
#define EMEI_CARTPOLE_SWINGUP 1      /* cartpole.py:135-156                                  */
#define EMEI_IP_REBOUND_BALANCING 2  /* inverted_pendulum.py:52-79   obs [x, th, v, w]       */
#define EMEI_IP_BOUNDARY_BALANCING 3 /* inverted_pendulum.py:82-111                          */
#define EMEI_IP_REBOUND_SWINGUP 4    /* inverted_pendulum.py:114-146                         */
#define EMEI_IP_BOUNDARY_SWINGUP 5   /* inverted_pendulum.py:149-183                         */
#define EMEI_I2P_REBOUND_BALANCING 6 /* inverted_double_pendulum.py:63-90   obs dim 6        */
#define EMEI_I2P_BOUNDARY_BALANCING 7 /* :93-122                                             */
#define EMEI_I2P_REBOUND_SWINGUP 8   /* :125-157                                             */
#define EMEI_I2P_BOUNDARY_SWINGUP 9  /* :160-196                                             */
#define EMEI_HOPPER 10               /* hopper.py:79-106       obs dim 12, action dim 3      */
#define EMEI_HALFCHEETAH 11          /* half_cheetah.py:59-67  obs dim 18, action dim 6      */
#define EMEI_CHARGED_BALL 12         /* charged_ball.py:110-111,158-160  obs dim 4           */
#define EMEI_NUM_FAMILIES 13

/* ---- cart-pole / analytic inverted-pendulum dynamics ---------------------------------------- */
typedef struct emei_cartpole_params {
  /* BaseCartPoleEnv constants (cartpole.py:22-31) or the inverted_pendulum.xml equivalents;
     computed on the host in double exactly as the reference computes them. */
  double gravity;
  double mass_pole;
  double total_mass;       /* mass_pole + mass_cart (cartpole.py:25) */
  double length;           /* half the pole length */
  double pole_mass_length; /* mass_pole * length (cartpole.py:51) */
  double force_mag;        /* cart-pole: force_mag (10.0); IP: motor gear (100.0) */
  double x_threshold;      /* cart-pole |x| bound (2.4 / 5) */
  double theta_threshold;  /* CartPoleBalancing |theta| bound (12 deg) */
  double x_left, x_right;  /* IP rail = model.jnt_range[0] (inverted_pendulum.xml:14) */
  double ctrl_low, ctrl_high; /* IP ctrlrange (inverted_pendulum.xml:23); ctrl is clamped like mj_step does */
  double dt;               /* seconds per sub-step = real_time_scale (base_control.py:73, mujoco_env.py:69) */
  int32_t freq_rate;       /* forward-Euler sub-steps per env step (base_control.py:160-164) */
  int32_t variant;         /* EMEI_CARTPOLE_* or EMEI_IP_* */
  int32_t action_kind;     /* EMEI_ACTION_* */
  int32_t reserved;
} emei_cartpole_params;

/* One env step for n environments.
 * Replaces BaseControlEnv.step (base_control.py:61-83) = _extract_action + ODE_approximation
 * (base_control.py:133-164, forward Euler, freq_rate sub-steps of dt) + BaseCartPoleEnv._dsdt
 * (cartpole.py:48-60) + get_batch_reward/terminal (cartpole.py:124-129,145-151); for the EMEI_IP_*
 * variants: EmeiMujocoEnv.step's shell (mujoco_env.py:157-167, forward-Euler rule :91-97, angle-wrapped
 * observation inverted_pendulum.py:45-49, reward/terminal :73-79,103-111,139-146,174-183) around
 * the analytic acceleration.
 *   state_in  [n,4]  read;  state_out [n,4] written (may alias state_in);
 *   obs_out   [n,4]  nullable; IP variants: state_out with theta wrapped to [-pi,pi); cart-pole: copy;
 *   action    [n]    encoding = p->action_kind;   reward [n] ; done [n] (0/1) ; stats nullable.
 * _f32 : all-float32 arithmetic (tolerance 1e-5 rel + 1e-6 abs per step vs the reference).
 * _f64 : cart-pole = the reference's exact mixed arithmetic (float64 derivative, float32 increment,
 *        float64 accumulate, SURVEY.md 0.3); IP = float64 throughout.  No FMA contraction. */
int emei_cartpole_step_f32(const float* state_in, float* state_out, float* obs_out, const void* action, float* reward,
                           uint8_t* done, double* stats, int64_t n, const emei_cartpole_params* p, emei_stream_t stream);
int emei_cartpole_step_f64(const double* state_in, double* state_out, double* obs_out, const void* action,
                           double* reward, uint8_t* done, double* stats, int64_t n, const emei_cartpole_params* p,
                           emei_stream_t stream);

/* ---- fused T-step rollout (float32) -------------------------------------------------------------
 * Replaces the collection loop that calls step(): zoo/util.py:33-93 (reset; while not done: action =
 * policy | env.action_space.sample(); step; record), batched, with gym's TimeLimit
 * (register_env.py max_episode_steps) and the per-episode reset done in-kernel.  The state stays in
 * registers for all `horizon` steps; per step the arithmetic is exactly emei_cartpole_step_f32's. */
typedef struct emei_rollout_params {
  int32_t horizon;           /* T: steps per env in this call */
  int32_t max_episode_steps; /* TimeLimit: truncated when the episode step count reaches it; <= 0: no limit */
  int32_t auto_reset;        /* 1: an env whose step was done (terminated | truncated) is re-initialised */
  int32_t random_policy;     /* 1: uniform random actions (action_space.sample()); 0: actions[T,n] supplied */
  int32_t init_kind;         /* reset sampler: 0 = uniform (cartpole.py:131-132,153-156), 1 = gaussian (mujoco_env.py:137-140) */
  int32_t init_pi_column;    /* uniform: column that gets +pi (-1 none) */
  uint64_t seed_reset;       /* Philox key base of the reset sampler: episode k of an env uses seed_reset + k*0xD1B54A32D192ED03 */
  uint64_t seed_action;      /* Philox key of the random policy stream of each env: 1 bit (Discrete) / one 32-bit word (Box) per step t0 + t */
  uint64_t env_offset;       /* global id of env 0 (sharding) */
  uint64_t t0;               /* global step index of the first step of this call (continues the action stream) */
  double init_low, init_high;              /* uniform range */
  double init_mean[4], init_sigma[4];      /* gaussian parameters */
  double action_low, action_high;          /* continuous random policy range */
} emei_rollout_params;

/*   state_io [n,4] ; episode_step_io int32[n] ; episode_return_io float[n] ; episode_index_io int32[n]  (read+written)
 *   actions  [horizon,n] in p->action_kind, or NULL when random_policy
 *   rec_*    optional transition records (all NULL or all set), the reference's dataset keys (zoo/util.py:62-67):
 *            observations [T,n,4], next_observations [T,n,4], actions [T,n] (p->action_kind element type),
 *            rewards [T,n], dones [T,n] u8 (terminated | truncated), timeouts [T,n] u8 (truncated)
 *   stats    nullable double[6], accumulated: {sum of rewards, #terminated, #truncated, #episodes finished,
 *            sum of finished-episode returns, sum of finished-episode lengths} (-> avg_reward / avg_length
 *            of zoo/util.py:87-91).  n <= 2^31 - 2^20. */
int emei_cartpole_rollout_f32(float* state_io, int32_t* episode_step_io, float* episode_return_io,
                              int32_t* episode_index_io, const void* actions, float* rec_observations,
                              float* rec_next_observations, void* rec_actions, float* rec_rewards, uint8_t* rec_dones,
                              uint8_t* rec_timeouts, double* stats, int64_t n, const emei_cartpole_params* p,
                              const emei_rollout_params* r, emei_stream_t stream);

/* ---- analytic inverted double pendulum (SURVEY 8f rank 3) ----------------------------------------
 * The reference's I2P accelerations are MuJoCo's (third-party mj_step); this is the reference's own Lagrangian
 * model, classic_control/auxiliary/lagrange_eqs.py:12-60 cartpole(2) (cart + two thin rods, relative hinge angles,
 * inertia 1/3 m l^2), with the complete potential energy (the script omits the height of pole 1's hinge for
 * n >= 2, lagrange_eqs.py:45), the constants of assets/inverted_double_pendulum.xml:25,31,32,35,38,45 and the
 * forward-Euler rule of mujoco_env.py:91-97. */
typedef struct emei_i2p_params {
  double gravity, mass_cart, mass_pole0, mass_pole1, length0, length1; /* lengths = half a pole (hinge -> COM) */
  double gear, ctrl_low, ctrl_high;                                    /* force = gear * clamp(ctrl) (xml:45) */
  double x_left, x_right;                                              /* slider range (xml:31) */
  double dt;                                                           /* real_time_scale */
  int32_t freq_rate;
  int32_t variant;     /* EMEI_I2P_* : SwingUp variants flip pole 0 (inverted_double_pendulum.py:146-148,181-183) */
  int32_t action_kind; /* EMEI_ACTION_* */
} emei_i2p_params;

/*   state_in/out [n,6] = [x, th0, th1, v, w0, w1] (qpos||qvel, angles unwrapped) ; obs_out [n,6] REQUIRED
 *   (current_obs, inverted_double_pendulum.py:56-60, precedence quirk `(th + pi) % 2 * pi - pi` replicated) ;
 *   action [n] ; reward [n], done [n] = get_batch_reward / get_batch_terminal of the variant on obs_out
 *   (:84-90,114-122,150-157,185-196), fused into the step kernel ; stats nullable double[2]. */
int emei_i2p_step_f32(const float* state_in, float* state_out, float* obs_out, const void* action, float* reward,
                      uint8_t* done, double* stats, int64_t n, const emei_i2p_params* p, emei_stream_t stream);
int emei_i2p_step_f64(const double* state_in, double* state_out, double* obs_out, const void* action, double* reward,
                      uint8_t* done, double* stats, int64_t n, const emei_i2p_params* p, emei_stream_t stream);

/* ---- derivatives of the analytic steps (Jacobians and vector-Jacobian products) --------------------
 * What is differentiated: the real-valued model emei_cartpole_step_* / emei_i2p_step_* evaluate -- freq_rate forward-Euler
 * sub-steps of the analytic acceleration, then the observation, then the variant's reward -- without state noise (the
 * stateless transition of get_batch_next_obs).
 *   _f64: plain float64 arithmetic.  The cart-pole family's forward step rounds each Euler increment through float32 (the
 *         reference's mixed rule); the derivative is that of y + h f(y) in float64, which matches a complex-step derivative
 *         to ~1e-12.  The forward step is unchanged.
 *   _f32: float32 through the generic device arithmetic: gradients are a tolerance product, not a bit product.
 * Action column: cart-pole continuous kinds d/da of force = force_mag * a; IP / I2P force = gear * clamp(ctrl), whose
 * gradient passes where ctrl_low <= ctrl <= ctrl_high (inclusive, as torch.clamp) and is 0 outside; discrete kinds: 0.
 * Observation: the IP angle wrap (th + pi) mod 2pi - pi has slope 1; the I2P current_obs quirk ((th + pi) mod 2) * pi - pi
 * has slope pi on both angles (inverted_double_pendulum.py:56-60, replicated by the forward), and the reward computed on that
 * observation inherits the factor.  `done` is not differentiable.  Non-finite inputs give non-finite gradients.
 * Validation as the step entry points (codes, row alignment); variants outside the family: EMEI_ERR_BAD_VARIANT. */
/* d(state_out, reward) / d(state_in, action) of emei_cartpole_step_* (cart-pole and EMEI_IP_* variants):
 *   jac [n,4,5]: jac[i][r][c] = d state_out[i][r] / d state_in[i][c] (c < 4); c = 4: d state_out[i][r] / d action[i]
 *   reward_grad [n,5] nullable: the same row for reward[i] */
int emei_cartpole_step_jacobian_f32(const float* state_in, const void* action, float* jac, float* reward_grad, int64_t n,
                                    const emei_cartpole_params* p, emei_stream_t stream);
int emei_cartpole_step_jacobian_f64(const double* state_in, const void* action, double* jac, double* reward_grad, int64_t n,
                                    const emei_cartpole_params* p, emei_stream_t stream);
/* vector-Jacobian product (autograd's backward) of the same step:
 *   g_state_in[i] = g_state_out[i] . d state_out / d state_in + g_obs[i] . d obs_out / d state_in + g_reward[i] d reward / d state_in
 *   g_state_out [n,4], g_obs [n,4], g_reward [n]: each nullable (= zero); g_state_in [n,4] written;
 *   g_action [n] written, nullable; must be NULL for discrete action kinds (else EMEI_ERR_BAD_ACTION_KIND).
 * The Jacobian is contracted in registers and never stored. */
int emei_cartpole_step_vjp_f32(const float* state_in, const void* action, const float* g_state_out, const float* g_obs,
                               const float* g_reward, float* g_state_in, float* g_action, int64_t n, const emei_cartpole_params* p,
                               emei_stream_t stream);
int emei_cartpole_step_vjp_f64(const double* state_in, const void* action, const double* g_state_out, const double* g_obs,
                               const double* g_reward, double* g_state_in, double* g_action, int64_t n, const emei_cartpole_params* p,
                               emei_stream_t stream);
/* the same pair for emei_i2p_step_*: rows of 6, jac [n,6,7], reward_grad [n,7], g_state_out / g_obs / g_state_in [n,6] */
int emei_i2p_step_jacobian_f32(const float* state_in, const void* action, float* jac, float* reward_grad, int64_t n,
                               const emei_i2p_params* p, emei_stream_t stream);
int emei_i2p_step_jacobian_f64(const double* state_in, const void* action, double* jac, double* reward_grad, int64_t n,
                               const emei_i2p_params* p, emei_stream_t stream);
int emei_i2p_step_vjp_f32(const float* state_in, const void* action, const float* g_state_out, const float* g_obs,
                          const float* g_reward, float* g_state_in, float* g_action, int64_t n, const emei_i2p_params* p,
                          emei_stream_t stream);
int emei_i2p_step_vjp_f64(const double* state_in, const void* action, const double* g_state_out, const double* g_obs,
                          const double* g_reward, double* g_state_in, double* g_action, int64_t n, const emei_i2p_params* p,
                          emei_stream_t stream);

/* ---- differentiable open-loop trajectories (T steps in one launch, their VJP in one reverse sweep) -------
 * The open-loop composition of `horizon` stateless steps of emei_cartpole_step_* (cart-pole and EMEI_IP_* variants) /
 * emei_i2p_step_* from caller rows: no state noise, no resets, no statistics, and an env whose done flag is set keeps
 * being integrated.  Every array is time-major; D = 4 (cart-pole family) or 6 (I2P):
 *   state0 [n,D] ; actions [horizon,n] (EMEI_ACTION_* encoding) ; states [horizon+1,n,D] ; obs [horizon,n,D] ;
 *   rewards, dones [horizon,n] ; g_state0 [n,D] ; g_states [horizon+1,n,D] ; g_obs [horizon,n,D] ; g_rewards, g_actions [horizon,n].
 * Forward: states[0] = state0; states[t+1], obs[t], rewards[t], dones[t] are bit-equal to the t-th of `horizon` chained
 * step calls (the step's own device functions; float32 cart-pole / IP: the lean arithmetic of the step kernel).  obs and
 * dones are nullable (not written); the cart-pole envs' observation is the next state, so they pass obs NULL.
 * VJP: the reverse sweep of the same composition under the derivative model above (float64 cart-pole: the float64 Euler
 * step; clamp inclusive; I2P observation angles slope pi):
 *   g_state0 = d L / d state0 and g_actions[t] = d L / d actions[t] for L = <g_states, states> + <g_obs, obs> + <g_rewards, rewards>.
 *   g_states, g_obs, g_rewards each nullable (= zero); g_actions nullable, and must be NULL for discrete action kinds (else
 *   EMEI_ERR_BAD_ACTION_KIND).  The cotangent is carried in registers from step to step; only g_actions and g_state0 are written.
 * Validation: n < 0 or horizon < 0 -> EMEI_ERR_BAD_SIZE, then the step / VJP entry points' checks in their order; n == 0 or
 * horizon == 0 returns EMEI_OK with nothing launched or written.  Cart-pole row arrays are 16-byte aligned (EMEI_ERR_MISALIGNED). */
int emei_cartpole_trajectory_f32(const float* state0, const void* actions, float* states, float* obs, float* rewards, uint8_t* dones,
                                 int64_t n, int64_t horizon, const emei_cartpole_params* p, emei_stream_t stream);
int emei_cartpole_trajectory_f64(const double* state0, const void* actions, double* states, double* obs, double* rewards,
                                 uint8_t* dones, int64_t n, int64_t horizon, const emei_cartpole_params* p, emei_stream_t stream);
int emei_cartpole_trajectory_vjp_f32(const float* states, const void* actions, const float* g_states, const float* g_obs,
                                     const float* g_rewards, float* g_state0, float* g_actions, int64_t n, int64_t horizon,
                                     const emei_cartpole_params* p, emei_stream_t stream);
int emei_cartpole_trajectory_vjp_f64(const double* states, const void* actions, const double* g_states, const double* g_obs,
                                     const double* g_rewards, double* g_state0, double* g_actions, int64_t n, int64_t horizon,
                                     const emei_cartpole_params* p, emei_stream_t stream);
/* the same pair for emei_i2p_step_*: rows of 6 */
int emei_i2p_trajectory_f32(const float* state0, const void* actions, float* states, float* obs, float* rewards, uint8_t* dones,
                            int64_t n, int64_t horizon, const emei_i2p_params* p, emei_stream_t stream);
int emei_i2p_trajectory_f64(const double* state0, const void* actions, double* states, double* obs, double* rewards, uint8_t* dones,
                            int64_t n, int64_t horizon, const emei_i2p_params* p, emei_stream_t stream);
int emei_i2p_trajectory_vjp_f32(const float* states, const void* actions, const float* g_states, const float* g_obs,
                                const float* g_rewards, float* g_state0, float* g_actions, int64_t n, int64_t horizon,
                                const emei_i2p_params* p, emei_stream_t stream);
int emei_i2p_trajectory_vjp_f64(const double* states, const void* actions, const double* g_states, const double* g_obs,
                                const double* g_rewards, double* g_state0, double* g_actions, int64_t n, int64_t horizon,
                                const emei_i2p_params* p, emei_stream_t stream);

/* ---- per-sub-step Gaussian state noise ("obs_noise_params", SURVEY 8f rank 4) -------------------
 * Replaces mujoco_env.py:98-104: after EVERY sub-step the reference overwrites the simulator state with
 * additive_gaussian_noise(qpos, qvel, obs_noise_params) (mujoco_env.py:197-249: one N(0, sigma_pos) /
 * N(0, sigma_vel) draw per hinge/slide joint coordinate).  INTENDED semantics, like the init sampler: the
 * reference slices rows instead of columns (:243-244), so with its batch of one it adds joint 0's draw to every
 * coordinate and drops the other joints' (documented in DESIGN.md, not replicated).  The reference's stream is
 * numpy's global Mersenne Twister; here coordinates 2k, 2k+1 of env e at global sub-step g = step * freq_rate + s
 * are the Box-Muller pair of Philox4x32-10 block 4g + k keyed by (seed, env_offset + e): the result depends on
 * neither the batch sharding nor the launch shape. */
typedef struct emei_noise_params {
  double sigma[6];     /* per state coordinate: IP [x, th, v, w] (first 4), I2P [x, th0, th1, v, w0, w1]; >= 0 */
  uint64_t seed;       /* Philox key */
  uint64_t env_offset; /* global id of env 0 (sharding) */
  uint64_t step;       /* env-step counter of this call (the caller increments it every step) */
} emei_noise_params;

/* emei_cartpole_step_* for the EMEI_IP_* variants / emei_i2p_step_* with the noise above; same arguments. */
int emei_ip_step_noisy_f32(const float* state_in, float* state_out, float* obs_out, const void* action, float* reward,
                           uint8_t* done, double* stats, int64_t n, const emei_cartpole_params* p,
                           const emei_noise_params* z, emei_stream_t stream);
int emei_ip_step_noisy_f64(const double* state_in, double* state_out, double* obs_out, const void* action,
                           double* reward, uint8_t* done, double* stats, int64_t n, const emei_cartpole_params* p,
                           const emei_noise_params* z, emei_stream_t stream);
int emei_i2p_step_noisy_f32(const float* state_in, float* state_out, float* obs_out, const void* action, float* reward,
                            uint8_t* done, double* stats, int64_t n, const emei_i2p_params* p,
                            const emei_noise_params* z, emei_stream_t stream);
int emei_i2p_step_noisy_f64(const double* state_in, double* state_out, double* obs_out, const void* action,
                            double* reward, uint8_t* done, double* stats, int64_t n, const emei_i2p_params* p,
                            const emei_noise_params* z, emei_stream_t stream);

/* ---- charged ball ----------------------------------------------------------------------------- */
typedef struct emei_charged_ball_params {
  double gravity_acc, mass_ball, radius, charge, time_step; /* charged_ball.py:13-17 */
  int32_t freq_rate;   /* sub-step = time_step / freq_rate (charged_ball.py:58,63) */
  int32_t action_kind; /* EMEI_ACTION_* ; continuous: E = charge * a (evaluated in float32, see DESIGN.md) */
} emei_charged_ball_params;

/* Replaces freq_rate x update_state(_get_update_info(E)) (charged_ball.py:54-82) with helpers
 * circle_to_free/free_to_circle/_get_angle/_angle_greater (:25-52), reward (:158-160), terminal (:110-111).
 * In-place on the three state arrays: on_circle uint8[n], circle [n,2]={theta,omega}, free [n,4]={x,y,vx,vy}
 * (free IS the observation, charged_ball.py:96-97). */
int emei_charged_ball_step_f32(uint8_t* on_circle, float* circle, float* free_state, const void* action, float* reward,
                               uint8_t* done, double* stats, int64_t n, const emei_charged_ball_params* p,
                               emei_stream_t stream);
int emei_charged_ball_step_f64(uint8_t* on_circle, double* circle, double* free_state, const void* action,
                               double* reward, uint8_t* done, double* stats, int64_t n,
                               const emei_charged_ball_params* p, emei_stream_t stream);

/* Fused T-step charged-ball rollout (float32): as emei_cartpole_rollout_f32 (zoo/util.py:33-93 batched) with the
 * three state arrays of emei_charged_ball_step_f32 kept in registers for all `horizon` steps; per step the arithmetic
 * is exactly emei_charged_ball_step_f32's.  terminated is always 0 (charged_ball.py:110-111), so episodes end by the
 * TimeLimit only (register_env.py:34-43: 500 / 1000 steps).  The in-kernel reset is charged_ball.py:84-94
 * (r->init_kind / init_* are ignored).  Records: observations / next_observations are the `free` array. */
int emei_charged_ball_rollout_f32(uint8_t* on_circle_io, float* circle_io, float* free_state_io, int32_t* episode_step_io,
                                  float* episode_return_io, int32_t* episode_index_io, const void* actions,
                                  float* rec_observations, float* rec_next_observations, void* rec_actions,
                                  float* rec_rewards, uint8_t* rec_dones, uint8_t* rec_timeouts, double* stats, int64_t n,
                                  const emei_charged_ball_params* p, const emei_rollout_params* r, emei_stream_t stream);

/* ---- fused rollouts in the arithmetic of the step entry points (both precisions) -------------------------
 * Same contract as emei_cartpole_rollout_f32 (zoo/util.py:33-93 batched: policy, step, TimeLimit, auto-reset, optional
 * records, six statistics) for what the packed float32 kernels do not cover: the float64 reference-exact mode, the
 * analytic inverted double pendulum (the four I2P tasks of zoo/conf/task/BI2P*.yaml) and obs_noise_params (Gaussian
 * state noise after every sub-step, mujoco_env.py:98-104).  One env per thread; per step the arithmetic is the device
 * function the step kernel calls:
 *   emei_cartpole_rollout_ref_f64 == horizon x emei_cartpole_step_f64   (z == NULL) / emei_ip_step_noisy_f64 (z != NULL)
 *   emei_cartpole_rollout_ref_f32 == horizon x emei_ip_step_noisy_f32   (z != NULL, EMEI_IP_* variants; with z == NULL it
 *        is the same arithmetic without noise, NOT the lean emei_cartpole_step_f32 bits -- use emei_cartpole_rollout_f32
 *        for those)
 *   emei_i2p_rollout_{f32,f64}    == horizon x emei_i2p_step_* / emei_i2p_step_noisy_*
 *   emei_charged_ball_rollout_ref_f64 == horizon x emei_charged_ball_step_f64 (emei_charged_ball_rollout_f32, not the _ref_f32
 *        symbol, is the one that equals emei_charged_ball_step_f32)
 * bit for bit, plus the bookkeeping.
 * Accuracy of the two float32 _ref symbols (and of emei_ip_step_noisy_f32): the float32 envelope of the lean kernels, 1e-5 rel +
 * 1e-6 abs per teacher-forced step against the float64 reference from the same float32 state, at any angle and freq_rate
 * (flags exact away from their thresholds).  The cart-pole / IP step runs its sub-steps in float64 on the widened state and
 * rounds once; the charged ball's landing angle uses the cancellation-free form of the lean kernel.  z->step = env-step counter of the FIRST step of the call (step t uses step + t).
 * In-kernel resets: the arithmetic of emei_init_uniform / emei_init_gaussian / emei_init_charged_ball in this precision
 * with seed = r->seed_reset + episode_index * 0xD1B54A32D192ED03.  Records and episode_return_io have the real type;
 * observations are [T, n, D] with D = 4 (6 for I2P: current_obs, inverted_double_pendulum.py:56-60).
 * I2P: init_mean / init_sigma are HOST arrays of 6 (reset_model: init_qpos || init_qvel, noise per coordinate). */
int emei_cartpole_rollout_ref_f32(float* state_io, int32_t* episode_step_io, float* episode_return_io, int32_t* episode_index_io,
                                  const void* actions, float* rec_observations, float* rec_next_observations, void* rec_actions,
                                  float* rec_rewards, uint8_t* rec_dones, uint8_t* rec_timeouts, double* stats, int64_t n,
                                  const emei_cartpole_params* p, const emei_rollout_params* r, const emei_noise_params* z,
                                  emei_stream_t stream);
int emei_cartpole_rollout_ref_f64(double* state_io, int32_t* episode_step_io, double* episode_return_io, int32_t* episode_index_io,
                                  const void* actions, double* rec_observations, double* rec_next_observations, void* rec_actions,
                                  double* rec_rewards, uint8_t* rec_dones, uint8_t* rec_timeouts, double* stats, int64_t n,
                                  const emei_cartpole_params* p, const emei_rollout_params* r, const emei_noise_params* z,
                                  emei_stream_t stream);
int emei_i2p_rollout_f32(float* state_io, int32_t* episode_step_io, float* episode_return_io, int32_t* episode_index_io,
                         const void* actions, float* rec_observations, float* rec_next_observations, void* rec_actions,
                         float* rec_rewards, uint8_t* rec_dones, uint8_t* rec_timeouts, double* stats, int64_t n,
                         const emei_i2p_params* p, const emei_rollout_params* r, const double* init_mean, const double* init_sigma,
                         const emei_noise_params* z, emei_stream_t stream);
int emei_i2p_rollout_f64(double* state_io, int32_t* episode_step_io, double* episode_return_io, int32_t* episode_index_io,
                         const void* actions, double* rec_observations, double* rec_next_observations, void* rec_actions,
                         double* rec_rewards, uint8_t* rec_dones, uint8_t* rec_timeouts, double* stats, int64_t n,
                         const emei_i2p_params* p, const emei_rollout_params* r, const double* init_mean, const double* init_sigma,
                         const emei_noise_params* z, emei_stream_t stream);
int emei_charged_ball_rollout_ref_f32(uint8_t* on_circle_io, float* circle_io, float* free_state_io, int32_t* episode_step_io,
                                      float* episode_return_io, int32_t* episode_index_io, const void* actions,
                                      float* rec_observations, float* rec_next_observations, void* rec_actions, float* rec_rewards,
                                      uint8_t* rec_dones, uint8_t* rec_timeouts, double* stats, int64_t n,
                                      const emei_charged_ball_params* p, const emei_rollout_params* r, emei_stream_t stream);
int emei_charged_ball_rollout_ref_f64(uint8_t* on_circle_io, double* circle_io, double* free_state_io, int32_t* episode_step_io,
                                      double* episode_return_io, int32_t* episode_index_io, const void* actions,
                                      double* rec_observations, double* rec_next_observations, void* rec_actions, double* rec_rewards,
                                      uint8_t* rec_dones, uint8_t* rec_timeouts, double* stats, int64_t n,
                                      const emei_charged_ball_params* p, const emei_rollout_params* r, emei_stream_t stream);

/* ---- sampling-based MPC over the true dynamics (CEM / MPPI; DESIGN.md 4.10) ------------------------------
 * One planner iteration is two launches: *_plan_eval_* scores K candidate action sequences of H steps from each of B start
 * states, emei_plan_update_* refits the [H, B] plan distribution from their returns.  Nothing of the env moves: like the
 * trajectory entry points this is an open-loop model query (no TimeLimit, resets, state noise or statistics).
 * Candidate actions: drawn in-kernel from Philox4x32-10 keyed by (seed, (env_offset + b) * 2^32 + k), so results do not
 * depend on how the start states are sharded:
 *   continuous kinds: step t uses the Box-Muller pair of block t >> 1 (cos half for even t, sin half for odd t),
 *     a = clamp(R(mean[t,b] + std[t,b] z)), product and sum rounded in double, clamped in R to [action_low, action_high]
 *     (a float32 action array in a float64 plan holds that value rounded to float32);
 *   discrete kinds: step t uses word t & 3 of block t >> 2, a = ((w >> 8) 2^-24 < float(mean[t,b])) ? 1 : 0, mean being the
 *     probability of action 1 (std unused, may be NULL).
 * Return R_bk = sum_{t<H} gamma^t r_t in double (ret = ret + disc r_t; disc = disc gamma; each operation rounded on its own);
 * the reward of the step that terminates counts, later steps do not.  Per step the arithmetic is that of the env's fused
 * rollout in the same precision (emei_cartpole_rollout_f32 / emei_charged_ball_rollout_f32 for float32 cart-pole, IP and
 * charged ball, the *_rollout_ref_* / emei_i2p_rollout_* kernels otherwise), so the rewards of a candidate equal a
 * teacher-forced rollout of its actions bit for bit.  The family params' action_kind is replaced by the plan's. */
#define EMEI_PLAN_CEM 0
#define EMEI_PLAN_MPPI 1
#define EMEI_PLAN_MAX_CANDIDATES 4096
typedef struct emei_plan_params {
  uint64_t seed;       /* Philox key of the candidate actions */
  uint64_t env_offset; /* global id of start state 0 (sharding) */
  double gamma;        /* discount, in [0, 1] */
  double temperature;  /* MPPI lambda, > 0 */
  double momentum;     /* alpha in [0, 1): mean <- alpha mean + (1 - alpha) fit_mean, the same for std */
  double min_std;      /* std floor, >= 0 */
  float action_low, action_high; /* continuous kinds: the action box (low <= high) */
  int32_t method;      /* EMEI_PLAN_CEM | EMEI_PLAN_MPPI */
  int32_t elites;      /* CEM: E in [1, K] */
  int32_t action_kind; /* EMEI_ACTION_*: discrete or continuous, and the element type of actions_out / best_actions */
} emei_plan_params;

/* eval: state0 [B,D] (cart-pole rows, or qpos || qvel with unwrapped angles, as the trajectory entry points take them;
 * 16-byte aligned) / the charged ball's on_circle [B], circle [B,2], free [B,4] (circle and free 16-byte aligned);
 * mean, std [H,B] in the real type; returns [B,K] double (written once); actions_out [H,B,K] in the action kind's type,
 * nullable (so actions_out viewed as [H, B*K] is the actions array of a teacher-forced rollout of B*K envs whose state is
 * each start repeated K times).  Validation: B < 0, H < 0 or H >= 2^31, K outside [1, 4096] -> EMEI_ERR_BAD_SIZE; NULL
 * params; the family params as the step entry points check them; the plan params (action kind -> EMEI_ERR_BAD_ACTION_KIND;
 * method, E outside [1, K] for CEM, temperature <= 0 for MPPI, gamma outside [0, 1], momentum outside [0, 1), min_std < 0,
 * action_low > action_high -> EMEI_ERR_BAD_PARAM); B == 0 or H == 0 returns EMEI_OK with nothing launched; then NULL state,
 * mean, returns (std for continuous kinds) and the alignment.  All before any launch. */
int emei_cartpole_plan_eval_f32(const float* state0, const float* mean, const float* std, double* returns, void* actions_out, int64_t B,
                                int64_t K, int64_t H, const emei_plan_params* plan, const emei_cartpole_params* p, emei_stream_t stream);
int emei_cartpole_plan_eval_f64(const double* state0, const double* mean, const double* std, double* returns, void* actions_out,
                                int64_t B, int64_t K, int64_t H, const emei_plan_params* plan, const emei_cartpole_params* p,
                                emei_stream_t stream);
int emei_i2p_plan_eval_f32(const float* state0, const float* mean, const float* std, double* returns, void* actions_out, int64_t B,
                           int64_t K, int64_t H, const emei_plan_params* plan, const emei_i2p_params* p, emei_stream_t stream);
int emei_i2p_plan_eval_f64(const double* state0, const double* mean, const double* std, double* returns, void* actions_out, int64_t B,
                           int64_t K, int64_t H, const emei_plan_params* plan, const emei_i2p_params* p, emei_stream_t stream);
int emei_charged_ball_plan_eval_f32(const uint8_t* on_circle, const float* circle, const float* free_state, const float* mean,
                                    const float* std, double* returns, void* actions_out, int64_t B, int64_t K, int64_t H,
                                    const emei_plan_params* plan, const emei_charged_ball_params* p, emei_stream_t stream);
int emei_charged_ball_plan_eval_f64(const uint8_t* on_circle, const double* circle, const double* free_state, const double* mean,
                                    const double* std, double* returns, void* actions_out, int64_t B, int64_t K, int64_t H,
                                    const emei_plan_params* plan, const emei_charged_ball_params* p, emei_stream_t stream);
/* update, one CTA per start state; reads returns [B,K], regenerates the chosen candidates' actions from the counters above
 * (same seed, env_offset and mean / std as the eval call) and refits mean_io / std_io [H,B] in place:
 *   CEM: the E best candidates under the total order (larger return first, ties to the smaller k, NaN below every number);
 *        fit_mean = their mean action, fit_std = their population std (discrete: fit_mean = their frequency of action 1);
 *   MPPI: w_k = exp((R_k - max R) / temperature) / sum (a weight that is not a number counts 0; all 0: uniform);
 *        fit_mean = sum w a, fit_std = sqrt(sum w (a - fit_mean)^2);
 *   both: mean <- momentum mean + (1 - momentum) fit_mean (discrete: clamped to [0, 1]);
 *         std <- max(momentum std + (1 - momentum) fit_std, min_std).
 * Sums are in double in a fixed order (bit-reproducible); results are rounded once to the real type.  std_io is required
 * for continuous kinds and unused for discrete ones.  best_actions [H,B] (the action kind's type) and best_return [B]
 * (double): the argmax candidate under the same order, each nullable.  Validation as the eval entry points, without family
 * params and alignment.  The update needs nothing but the returns, so a caller may score candidates with a model of its own
 * (actions_out gives it the actions) and refit with this kernel. */
int emei_plan_update_f32(const double* returns, float* mean_io, float* std_io, void* best_actions, double* best_return, int64_t B,
                         int64_t K, int64_t H, const emei_plan_params* plan, emei_stream_t stream);
int emei_plan_update_f64(const double* returns, double* mean_io, double* std_io, void* best_actions, double* best_return, int64_t B,
                         int64_t K, int64_t H, const emei_plan_params* plan, emei_stream_t stream);

/* ---- policy search over the true dynamics: linear feedback policies, ARS (DESIGN.md 4.11) ------------------------
 * A policy of an env with observation dimension D (cart-pole, IP, charged ball: 4; I2P: 6) is theta = (w_0 .. w_{D-1}, c), P = D + 1
 * doubles.  At every step it acts on the observation the env's step() returns in that state (IP: the wrapped angle; I2P: the
 * reference's (theta + pi) % 2 * pi - pi; charged ball: the free state; the first action: the start state's observation):
 *   u = c; u = u + w_j double(obs_j) for j = 0 .. D-1, each product and sum rounded on its own (no contraction);
 *   continuous kinds: a = clamp(R(u)) to [action_low, action_high], clamped in R (a float32 action array in a float64 eval holds
 *     that value rounded to float32); discrete kinds: a = u > 0 ? 1 : 0 (NaN: 0).
 * One ARS iteration (Mania, Guy & Recht 2018, V1-t) is emei_policy_perturb (2N candidates around theta), *_policy_eval_* (their
 * returns from E start states) and emei_policy_update (the step along the b best directions).  Nothing of the env moves. */
#define EMEI_POLICY_MAX_DIRECTIONS 4096
#define EMEI_POLICY_MAX_PARAMS 8
typedef struct emei_policy_params {
  uint64_t seed;                 /* Philox key of the directions delta_k (perturb / update) */
  double gamma;                  /* eval: discount, in [0, 1] */
  double noise;                  /* perturb: nu, finite and >= 0 */
  double step_size;              /* update: alpha, finite */
  float action_low, action_high; /* eval, continuous kinds: the action box (low <= high) */
  int32_t action_kind;           /* eval: EMEI_ACTION_*, discrete or continuous and the element type of actions_out */
  int32_t top;                   /* update: b, the number of directions stepped along, in [1, N] */
} emei_policy_params;

/* eval: params [C,P] double (P = D + 1); start states as the plan eval takes them: state0 [E,D] (16-byte aligned; angles
 * unwrapped) / the charged ball's on_circle [E], circle [E,2], free [E,4] (circle and free 16-byte aligned).  Every (c, e) runs
 * closed loop from start e for H steps; returns [C,E] double = sum_{t<H} gamma^t r_t in double (ret = ret + disc r_t; disc =
 * disc gamma), the reward of the step that terminates counts, later steps do not; no TimeLimit, reset or noise.  actions_out
 * [H,C,E] in the action kind's type, nullable; when given, a pair keeps stepping after it terminates, so actions_out viewed as
 * [H, C*E] teacher-forces a rollout of C*E envs (start e of candidate c at row c*E + e, auto_reset off, no TimeLimit) whose
 * rewards and observations are the eval's bit for bit.  Per step the arithmetic is the plan eval's, that of the env's own
 * rollout in that precision.  The family params' action_kind is replaced by the policy's.
 * Validation, in order: C, E < 0 or > 2^31, H < 0 or >= 2^31 -> EMEI_ERR_BAD_SIZE; NULL policy / family params; the family
 * params; action kind (EMEI_ERR_BAD_ACTION_KIND; the double pendulum's entry points refuse discrete kinds too), gamma outside
 * [0, 1] or action_low > action_high for a continuous kind -> EMEI_ERR_BAD_PARAM; C, E or H == 0 returns EMEI_OK with
 * nothing launched; then NULL state, params, returns and the alignment.  All before any launch. */
int emei_cartpole_policy_eval_f32(const float* state0, const double* params, double* returns, void* actions_out, int64_t C, int64_t E,
                                  int64_t H, const emei_policy_params* policy, const emei_cartpole_params* p, emei_stream_t stream);
int emei_cartpole_policy_eval_f64(const double* state0, const double* params, double* returns, void* actions_out, int64_t C, int64_t E,
                                  int64_t H, const emei_policy_params* policy, const emei_cartpole_params* p, emei_stream_t stream);
int emei_i2p_policy_eval_f32(const float* state0, const double* params, double* returns, void* actions_out, int64_t C, int64_t E,
                             int64_t H, const emei_policy_params* policy, const emei_i2p_params* p, emei_stream_t stream);
int emei_i2p_policy_eval_f64(const double* state0, const double* params, double* returns, void* actions_out, int64_t C, int64_t E,
                             int64_t H, const emei_policy_params* policy, const emei_i2p_params* p, emei_stream_t stream);
int emei_charged_ball_policy_eval_f32(const uint8_t* on_circle, const float* circle, const float* free_state, const double* params,
                                      double* returns, void* actions_out, int64_t C, int64_t E, int64_t H,
                                      const emei_policy_params* policy, const emei_charged_ball_params* p, emei_stream_t stream);
int emei_charged_ball_policy_eval_f64(const uint8_t* on_circle, const double* circle, const double* free_state, const double* params,
                                      double* returns, void* actions_out, int64_t C, int64_t E, int64_t H,
                                      const emei_policy_params* policy, const emei_charged_ball_params* p, emei_stream_t stream);
/* perturb: direction k < N draws delta_k in R^P from Philox4x32-10 keyed by (seed, k) with purpose word 8: block j gives
 * delta_{2j} = rad cs and delta_{2j+1} = rad sn of the Box-Muller pair (the library's sampler).  Writes params [2N,P]:
 * params[2k] = theta + nu delta_k, params[2k+1] = theta - nu delta_k, each element one rounded product and one rounded sum.
 * theta [P] double.  Validation: N outside [1, 4096] or P outside [1, 8] -> EMEI_ERR_BAD_SIZE; NULL policy params; noise not
 * finite or < 0 -> EMEI_ERR_BAD_PARAM; NULL theta / params. */
int emei_policy_perturb(const double* theta, double* params, int64_t N, int64_t P, const emei_policy_params* policy,
                        emei_stream_t stream);
/* update (one CTA): r_k+ / r_k- = the mean over e (ascending, in double) of returns [2N,E] rows 2k / 2k+1.  Direction k is
 * eligible when both are finite; the b' = min(top, #eligible) eligible directions with the largest max(r_k+, r_k-) (ties to the
 * smaller k) give sigma_R, the population std of their 2b' returns, and
 *   theta <- theta + step_size / (b' sigma_R) sum_k (r_k+ - r_k-) delta_k
 * with delta_k regenerated from (seed, k).  When b' = 0 or sigma_R is not a finite number > 0, theta is unchanged.  Sums run in a fixed
 * order (bit-reproducible).  stats double[4], nullable: b', sigma_R, the best eligible max(r_k+, r_k-) and the mean of every
 * finite r_k+- (NaN where there is none).  Validation: N outside [1, 4096], E outside [1, 2^31] or P outside [1, 8] ->
 * EMEI_ERR_BAD_SIZE; NULL policy params; top outside [1, N] or step_size not finite -> EMEI_ERR_BAD_PARAM; NULL returns /
 * theta_io. */
int emei_policy_update(const double* returns, double* theta_io, double* stats, int64_t N, int64_t E, int64_t P,
                       const emei_policy_params* policy, emei_stream_t stream);

/* ---- model-based scoring: get_batch_reward + get_batch_terminal fused ------------------------- */
typedef struct emei_scoring_params {
  int32_t family;                  /* EMEI_* family id */
  int32_t terminate_when_unhealthy; /* Hopper (hopper.py:31) */
  double forward_reward_weight, ctrl_cost_weight, healthy_reward; /* hopper.py:26-28, half_cheetah.py:22-23 */
  double healthy_state_lo, healthy_state_hi; /* hopper.py:33 */
  double healthy_z_lo, healthy_z_hi;         /* hopper.py:34 */
  double dt;                        /* MujocoEnv.dt = real_time_scale * freq_rate */
  double x_threshold, theta_threshold; /* cart-pole */
  double x_left, x_right;           /* IP / I2P rail (model.jnt_range[0]) */
  double radius;                    /* charged ball */
} emei_scoring_params;

/* Replaces get_batch_reward + get_batch_terminal of every in-scope env:
 * cartpole.py:124-129,145-151; inverted_pendulum.py:73-79,103-111,139-146,174-183;
 * inverted_double_pendulum.py:84-90,114-122,150-157,185-196; hopper.py:79-106; half_cheetah.py:59-67;
 * charged_ball.py:110-111,158-160.
 *   obs [n,D] ; pre_obs [n,D] (only column 0 is read; Hopper/HalfCheetah only; nullable otherwise);
 *   reward [n] ; done [n] ; stats nullable ;
 *   sumsq : DEVICE double* holding the batch-wide sum of squared actions (Hopper/HalfCheetah control
 *           cost is summed over the WHOLE batch, hopper.py:98, half_cheetah.py:61); produced by
 *           emei_sumsq_* (and all-reduced across ranks by the caller when the batch is sharded);
 *           ignored for other families (nullable). */
int emei_reward_terminal_f32(const float* obs, const float* pre_obs, float* reward, uint8_t* done, double* stats,
                             const double* sumsq, int64_t n, const emei_scoring_params* p, emei_stream_t stream);
int emei_reward_terminal_f64(const double* obs, const double* pre_obs, double* reward, uint8_t* done, double* stats,
                             const double* sumsq, int64_t n, const emei_scoring_params* p, emei_stream_t stream);

/* Trajectory form of the same scoring (the layout an MBRL scorer holds its imagined rollouts in):
 *   obs_seq [horizon + 1, n_envs, D] ; transition (t, j) has obs = obs_seq[t + 1, j], pre_obs = obs_seq[t, j]
 *   (hopper.py:95-97 / half_cheetah.py:60: x_velocity = (obs[:,0] - pre_obs[:,0]) / dt) ;
 *   reward [horizon, n_envs] ; done [horizon, n_envs] ; sumsq over the action tensor [horizon, n_envs, A].
 * Equal, bit for bit, to emei_reward_terminal_* on obs = obs_seq[1:], pre_obs = obs_seq[:-1] flattened -- and that
 * call takes the same kernel whenever pre_obs + k*D == obs (k >= 256): one thread walks the time steps of an env and
 * carries obs[t][0] in a register, so every observation row is read ONCE (65 / 101 bytes per Hopper / HalfCheetah
 * transition instead of the 113 / 173 bytes of DRAM traffic a separate strided pre_obs[:,0] column costs).
 * n_envs * D * sizeof(real) must be a multiple of 16. */
int emei_reward_terminal_seq_f32(const float* obs_seq, float* reward, uint8_t* done, double* stats, const double* sumsq,
                                 int64_t n_envs, int64_t horizon, const emei_scoring_params* p, emei_stream_t stream);
int emei_reward_terminal_seq_f64(const double* obs_seq, double* reward, uint8_t* done, double* stats, const double* sumsq,
                                 int64_t n_envs, int64_t horizon, const emei_scoring_params* p, emei_stream_t stream);

/* sum of squares of n_elems values, accumulated in double, written to *out (device).
 * Replaces np.sum(np.square(action)) (hopper.py:98, half_cheetah.py:61).  One launch, deterministic:
 * per-CTA partials go to `workspace` and the last CTA adds them in index order (no floating-point
 * atomics), so repeated calls on the same data return the same bits.
 *   workspace : DEVICE buffer of EMEI_SUMSQ_WORKSPACE_BYTES bytes, 8-byte aligned, zero-filled ONCE
 *               by the caller before its first use (the kernel leaves its ticket counter at zero);
 *               not shared between concurrent streams. */
#define EMEI_SUMSQ_WORKSPACE_BYTES ((148 * 8 + 1) * 8)
int emei_sumsq_f32(const float* x, int64_t n_elems, double* out, double* workspace, emei_stream_t stream);
int emei_sumsq_f64(const double* x, int64_t n_elems, double* out, double* workspace, emei_stream_t stream);
/* the plain sum of n_elems values: the reduction of emei_sumsq_* without the square, same workspace contract and the same
 * run-to-run bits (the batch-wide sum of the reward cotangents that the control cost's derivative needs). */
int emei_sum_f32(const float* x, int64_t n_elems, double* out, double* workspace, emei_stream_t stream);
int emei_sum_f64(const double* x, int64_t n_elems, double* out, double* workspace, emei_stream_t stream);

/* ---- derivatives of the scoring (vector-Jacobian products) ---------------------------------------
 * What is differentiated: the real-valued reward emei_reward_terminal_* evaluates on the caller's rows, almost everywhere.
 * `done` and Hopper's healthy term are piecewise constant: no gradient.  Per family (o = obs row, p = pre_obs row):
 *   cart-pole balancing, IP / I2P balancing : constant reward, zero gradient
 *   cart-pole swing-up    : d/do2 = -sin(o2)/2          IP swing-ups: d/do1 = sin(o1)/2
 *   I2P swing-ups         : d/do1 = (sin o1 + sin(o1+o2))/4, d/do2 = sin(o1+o2)/4; boundary also d/do4 = -1e-2 o4, d/do5 = -2e-4 o5
 *   Hopper, HalfCheetah   : d/do0 = fwd_w/dt, d/dp0 = -fwd_w/dt, d/da = -2 ctrl_w a summed over EVERY reward of the batch:
 *                           g_action = -2 ctrl_w G action with G = sum of the reward cotangents (emei_sum_*; all-reduced by
 *                           the caller when the control cost is global over a sharded batch)
 *   charged ball          : d/do0,1 = -o0,1 / (radius rho), rho = sqrt(o0^2 + o1^2); 0 at rho = 0
 * _f32 evaluates these in float32 (a tolerance product).  Non-finite inputs give non-finite gradients where the derivative
 * reads them.  Validation: n < 0 (n_envs, horizon < 0) -> EMEI_ERR_BAD_SIZE; then the checks of emei_reward_terminal_*
 * in its order (params, family -> EMEI_ERR_BAD_VARIANT, Hopper / HalfCheetah dt <= 0 -> EMEI_ERR_BAD_PARAM); n == 0 or
 * horizon == 0 is a no-op.  obs may be NULL only for the families whose gradient does not read it (the constant rewards,
 * Hopper, HalfCheetah); g_reward is required; a non-NULL g_action needs action and g_reward_sum and is rejected
 * (EMEI_ERR_BAD_PARAM) for the families whose reward does not read the action.  obs, action, every gradient array: 16-byte
 * aligned. */
/* VJP of emei_reward_terminal_*: g_reward [n] ; g_reward_sum DEVICE double* = G ; g_obs [n,D], g_pre_obs [n,D] (dense rows),
 * g_action [n,A] (A = emei_family_action_dim): each nullable (not written). */
int emei_reward_vjp_f32(const float* obs, const float* action, const float* g_reward, const double* g_reward_sum, float* g_obs,
                        float* g_pre_obs, float* g_action, int64_t n, const emei_scoring_params* p, emei_stream_t stream);
int emei_reward_vjp_f64(const double* obs, const double* action, const double* g_reward, const double* g_reward_sum,
                        double* g_obs, double* g_pre_obs, double* g_action, int64_t n, const emei_scoring_params* p,
                        emei_stream_t stream);
/* VJP of emei_reward_terminal_seq_*: obs_seq [horizon+1,n_envs,D] ; g_reward [horizon,n_envs] ;
 * g_obs_seq [horizon+1,n_envs,D] (required, every row written once): row t = d/d obs of transition t-1 + d/d pre_obs of
 * transition t ; g_action [horizon,n_envs,A] nullable, G summed over all horizon * n_envs rewards.
 * n_envs * D * sizeof(real) must be a multiple of 16 (as for emei_reward_terminal_seq_*). */
int emei_reward_seq_vjp_f32(const float* obs_seq, const float* action, const float* g_reward, const double* g_reward_sum,
                            float* g_obs_seq, float* g_action, int64_t n_envs, int64_t horizon, const emei_scoring_params* p,
                            emei_stream_t stream);
int emei_reward_seq_vjp_f64(const double* obs_seq, const double* action, const double* g_reward, const double* g_reward_sum,
                            double* g_obs_seq, double* g_action, int64_t n_envs, int64_t horizon, const emei_scoring_params* p,
                            emei_stream_t stream);

/* ---- batched initial-state sampling (counter-based Philox4x32-10; see DESIGN.md) -------------- */
/* value(env, column) depends only on (seed, env_offset + row, column): independent of sharding. */
/* cartpole.py:131-132,153-156: U(-0.05,0.05) on 4 columns, + pi on column `pi_column` (-1 = none) */
int emei_init_uniform_f32(float* out, int64_t n, int32_t dim, double low, double high, int32_t pi_column,
                          uint64_t seed, uint64_t env_offset, emei_stream_t stream);
int emei_init_uniform_f64(double* out, int64_t n, int32_t dim, double low, double high, int32_t pi_column,
                          uint64_t seed, uint64_t env_offset, emei_stream_t stream);
/* mujoco_env.py:137-140,197-249 (+ transform_state_to_obs :142-144): out[r,c] = mean[c] + sigma[c]*N(0,1);
 * mean/sigma are HOST arrays of length dim (dim <= 32), copied by value into the launch. */
int emei_init_gaussian_f32(float* out, int64_t n, int32_t dim, const double* mean, const double* sigma, uint64_t seed,
                           uint64_t env_offset, emei_stream_t stream);
int emei_init_gaussian_f64(double* out, int64_t n, int32_t dim, const double* mean, const double* sigma, uint64_t seed,
                           uint64_t env_offset, emei_stream_t stream);
/* charged_ball.py:84-94: [theta,omega] = U(-.5,.5,2) + [pi,0]; on_circle = 1; free = circle_to_free */
int emei_init_charged_ball_f32(uint8_t* on_circle, float* circle, float* free_state, int64_t n, double radius,
                               uint64_t seed, uint64_t env_offset, emei_stream_t stream);
int emei_init_charged_ball_f64(uint8_t* on_circle, double* circle, double* free_state, int64_t n, double radius,
                               uint64_t seed, uint64_t env_offset, emei_stream_t stream);

/* ---- freeze / unfreeze --------------------------------------------------------------------------
 * Replaces `frozen_state = state.copy()` / `state = frozen_state.copy()` (base_control.py:32-36,
 * mujoco_env.py:114-120): device-side 128-bit vectorised snapshot copy.  dst/src 16-byte aligned
 * unless bytes % 16 != 0 (byte tail handled). */
int emei_snapshot_copy(void* dst, const void* src, int64_t bytes, emei_stream_t stream);

/* ---- rollout records -> dataset order --------------------------------------------------------------
 * The reference writes its offline datasets episode after episode (zoo/util.py:33-93,108-111: flat arrays
 * observations, next_observations, actions, rewards, dones, timeouts).  The fused rollouts record time-major
 * [horizon, n] arrays; this transposes one of them to env-major [n, horizon] (each env's trajectory, hence each
 * of its episodes, contiguous).  elem_bytes: 1 (dones, timeouts, uint8 actions), 4 (float32 rewards, float/int32
 * actions), 8 (float64 rewards, int64/double actions), 16 (float32 observation rows of 4), 24 (float32 rows of 6: the
 * inverted double pendulum), 32 (float64 rows of 4), 48 (float64 rows of 6); any other size is EMEI_ERR_BAD_PARAM.
 * in/out aligned to elem_bytes for 1, 4, 8 and 16, to 8 for 24 and to 16 for 32 and 48 (else EMEI_ERR_MISALIGNED). */
int emei_records_transpose(const void* in, void* out, int64_t horizon, int64_t n, int32_t elem_bytes, emei_stream_t stream);

/* ---- statistics --------------------------------------------------------------------------------- */
int emei_stats_reset(double* stats, emei_stream_t stream); /* zero double[2] */

/* ---- misc ----------------------------------------------------------------------------------------- */
int emei_version(void);
const char* emei_error_string(int code);
/* obs / action width of a family (e.g. HOPPER -> 12 / 3); -1 for an unknown family */
int emei_family_obs_dim(int family);
int emei_family_action_dim(int family);

#ifdef __cplusplus
}
#endif
#endif /* EMEI_B200_H */
