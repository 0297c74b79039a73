// extern "C" entry points of the fused float32 rollouts (rollout_f32.cuh).
#include "rollout_f32.cuh"

using namespace emei;

extern "C" int emei_cartpole_rollout_f32(float* state_io, int32_t* episode_step_io, float* episode_return_io,
                                         int32_t* episode_index_io, const void* actions, float* rec_observations,
                                         float* rec_next_observations, void* rec_actions, float* rec_rewards,
                                         uint8_t* rec_dones, uint8_t* rec_timeouts, double* stats, int64_t n,
                                         const emei_cartpole_params* p, const emei_rollout_params* r,
                                         emei_stream_t stream) {
  if (n < 0 || n > kCartPoleMaxLaunch) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(p);
  EMEI_CHECK_PTR(r);
  if (const int e = check_cartpole_params(*p)) return e;
  if (r->horizon < 0 || (r->init_kind != 0 && r->init_kind != 1)) return EMEI_ERR_BAD_PARAM;
  if (n == 0 || r->horizon == 0) return EMEI_OK;
  EMEI_CHECK_PTR(state_io);
  EMEI_CHECK_ALIGN16(state_io);
  const RolloutIO<float> io = {episode_step_io, episode_return_io, episode_index_io, actions, rec_observations, rec_next_observations,
                               rec_actions, rec_rewards, rec_dones, rec_timeouts, stats};
  RolloutConsts<4> rc;
  if (const int e = make_rollout(r, io, true, nullptr, nullptr, rc)) return e;
  const CartPoleF32Consts k = make_cartpole_f32_consts(*p);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const bool ip = p->variant > EMEI_CARTPOLE_SWINGUP;
  const int ak = p->action_kind;
  if (!ip) {
    if (p->freq_rate == 1) launch_cartpole_rollout<false, 1>(ak, state_io, io, n, k, rc, s);
    else if (p->freq_rate == 4) launch_cartpole_rollout<false, 4>(ak, state_io, io, n, k, rc, s);
    else launch_cartpole_rollout<false, 0>(ak, state_io, io, n, k, rc, s);
  } else {
    if (p->freq_rate == 1) launch_cartpole_rollout<true, 1>(ak, state_io, io, n, k, rc, s);
    else if (p->freq_rate == 4) launch_cartpole_rollout<true, 4>(ak, state_io, io, n, k, rc, s);
    else launch_cartpole_rollout<true, 0>(ak, state_io, io, n, k, rc, s);
  }
  return launch_status();
}

extern "C" int emei_charged_ball_rollout_f32(uint8_t* on_circle_io, float* circle_io, float* free_state_io,
                                             int32_t* episode_step_io, float* episode_return_io, int32_t* episode_index_io,
                                             const void* actions, float* rec_observations, float* rec_next_observations,
                                             void* rec_actions, float* rec_rewards, uint8_t* rec_dones,
                                             uint8_t* rec_timeouts, double* stats, int64_t n,
                                             const emei_charged_ball_params* p, const emei_rollout_params* r,
                                             emei_stream_t stream) {
  if (n < 0 || n > kCartPoleMaxLaunch) return EMEI_ERR_BAD_SIZE;
  EMEI_CHECK_PTR(p);
  EMEI_CHECK_PTR(r);
  if (const int e = check_charged_ball_params(*p)) return e;
  if (r->horizon < 0) return EMEI_ERR_BAD_PARAM;
  if (n == 0 || r->horizon == 0) return EMEI_OK;
  EMEI_CHECK_PTR(on_circle_io);
  EMEI_CHECK_PTR(circle_io);
  EMEI_CHECK_PTR(free_state_io);
  EMEI_CHECK_ALIGN16(circle_io);
  EMEI_CHECK_ALIGN16(free_state_io);
  const RolloutIO<float> io = {episode_step_io, episode_return_io, episode_index_io, actions, rec_observations, rec_next_observations,
                               rec_actions, rec_rewards, rec_dones, rec_timeouts, stats};
  RolloutConsts<4> rc;
  if (const int e = make_rollout(r, io, true, nullptr, nullptr, rc)) return e;
  rc.init_kind = 2;  // charged_ball.py:84-94 is the only reset sampler of this family
  launch_charged_ball_rollout(p->action_kind, on_circle_io, circle_io, free_state_io, io, n, make_cb_f32_consts(*p), rc,
                              static_cast<cudaStream_t>(stream));
  return launch_status();
}
