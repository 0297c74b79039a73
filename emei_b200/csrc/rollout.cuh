// The rollout contract shared by the packed float32 rollout kernel (rollout_f32.cuh) and the reference-arithmetic rollout
// kernel (rollout_ref.cuh): the kernel form of emei_rollout_params, the I/O pointers, the argument checks, the random
// policy's stream and the reset seed of an episode.
#pragma once
#include "kernels.cuh"

namespace emei {

// The kernel form of emei_rollout_params.  G: the columns of the Gaussian reset's tables, 4 in the packed kernel and 6 in the
// reference kernel (the double pendulum).  The packed kernel's reset sampler is a call that takes this struct by reference,
// so that kernel keeps a local copy of it: two more columns would add 32-48 bytes to the stack frame of each of its
// cart-pole instances.
template <int G>
struct RolloutConsts {
  int horizon, max_episode_steps, auto_reset, random_policy, init_kind /*0 uniform, 1 gaussian, 2 charged ball*/, init_pi_column;
  unsigned long long seed_reset, seed_action, env_offset, t0;
  double init_low, init_high, mean[G], sigma[G];
  float act_low, act_high;
};

// everything that is not the env family's own state; R is the real type of the records and episode returns
template <typename R>
struct RolloutIO {
  int32_t* ep_step;
  R* ep_return;
  int32_t* ep_index;
  const void* actions;
  R* rec_obs;
  R* rec_next;
  void* rec_act;
  R* rec_rew;
  uint8_t* rec_done;
  uint8_t* rec_timeout;
  double* stats;
};

// Checks of the episode buffers, horizon, actions and records (all-or-nothing; align_obs: the two observation arrays must be
// 16-byte aligned), then the conversion of *r.  mean / sigma: the Gaussian reset's tables (nullptr: the first four columns
// come from r, the others are 0).  Returns EMEI_OK or an error code.
template <typename R, int G>
inline int make_rollout(const emei_rollout_params* r, const RolloutIO<R>& io, bool align_obs, const double* mean, const double* sigma,
                        RolloutConsts<G>& rc) {
  EMEI_CHECK_PTR(io.ep_step);
  EMEI_CHECK_PTR(io.ep_return);
  EMEI_CHECK_PTR(io.ep_index);
  if (r->horizon < 0) return EMEI_ERR_BAD_PARAM;
  if (!r->random_policy) EMEI_CHECK_PTR(io.actions);
  if (io.rec_obs != nullptr) {
    EMEI_CHECK_PTR(io.rec_next);
    EMEI_CHECK_PTR(io.rec_act);
    EMEI_CHECK_PTR(io.rec_rew);
    EMEI_CHECK_PTR(io.rec_done);
    EMEI_CHECK_PTR(io.rec_timeout);
    if (align_obs) {
      EMEI_CHECK_ALIGN16(io.rec_obs);
      EMEI_CHECK_ALIGN16(io.rec_next);
    }
  }
  rc.horizon = r->horizon;
  rc.max_episode_steps = r->max_episode_steps;
  rc.auto_reset = r->auto_reset;
  rc.random_policy = r->random_policy;
  rc.init_kind = r->init_kind;
  rc.init_pi_column = r->init_pi_column;
  rc.seed_reset = r->seed_reset;
  rc.seed_action = r->seed_action;
  rc.env_offset = r->env_offset;
  rc.t0 = r->t0;
  rc.init_low = r->init_low;
  rc.init_high = r->init_high;
  for (int j = 0; j < G; ++j) {
    rc.mean[j] = mean != nullptr ? mean[j] : (j < 4 ? r->init_mean[j] : 0.0);
    rc.sigma[j] = sigma != nullptr ? sigma[j] : (j < 4 ? r->init_sigma[j] : 0.0);
  }
  rc.act_low = static_cast<float>(r->action_low);
  rc.act_high = static_cast<float>(r->action_high);
  return EMEI_OK;
}

// w[j] for a run-time j without putting the array in local memory
__device__ __forceinline__ uint32_t select_word(const uint32_t (&w)[4], unsigned j) {
  const uint32_t lo = (j & 1u) ? w[1] : w[0], hi = (j & 1u) ? w[3] : w[2];
  return (j & 2u) ? hi : lo;
}

__device__ __forceinline__ double block_sum_double(double v, double* smem /*[kBlock/32]*/) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) smem[warp] = v;
  __syncthreads();
  double t = lane < kBlock / 32 ? smem[lane] : 0.0;
  return warp_sum(t);  // valid in every lane of every warp
}

// Philox key of the reset sample of an env's episode k (include/emei_b200.h)
__device__ __forceinline__ unsigned long long reset_seed(unsigned long long seed_reset, int k) {
  return seed_reset + static_cast<unsigned long long>(k) * 0xD1B54A32D192ED03ull;
}

}  // namespace emei
