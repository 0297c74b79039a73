// Shared device helpers for the emei_b200 kernels (sm_100a).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/emei_b200.h"

namespace emei {

constexpr int kBlock = 256;   // threads per CTA for the streaming kernels
constexpr int kNumSMs = 148;  // B200 (upper bound used for workspace sizes; launches query the device, sm_count())
constexpr int kMaxDevices = 64;

inline int current_device() {
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess || d < 0 || d >= kMaxDevices) d = 0;
  return d;
}

// SM count of the CURRENT device (a process may drive envs on several GPUs); cached per device, immutable after first use
inline int sm_count() {
  static int cache[kMaxDevices] = {};
  const int d = current_device();
  int v = cache[d];
  if (v <= 0) {
    if (cudaDeviceGetAttribute(&v, cudaDevAttrMultiProcessorCount, d) != cudaSuccess || v <= 0) v = kNumSMs;
    cache[d] = v;  // benign race: every thread writes the same value
  }
  return v;
}

#define EMEI_CHECK_PTR(p) \
  if ((p) == nullptr) return EMEI_ERR_NULL_POINTER
#define EMEI_CHECK_ALIGN16(p) \
  if ((reinterpret_cast<uintptr_t>(p) & 15u) != 0) return EMEI_ERR_MISALIGNED

inline int launch_status() {
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? EMEI_OK : static_cast<int>(e);
}

// ---------------------------------------------------------------------------------------------
// parameter checks shared by the entry points of each family, in the order every entry point applies them
// ---------------------------------------------------------------------------------------------
inline bool action_kind_valid(int ak) { return ak >= EMEI_ACTION_DISCRETE_U8 && ak <= EMEI_ACTION_CONTINUOUS_F64; }
inline int check_cartpole_params(const emei_cartpole_params& p) {
  if (p.variant < EMEI_CARTPOLE_BALANCING || p.variant > EMEI_IP_BOUNDARY_SWINGUP) return EMEI_ERR_BAD_VARIANT;
  if (!action_kind_valid(p.action_kind)) return EMEI_ERR_BAD_ACTION_KIND;
  if (p.freq_rate < 1 || !(p.dt > 0.0)) return EMEI_ERR_BAD_PARAM;
  return EMEI_OK;
}
inline int check_i2p_params(const emei_i2p_params& p) {
  if (p.variant < EMEI_I2P_REBOUND_BALANCING || p.variant > EMEI_I2P_BOUNDARY_SWINGUP) return EMEI_ERR_BAD_VARIANT;
  if (!action_kind_valid(p.action_kind)) return EMEI_ERR_BAD_ACTION_KIND;
  if (p.freq_rate < 1 || !(p.dt > 0.0) || !(p.mass_cart > 0.0) || !(p.mass_pole0 > 0.0) || !(p.mass_pole1 > 0.0) ||
      !(p.length0 > 0.0) || !(p.length1 > 0.0))
    return EMEI_ERR_BAD_PARAM;
  return EMEI_OK;
}
inline int check_charged_ball_params(const emei_charged_ball_params& p) {
  if (!action_kind_valid(p.action_kind)) return EMEI_ERR_BAD_ACTION_KIND;
  if (p.freq_rate < 1 || !(p.time_step > 0.0) || !(p.radius > 0.0) || !(p.mass_ball > 0.0)) return EMEI_ERR_BAD_PARAM;
  return EMEI_OK;
}
// state noise: sigma[0, dim) >= 0 (no noise: EMEI_OK)
inline int check_noise_params(const emei_noise_params* z, int dim) {
  if (z != nullptr)
    for (int j = 0; j < dim; ++j)
      if (!(z->sigma[j] >= 0.0)) return EMEI_ERR_BAD_PARAM;
  return EMEI_OK;
}

inline int grid_for(int64_t n, int per_block) {
  int64_t g = (n + per_block - 1) / per_block;
  return static_cast<int>(g);
}

// persistent launch: enough CTAs to cover n once, capped at ctas_per_sm resident CTAs on every SM
// (the kernels grid-stride over the rest, so every SM carries the same number of units +-1)
inline int persistent_grid(int64_t n, int per_block, int ctas_per_sm) {
  const int64_t want = (n + per_block - 1) / per_block;
  const int64_t cap = static_cast<int64_t>(sm_count()) * ctas_per_sm;
  return static_cast<int>(want < 1 ? 1 : (want > cap ? cap : want));
}

// persistent grid sized by the kernel's ACTUAL residency (registers / shared memory decide how many
// CTAs fit on an SM; a grid larger than one resident wave would run a ragged second wave).  The
// occupancy query result is cached per kernel instantiation (immutable after first use).
template <typename... KArgs>
inline int resident_grid(void (*kernel)(KArgs...), int64_t n) {
  static int per_sm[kMaxDevices] = {};  // per kernel instantiation AND per device
  const int d = current_device();
  int nb = per_sm[d];
  if (nb < 1) {
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kernel, kBlock, 0) != cudaSuccess || nb < 1) nb = 4;
    per_sm[d] = nb;
  }
  return persistent_grid(n, kBlock, nb);
}

// ---------------------------------------------------------------------------------------------
// Programmatic dependent launch (sm_90+): a rollout is a chain of short (~10 us) step kernels on one
// stream, so the launch latency between them is a visible fraction of the step.  Kernels launched
// through launch_pdl() may start (CTA scheduling, parameter loads, index arithmetic) while the tail
// of the previous kernel in the stream drains; they call pdl_wait() before their first global
// memory access, which blocks until the previous grid has fully completed and its writes are
// visible, and pdl_trigger() at their top so that THEIR successor may be staged early in turn.
// With a non-participating neighbour (memcpy, a torch kernel) both calls are no-ops and ordering is
// the ordinary stream order.  Captured into CUDA graphs as programmatic edges.
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }

// smem: dynamic shared memory bytes (the overload without it launches with none)
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), int grid, int block, size_t smem, cudaStream_t stream, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(static_cast<unsigned>(grid), 1, 1);
  cfg.blockDim = dim3(static_cast<unsigned>(block), 1, 1);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), int grid, int block, cudaStream_t stream, Args... args) {
  return launch_pdl(kernel, grid, block, size_t{0}, stream, args...);
}

// ---------------------------------------------------------------------------------------------
// vector types: one env row (4 scalars) per 128-bit (f32) / 2 x 128-bit (f64) access
// ---------------------------------------------------------------------------------------------
template <typename R>
struct Vec4;
template <>
struct Vec4<float> {
  float x, y, z, w;
  __device__ __forceinline__ static Vec4 load(const float* p) {
    float4 v = *reinterpret_cast<const float4*>(p);
    return {v.x, v.y, v.z, v.w};
  }
  __device__ __forceinline__ void store(float* p) const { *reinterpret_cast<float4*>(p) = make_float4(x, y, z, w); }
};
template <>
struct Vec4<double> {
  double x, y, z, w;
  __device__ __forceinline__ static Vec4 load(const double* p) {
    double2 a = reinterpret_cast<const double2*>(p)[0];
    double2 b = reinterpret_cast<const double2*>(p)[1];
    return {a.x, a.y, b.x, b.y};
  }
  __device__ __forceinline__ void store(double* p) const {
    reinterpret_cast<double2*>(p)[0] = make_double2(x, y);
    reinterpret_cast<double2*>(p)[1] = make_double2(z, w);
  }
};

// ---------------------------------------------------------------------------------------------
// actions
// ---------------------------------------------------------------------------------------------
// discrete: +mag if a == 1 else -mag ; continuous: float32 product mag*a (the reference evaluates
// `python_float * np.float32` in float32 under NEP 50), widened to R.
template <typename R>
__device__ __forceinline__ R load_force(const void* action, int64_t i, int kind, R mag) {
  switch (kind) {
    case EMEI_ACTION_DISCRETE_U8:
      return static_cast<const uint8_t*>(action)[i] == 1 ? mag : -mag;
    case EMEI_ACTION_DISCRETE_I32:
      return static_cast<const int32_t*>(action)[i] == 1 ? mag : -mag;
    case EMEI_ACTION_DISCRETE_I64:
      return static_cast<const long long*>(action)[i] == 1 ? mag : -mag;
    case EMEI_ACTION_CONTINUOUS_F32:
      return static_cast<R>(__fmul_rn(static_cast<float>(mag), static_cast<const float*>(action)[i]));
    default:
      return static_cast<R>(__fmul_rn(static_cast<float>(mag), static_cast<float>(static_cast<const double*>(action)[i])));
  }
}
// raw continuous control value (IP: ctrl in double = widened float32 action)
template <typename R>
__device__ __forceinline__ R load_ctrl(const void* action, int64_t i, int kind) {
  switch (kind) {
    case EMEI_ACTION_DISCRETE_U8:
      return static_cast<R>(static_cast<const uint8_t*>(action)[i]);
    case EMEI_ACTION_DISCRETE_I32:
      return static_cast<R>(static_cast<const int32_t*>(action)[i]);
    case EMEI_ACTION_DISCRETE_I64:
      return static_cast<R>(static_cast<const long long*>(action)[i]);
    case EMEI_ACTION_CONTINUOUS_F32:
      return static_cast<R>(static_cast<const float*>(action)[i]);
    default:
      return static_cast<R>(static_cast<const double*>(action)[i]);
  }
}

// ---------------------------------------------------------------------------------------------
// per-launch statistics: sum(reward), count(done).  warp shuffle -> smem -> one atomic per CTA
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Per-thread reward partial + done COUNT of the thread's units.  Must be called by ALL threads of the CTA.
__device__ __forceinline__ void block_stats_accumulate_counts(double* stats, double reward_sum, unsigned done_count) {
  if (stats == nullptr) return;  // uniform across the grid
  __shared__ double s_r2[kBlock / 32];
  __shared__ unsigned s_d2[kBlock / 32];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const double r = warp_sum(reward_sum);
  const unsigned d = __reduce_add_sync(0xffffffffu, done_count);
  if (lane == 0) {
    s_r2[warp] = r;
    s_d2[warp] = d;
  }
  __syncthreads();
  if (warp == 0) {
    const int nw = blockDim.x >> 5;
    double rr = lane < nw ? s_r2[lane] : 0.0;
    unsigned dd = lane < nw ? s_d2[lane] : 0u;
    rr = warp_sum(rr);
    dd = __reduce_add_sync(0xffffffffu, dd);
    if (lane == 0) {
      atomicAdd(&stats[0], rr);
      atomicAdd(&stats[1], static_cast<double>(dd));  // exact: counts << 2^53
    }
  }
}

// ---------------------------------------------------------------------------------------------
// floored modulo (python / numpy `%` for floats): sign of the divisor
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double py_mod(double a, double b) {
  double m = fmod(a, b);
  if (m != 0.0) {
    if ((b < 0.0) != (m < 0.0)) m += b;
  } else {
    m = copysign(0.0, b);
  }
  return m;
}
__device__ __forceinline__ float py_mod(float a, float b) {
  float m = fmodf(a, b);
  if (m != 0.0f) {
    if ((b < 0.0f) != (m < 0.0f)) m += b;
  } else {
    m = copysignf(0.0f, b);
  }
  return m;
}

// python `a % 2` (the double pendulum's observation, inverted_double_pendulum.py:59) without fmod's remainder loop:
// a - 2 trunc(a / 2) consists of exact operations only for every finite a (a / 2 and 2 t are scalings by a power of two; for
// |a| >= 2^p the float is an even integer and the difference is 0, below that the difference of the two is representable), so it
// IS fmod(a, 2) -- same bits, the sign of a zero aside, which python's fix-up below discards; Inf -> NaN, NaN -> NaN like fmod.
__device__ __forceinline__ double py_mod2(double a) {
  double m = a - 2.0 * trunc(a * 0.5);
  if (m != 0.0) {
    if (m < 0.0) m += 2.0;
  } else {
    m = 0.0;
  }
  return m;
}
__device__ __forceinline__ float py_mod2(float a) {
  float m = a - 2.0f * truncf(a * 0.5f);
  if (m != 0.0f) {
    if (m < 0.0f) m += 2.0f;
  } else {
    m = 0.0f;
  }
  return m;
}

// float32 observation wrap `(theta + pi) % (2 pi) - pi` (inverted_pendulum.py:45-49) by Cody-Waite
// reduction: exact for |theta| < pi (forming theta + pi in float32 would cost 1.2e-7 of the 1e-6 budget),
// error <= ulp(theta) beyond.  Result in [-pi_f, pi_f); NaN / Inf -> NaN like the reference.
__device__ __forceinline__ float wrap_pi_f32(float th) {
  const float k = rintf(th * 0.15915494309189535f);
  float r = fmaf(-k, 6.28125f, th);  // 2 pi = 6.28125 + 1.9353071795864769e-3
  r = fmaf(-k, 1.9353071795864769e-3f, r);
  r = r >= 3.14159265358979323846f ? r - 6.28318530717958647692f : r;
  r = r < -3.14159265358979323846f ? r + 6.28318530717958647692f : r;
  return r;
}

template <typename R>
__device__ __forceinline__ bool is_finite(R v) {
  return isfinite(v);
}

__device__ __forceinline__ void sincos_r(float a, float* s, float* c) { sincosf(a, s, c); }
__device__ __forceinline__ void sincos_r(double a, double* s, double* c) { sincos(a, s, c); }
__device__ __forceinline__ float cos_r(float a) { return cosf(a); }
__device__ __forceinline__ double cos_r(double a) { return cos(a); }
__device__ __forceinline__ float sin_r(float a) { return sinf(a); }
__device__ __forceinline__ double sin_r(double a) { return sin(a); }
__device__ __forceinline__ float sqrt_r(float a) { return sqrtf(a); }
__device__ __forceinline__ double sqrt_r(double a) { return sqrt(a); }
__device__ __forceinline__ float asin_r(float a) { return asinf(a); }
__device__ __forceinline__ double asin_r(double a) { return asin(a); }
__device__ __forceinline__ float abs_r(float a) { return fabsf(a); }
__device__ __forceinline__ double abs_r(double a) { return fabs(a); }

// ---------------------------------------------------------------------------------------------
// Philox4x32-10 (Salmon et al. 2011), counter-based: value = f(seed, env id, column)
// ---------------------------------------------------------------------------------------------
struct Philox {
  static constexpr uint32_t kM0 = 0xD2511F53u, kM1 = 0xCD9E8D57u, kW0 = 0x9E3779B9u, kW1 = 0xBB67AE85u;
  __host__ __device__ static inline void round(uint32_t (&c)[4], uint32_t k0, uint32_t k1) {
    const uint64_t p0 = static_cast<uint64_t>(kM0) * c[0];
    const uint64_t p1 = static_cast<uint64_t>(kM1) * c[2];
    const uint32_t hi0 = static_cast<uint32_t>(p0 >> 32), lo0 = static_cast<uint32_t>(p0);
    const uint32_t hi1 = static_cast<uint32_t>(p1 >> 32), lo1 = static_cast<uint32_t>(p1);
    const uint32_t n0 = hi1 ^ c[1] ^ k0, n1 = lo1, n2 = hi0 ^ c[3] ^ k1, n3 = lo0;
    c[0] = n0;
    c[1] = n1;
    c[2] = n2;
    c[3] = n3;
  }
  // counter = (env_lo, env_hi, block, purpose), key = (seed_lo, seed_hi)
  __host__ __device__ static inline void generate(uint64_t seed, uint64_t env, uint32_t block, uint32_t purpose,
                                                  uint32_t (&out)[4]) {
    uint32_t c[4] = {static_cast<uint32_t>(env), static_cast<uint32_t>(env >> 32), block, purpose};
    uint32_t k0 = static_cast<uint32_t>(seed), k1 = static_cast<uint32_t>(seed >> 32);
#pragma unroll
    for (int r = 0; r < 10; ++r) {
      round(c, k0, k1);
      k0 += kW0;
      k1 += kW1;
    }
    out[0] = c[0];
    out[1] = c[1];
    out[2] = c[2];
    out[3] = c[3];
  }
};

// Philox purpose words (the counter's last word): one per random stream of the library
constexpr uint32_t kPurposeUniform = 1;        // initial states, uniform families
constexpr uint32_t kPurposeGaussian = 2;       // initial states, Gaussian families
constexpr uint32_t kPurposeChargedBall = 3;    // initial states, charged ball
constexpr uint32_t kPurposeRolloutAction = 4;  // the rollouts' random policy
constexpr uint32_t kPurposeRolloutReset = 5;   // the float32 rollouts' lean uniform reset
constexpr uint32_t kPurposeObsNoise = 6;       // per-sub-step state noise (bits 8..: the high word of the block index)

// 53-bit uniform in [0,1) from two 32-bit words (same construction as numpy's next_double)
__host__ __device__ inline double u01_from_bits(uint32_t hi, uint32_t lo) {
  const uint64_t a = hi >> 5, b = lo >> 6;  // 27 + 26 bits
  return (static_cast<double>(a) * 67108864.0 + static_cast<double>(b)) * (1.0 / 9007199254740992.0);
}

}  // namespace emei
