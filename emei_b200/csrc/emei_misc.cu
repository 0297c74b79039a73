// snapshot copy (freeze/unfreeze), statistics reset, version / error strings.
#include "common.cuh"

namespace emei {

// 128-bit grid-stride copy; 4 independent loads in flight per thread before the stores.
__global__ void __launch_bounds__(kBlock) snapshot_copy_kernel(uint4* __restrict__ dst, const uint4* __restrict__ src,
                                                               int64_t nvec) {
  const int64_t stride = static_cast<int64_t>(gridDim.x) * kBlock;
  int64_t j = static_cast<int64_t>(blockIdx.x) * kBlock + threadIdx.x;
  for (; j + 3 * stride < nvec; j += 4 * stride) {
    uint4 a = __ldcs(src + j), b = __ldcs(src + j + stride), c = __ldcs(src + j + 2 * stride),
          d = __ldcs(src + j + 3 * stride);
    __stcs(dst + j, a);
    __stcs(dst + j + stride, b);
    __stcs(dst + j + 2 * stride, c);
    __stcs(dst + j + 3 * stride, d);
  }
  for (; j < nvec; j += stride) __stcs(dst + j, __ldcs(src + j));
}

__global__ void snapshot_tail_kernel(uint8_t* __restrict__ dst, const uint8_t* __restrict__ src, int64_t begin,
                                     int64_t bytes) {
  const int64_t j = begin + threadIdx.x;
  if (j < bytes) dst[j] = src[j];
}

// Time-major rollout records [T, n] (one element per (step, env)) -> env-major [n, T]: every env's trajectory becomes
// contiguous, which is the order of the reference's dataset files (zoo/util.py:33-93 appends whole episodes one
// after another).  32 x 32 tiles through shared memory: reads coalesced along n, writes coalesced along T.
// HBM-bound: 2 x bytes.
template <typename E>
__global__ void __launch_bounds__(kBlock) records_transpose_kernel(const E* __restrict__ in, E* __restrict__ out, int64_t T,
                                                                   int64_t n, int64_t tiles_n, int64_t tiles) {
  __shared__ E tile[32][33];
  const int lx = threadIdx.x & 31, ly = threadIdx.x >> 5;  // 32 x 8
  for (int64_t tl = blockIdx.x; tl < tiles; tl += gridDim.x) {
    const int64_t t0 = (tl / tiles_n) * 32, i0 = (tl % tiles_n) * 32;
#pragma unroll
    for (int r = 0; r < 32; r += 8) {
      const int64_t t = t0 + ly + r, i = i0 + lx;
      if (t < T && i < n) tile[ly + r][lx] = in[t * n + i];
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 32; r += 8) {
      const int64_t i = i0 + ly + r, t = t0 + lx;
      if (t < T && i < n) out[i * T + t] = tile[lx][ly + r];
    }
    __syncthreads();
  }
}

// Wide elements (observation rows of 24, 32 or 48 bytes: 6 x float32, 4 x float64, 6 x float64) moved as K words W
// (uint2 for 24 bytes, which a [T, n, 6] float32 tensor only aligns to 8; uint4 otherwise).  A 32 x 32 tile of 48-byte
// elements is 50.7 KB, over the 48 KB of static shared memory, so the tile is 16 steps x 32 envs (25.3 KB at 48 bytes).
// It stays coalesced both ways because an element is wide: a tile row read is 32 contiguous elements of in (768 to
// 1536 bytes) and a tile row written is 16 contiguous elements of out (384 to 768 bytes), each taken by consecutive
// threads word after word.  The shared rows are padded by one element ((32 + 1) * K words), so that the row stride is
// K words modulo the bank width: in both phases consecutive threads touch consecutive banks.
constexpr int kWideTileT = 16, kWideTileN = 32;

template <typename W, int K>
__global__ void __launch_bounds__(kBlock) records_transpose_wide_kernel(const W* __restrict__ in, W* __restrict__ out, int64_t T,
                                                                        int64_t n, int64_t tiles_n, int64_t tiles) {
  constexpr int kRow = (kWideTileN + 1) * K;  // words per shared row (one time step of the tile)
  constexpr int kIn = kWideTileN * K;         // words per tile row read from in (one time step)
  constexpr int kOut = kWideTileT * K;        // words per tile row written to out (one env)
  constexpr int kWords = kWideTileT * kWideTileN * K;
  static_assert(kWords % kBlock == 0, "whole passes over the tile");
  __shared__ W tile[kWideTileT][kRow];
  for (int64_t tl = blockIdx.x; tl < tiles; tl += gridDim.x) {
    const int64_t t0 = (tl / tiles_n) * kWideTileT, i0 = (tl % tiles_n) * kWideTileN;
#pragma unroll
    for (int p = 0; p < kWords / kBlock; ++p) {
      const int j = p * kBlock + threadIdx.x;
      const int r = j / kIn, w = j % kIn;  // step r of the tile, word w of its row = word w % K of env w / K
      const int64_t t = t0 + r;
      if (t < T && i0 + w / K < n) tile[r][w] = in[(t * n + i0) * K + w];
    }
    __syncthreads();
#pragma unroll
    for (int p = 0; p < kWords / kBlock; ++p) {
      const int j = p * kBlock + threadIdx.x;
      const int c = j / kOut, w = j % kOut;  // env c of the tile, word w of its row = word w % K of step w / K
      const int64_t i = i0 + c;
      if (t0 + w / K < T && i < n) out[(i * T + t0) * K + w] = tile[w / K][c * K + w % K];
    }
    __syncthreads();
  }
}

template <typename E>
inline void launch_records_transpose(const void* in, void* out, int64_t T, int64_t n, cudaStream_t s) {
  const int64_t tiles_n = (n + 31) / 32, tiles = tiles_n * ((T + 31) / 32);
  const int64_t cap = static_cast<int64_t>(kNumSMs) * 8;
  const int grid = static_cast<int>(tiles < cap ? tiles : cap);
  records_transpose_kernel<E><<<grid, kBlock, 0, s>>>(static_cast<const E*>(in), static_cast<E*>(out), T, n, tiles_n, tiles);
}

template <typename W, int K>
inline void launch_records_transpose_wide(const void* in, void* out, int64_t T, int64_t n, cudaStream_t s) {
  const int64_t tiles_n = (n + kWideTileN - 1) / kWideTileN, tiles = tiles_n * ((T + kWideTileT - 1) / kWideTileT);
  const int64_t cap = static_cast<int64_t>(kNumSMs) * 8;
  const int grid = static_cast<int>(tiles < cap ? tiles : cap);
  records_transpose_wide_kernel<W, K><<<grid, kBlock, 0, s>>>(static_cast<const W*>(in), static_cast<W*>(out), T, n, tiles_n, tiles);
}

// the alignment a record element of elem_bytes needs (that of the words it is moved in); 0: not a record element size
inline int records_elem_align(int32_t elem_bytes) {
  switch (elem_bytes) {
    case 1: case 4: case 8: case 16: return elem_bytes;
    case 24: return 8;
    case 32: case 48: return 16;
    default: return 0;
  }
}

}  // namespace emei

extern "C" {

int emei_records_transpose(const void* in, void* out, int64_t horizon, int64_t n, int32_t elem_bytes, emei_stream_t stream) {
  using namespace emei;
  if (horizon < 0 || n < 0) return EMEI_ERR_BAD_SIZE;
  const int align = records_elem_align(elem_bytes);
  if (align == 0) return EMEI_ERR_BAD_PARAM;
  if (horizon == 0 || n == 0) return EMEI_OK;
  EMEI_CHECK_PTR(in);
  EMEI_CHECK_PTR(out);
  if (((reinterpret_cast<uintptr_t>(in) | reinterpret_cast<uintptr_t>(out)) & static_cast<uintptr_t>(align - 1)) != 0)
    return EMEI_ERR_MISALIGNED;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  switch (elem_bytes) {
    case 1: launch_records_transpose<uint8_t>(in, out, horizon, n, s); break;
    case 4: launch_records_transpose<uint32_t>(in, out, horizon, n, s); break;
    case 8: launch_records_transpose<uint2>(in, out, horizon, n, s); break;
    case 16: launch_records_transpose<uint4>(in, out, horizon, n, s); break;
    case 24: launch_records_transpose_wide<uint2, 3>(in, out, horizon, n, s); break;
    case 32: launch_records_transpose_wide<uint4, 2>(in, out, horizon, n, s); break;
    default: launch_records_transpose_wide<uint4, 3>(in, out, horizon, n, s); break;
  }
  return launch_status();
}

int emei_snapshot_copy(void* dst, const void* src, int64_t bytes, emei_stream_t stream) {
  using namespace emei;
  if (bytes < 0) return EMEI_ERR_BAD_SIZE;
  if (bytes == 0) return EMEI_OK;
  EMEI_CHECK_PTR(dst);
  EMEI_CHECK_PTR(src);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const bool aligned = ((reinterpret_cast<uintptr_t>(dst) | reinterpret_cast<uintptr_t>(src)) & 15u) == 0;
  if (!aligned) {  // rare: fall back to the runtime's D2D copy engine path
    cudaError_t e = cudaMemcpyAsync(dst, src, static_cast<size_t>(bytes), cudaMemcpyDeviceToDevice, s);
    return e == cudaSuccess ? EMEI_OK : static_cast<int>(e);
  }
  const int64_t nvec = bytes / 16;
  if (nvec > 0) {
    int64_t want = (nvec + kBlock * 4 - 1) / (kBlock * 4);
    const int64_t cap = static_cast<int64_t>(kNumSMs) * 8;
    const int grid = static_cast<int>(want < 1 ? 1 : (want > cap ? cap : want));
    snapshot_copy_kernel<<<grid, kBlock, 0, s>>>(static_cast<uint4*>(dst), static_cast<const uint4*>(src), nvec);
  }
  if (nvec * 16 < bytes)
    snapshot_tail_kernel<<<1, 16, 0, s>>>(static_cast<uint8_t*>(dst), static_cast<const uint8_t*>(src), nvec * 16, bytes);
  return launch_status();
}

int emei_stats_reset(double* stats, emei_stream_t stream) {
  EMEI_CHECK_PTR(stats);
  cudaError_t e = cudaMemsetAsync(stats, 0, 2 * sizeof(double), static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? EMEI_OK : static_cast<int>(e);
}

int emei_version(void) { return EMEI_B200_VERSION; }

const char* emei_error_string(int code) {
  switch (code) {
    case EMEI_OK:
      return "ok";
    case EMEI_ERR_NULL_POINTER:
      return "emei_b200: required pointer is NULL";
    case EMEI_ERR_BAD_VARIANT:
      return "emei_b200: unknown env family / variant";
    case EMEI_ERR_BAD_ACTION_KIND:
      return "emei_b200: unknown action encoding";
    case EMEI_ERR_BAD_SIZE:
      return "emei_b200: negative or out-of-range size";
    case EMEI_ERR_MISALIGNED:
      return "emei_b200: pointer must be 16-byte aligned";
    case EMEI_ERR_BAD_PARAM:
      return "emei_b200: invalid parameter value (freq_rate < 1, dt <= 0, ...)";
    default:
      return code > 0 ? cudaGetErrorString(static_cast<cudaError_t>(code)) : "emei_b200: unknown error code";
  }
}

int emei_family_obs_dim(int family) {
  if (family < 0 || family >= EMEI_NUM_FAMILIES) return -1;
  if (family == EMEI_HOPPER) return 12;
  if (family == EMEI_HALFCHEETAH) return 18;
  if (family >= EMEI_I2P_REBOUND_BALANCING && family <= EMEI_I2P_BOUNDARY_SWINGUP) return 6;
  return 4;
}

int emei_family_action_dim(int family) {
  if (family < 0 || family >= EMEI_NUM_FAMILIES) return -1;
  if (family == EMEI_HOPPER) return 3;
  if (family == EMEI_HALFCHEETAH) return 6;
  return 1;
}

}  // extern "C"
