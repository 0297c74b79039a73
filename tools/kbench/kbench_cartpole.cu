// Kernel-level experiment harness (development tool, not shipped): times variants of the float32
// cart-pole step kernel and a pure streaming kernel with the same 41 B/env traffic, on a ring of
// batches larger than L2, K launches captured in one CUDA graph (same protocol as bench.py).
//   nvcc -O3 -std=c++17 -gencode arch=compute_100a,code=sm_100a -o /tmp/kbench tools/kbench/kbench_cartpole.cu
#include <cstdio>
#include <cstdlib>
#include <vector>
#include "../../emei_b200/csrc/cartpole_tma.cuh"

using namespace emei;
#include <cstring>
static const char* g_filter = nullptr;  // argv[4]: run only the variants whose name contains it
#define SKIP(name) if (g_filter && !strstr(name, g_filter)) return

#define CK(x) do { cudaError_t err_ = (x); if (err_ != cudaSuccess) { printf("CUDA error %s at %s:%d\n", cudaGetErrorString(err_), __FILE__, __LINE__); exit(1);} } while (0)

// pure streaming: same loads/stores, no math (the memory-system floor for this access pattern)
template <int MINB>
__global__ void __launch_bounds__(kBlock, MINB)
stream_kernel(const float4* in, float4* out, const float* __restrict__ act, float* __restrict__ rew, uint8_t* __restrict__ done, uint32_t n) {
  const uint32_t stride = gridDim.x * kBlock;
  pdl_trigger();
  pdl_wait();
  for (uint32_t i = blockIdx.x * kBlock + threadIdx.x; i < n; i += stride) {
    float4 y = in[i];
    float a = __ldg(act + i);
    y.x += a;
    out[i] = y;
    rew[i] = y.y;
    done[i] = y.z > 0.f;
  }
}

// compute only: the same per-env arithmetic on register-resident synthetic states, no HBM traffic.
// OLD = full sincos at every sub-step (the first two generations); otherwise the shipped integrator (one sincos + angle addition)
template <int MINB, int FR, bool OLD>
__global__ void __launch_bounds__(kBlock, MINB)
compute_kernel(float* out, uint32_t n, const CartPoleF32Consts k) {
  const uint32_t stride = gridDim.x * kBlock;
  float acc = 0.f;
  for (uint32_t i = blockIdx.x * kBlock + threadIdx.x; i < n; i += stride) {
    float4 y = make_float4(1e-6f * i, 0.5f, 2e-6f * i, -1.0f);
    const float f_mt = 1e-7f * i;
    float c;
    if (OLD) {
#pragma unroll
      for (int sub = 0; sub < FR; ++sub) f32::cartpole_substep<false>(y.x, y.y, y.z, y.w, f_mt, 0u, k.k);
      c = f32::cos_core(y.z);
    } else {
      f32::LaneMax<float> dm;
      c = f32::cartpole_integrate<float, FR>(y.x, y.y, y.z, y.w, -f_mt, 0u, k.k, FR, dm);
      acc += dm.m;
    }
    acc += fmaf(c, 0.5f, 0.5f) + y.x + y.y + y.w;
  }
  if (acc == 12345.678f) out[0] = acc;
}

// compute only, packed f32x2: two envs per thread (the arithmetic of the shipped step kernel)
template <int MINB, int FR, bool OLD>
__global__ void __launch_bounds__(kBlock, MINB)
compute2_kernel(float* out, uint32_t n, const CartPoleF32Consts k) {
  using f32::f2;
  const uint32_t stride = gridDim.x * kBlock * 2;
  float acc = 0.f;
  for (uint32_t i = blockIdx.x * kBlock * 2 + threadIdx.x; i < n; i += stride) {
    f2 X = f32::f2_pack(1e-6f * i, 2e-6f * i), V = f32::f2_pack(0.5f, 0.25f), TH = f32::f2_pack(2e-6f * i, 1e-6f * i), W = f32::f2_pack(-1.f, 1.f);
    const f2 nf = f32::f2_pack(1e-7f * i, -1e-7f * i);
    f2 C;
    if (OLD) {
#pragma unroll
      for (int sub = 0; sub < FR; ++sub) f32::cartpole_substep2(X, V, TH, W, nf, 0u, k.k);
      C = f32::cos_core(TH);
    } else {
      f32::LaneMax<f2> dm;
      C = f32::cartpole_integrate<f2, FR>(X, V, TH, W, nf, 0u, k.k, FR, dm);
      acc += dm.a + dm.b;
    }
    float a, b, c, d;
    f32::f2_unpack(C, a, b);
    f32::f2_unpack(vadd(vadd(X, V), W), c, d);
    acc += a + b + c + d;
  }
  if (acc == 12345.678f) out[0] = acc;
}

struct Ring {
  std::vector<float*> in, out, act, rew; std::vector<uint8_t*> done;
};

template <typename F>
float time_graph(F launch, int K, cudaStream_t s, int reps = 5) {
  if (getenv("KBENCH_NOGRAPH")) {  // plain stream launches (what ncu can see)
    for (int i = 0; i < 3; ++i) launch(i);
    CK(cudaStreamSynchronize(s));
    return 0.f;
  }
  cudaGraph_t g; cudaGraphExec_t ge;
  CK(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
  for (int i = 0; i < K; ++i) launch(i);
  CK(cudaStreamEndCapture(s, &g));
  CK(cudaGraphInstantiate(&ge, g, 0));
  CK(cudaGraphLaunch(ge, s)); CK(cudaStreamSynchronize(s));
  cudaEvent_t e0, e1; cudaEventCreate(&e0); cudaEventCreate(&e1);
  float best = 1e30f;
  for (int r = 0; r < reps; ++r) {
    CK(cudaEventRecord(e0, s)); CK(cudaGraphLaunch(ge, s)); CK(cudaEventRecord(e1, s)); CK(cudaStreamSynchronize(s));
    float ms; cudaEventElapsedTime(&ms, e0, e1); if (ms < best) best = ms;
  }
  cudaGraphExecDestroy(ge); cudaGraphDestroy(g);
  return best * 1e3f / K;  // us per launch
}

template <int FR>
void run_tma(const char* name, Ring& R, uint32_t n, int K, cudaStream_t s, int slots_cap = 0) {
  SKIP(name);
  emei_cartpole_params p = {};
  p.gravity = 9.8; p.mass_pole = 0.1; p.total_mass = 1.1; p.length = 0.5; p.pole_mass_length = 0.05; p.force_mag = 10.0;
  p.x_threshold = 5.0; p.theta_threshold = 0.2; p.dt = 0.02; p.freq_rate = 4; p.variant = EMEI_CARTPOLE_SWINGUP;
  p.action_kind = EMEI_ACTION_CONTINUOUS_F32;
  CartPoleF32Consts k = make_cartpole_f32_consts(p);
  const int64_t chunks = (n + kChunk - 1) / kChunk;
  const int grid = (int)(chunks < kNumSMs ? chunks : kNumSMs);
  int n_slots; size_t smem;
  tma_ring_shape(4, (chunks + grid - 1) / grid, &n_slots, &smem);
  // the shipped flags (launch_cartpole_f32_tma): actions staged by TMA, L2 prefetch of the first `depth` chunks
  const int64_t per_cta = (chunks + grid - 1) / grid;
  const int depth = (int)(per_cta / 5 + 1 < 3 ? 3 : (per_cta / 5 + 1 > 8 ? 8 : per_cta / 5 + 1));
  const int flags = 1 | 2 | (depth << 16);
  if (slots_cap && n_slots > slots_cap) { n_slots = slots_cap; smem = (size_t)n_slots * kChunk * 20 + 2 * n_slots * 8 + (kTmaThreads / 32) * 12 + 16; }
  double* stats; CK(cudaMalloc(&stats, 16)); CK(cudaMemset(stats, 0, 16));
  const int ring = (int)R.in.size();
  auto kern = cartpole_step_f32_tma_kernel<false, EMEI_ACTION_CONTINUOUS_F32, FR, false>;
  CK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  auto launch = [&](int i) {
    int j = i % ring;
    launch_pdl(kern, grid, kTmaThreads, smem, s, (const float4*)R.in[j], (float4*)R.out[j], (float4*)nullptr, (const void*)R.act[j], R.rew[j], R.done[j], stats, n, n_slots, flags, k);
  };
  float us = time_graph(launch, K, s);
  CK(cudaGetLastError());
  printf("%-44s grid=%5d  %7.2f us/launch  %6.1f Genv-steps/s  %6.0f GB/s (41 B/env)  slots=%d smem=%zu\n", name, grid, us, n / us * 1e-3, 41.0 * n / us * 1e-3, n_slots, smem);
  cudaFree(stats);
}

template <int MINB, int FR, bool OLD>
void run_compute(const char* name, Ring& R, uint32_t n, int K, cudaStream_t s) {
  SKIP(name);
  emei_cartpole_params p = {};
  p.gravity = 9.8; p.mass_pole = 0.1; p.total_mass = 1.1; p.length = 0.5; p.pole_mass_length = 0.05; p.force_mag = 10.0;
  p.x_threshold = 5.0; p.theta_threshold = 0.2; p.dt = 0.02; p.freq_rate = 4; p.variant = EMEI_CARTPOLE_SWINGUP;
  CartPoleF32Consts k = make_cartpole_f32_consts(p);
  int grid = persistent_grid(n, kBlock, MINB);
  auto launch = [&](int i) { compute_kernel<MINB, FR, OLD><<<grid, kBlock, 0, s>>>(R.rew[0], n, k); };
  float us = time_graph(launch, K, s);
  CK(cudaGetLastError());
  printf("%-44s grid=%5d  %7.2f us/launch\n", name, grid, us);
}

template <int MINB, int FR, bool OLD>
void run_compute2(const char* name, Ring& R, uint32_t n, int K, cudaStream_t s) {
  SKIP(name);
  emei_cartpole_params p = {};
  p.gravity = 9.8; p.mass_pole = 0.1; p.total_mass = 1.1; p.length = 0.5; p.pole_mass_length = 0.05; p.force_mag = 10.0;
  p.x_threshold = 5.0; p.theta_threshold = 0.2; p.dt = 0.02; p.freq_rate = 4; p.variant = EMEI_CARTPOLE_SWINGUP;
  CartPoleF32Consts k = make_cartpole_f32_consts(p);
  int grid = persistent_grid(n, 2 * kBlock, MINB);
  auto launch = [&](int i) { compute2_kernel<MINB, FR, OLD><<<grid, kBlock, 0, s>>>(R.rew[0], n, k); };
  float us = time_graph(launch, K, s);
  CK(cudaGetLastError());
  printf("%-44s grid=%5d  %7.2f us/launch\n", name, grid, us);
}

template <int MINB, bool PDL>
void run_stream(const char* name, Ring& R, uint32_t n, int K, cudaStream_t s) {
  SKIP(name);
  int grid = persistent_grid(n, kBlock, MINB);
  const int ring = (int)R.in.size();
  auto launch = [&](int i) {
    int j = i % ring;
    if (PDL) launch_pdl(stream_kernel<MINB>, grid, kBlock, s, (const float4*)R.in[j], (float4*)R.out[j], (const float*)R.act[j], R.rew[j], R.done[j], n);
    else stream_kernel<MINB><<<grid, kBlock, 0, s>>>((const float4*)R.in[j], (float4*)R.out[j], R.act[j], R.rew[j], R.done[j], n);
  };
  float us = time_graph(launch, K, s);
  CK(cudaGetLastError());
  printf("%-44s grid=%5d  %7.2f us/launch  %6.1f Genv-steps/s  %6.0f GB/s (41 B/env)\n", name, grid, us, n / us * 1e-3, 41.0 * n / us * 1e-3);
}

int main(int argc, char** argv) {
  const uint32_t n = argc > 1 ? (uint32_t)atol(argv[1]) : (1u << 20);
  const int ring = argc > 2 ? atoi(argv[2]) : 8;
  const int K = argc > 3 ? atoi(argv[3]) : 400;
  if (argc > 4) g_filter = argv[4];
  setvbuf(stdout, NULL, _IONBF, 0);
  cudaStream_t s; CK(cudaStreamCreate(&s));
  Ring R;
  std::vector<float> h(4 * (size_t)n), ha(n);
  srand(1);
  const float sc[4] = {4.f, 5.f, 3.14159f, 8.f};
  for (size_t i = 0; i < 4 * (size_t)n; ++i) h[i] = (2.f * rand() / RAND_MAX - 1.f) * sc[i & 3];
  for (size_t i = 0; i < n; ++i) ha[i] = 2.f * rand() / RAND_MAX - 1.f;
  for (int j = 0; j < ring; ++j) {
    float *a, *b, *c, *d; uint8_t* e;
    CK(cudaMalloc(&a, 16 * (size_t)n)); CK(cudaMalloc(&b, 16 * (size_t)n)); CK(cudaMalloc(&c, 4 * (size_t)n)); CK(cudaMalloc(&d, 4 * (size_t)n)); CK(cudaMalloc(&e, n));
    CK(cudaMemcpy(a, h.data(), 16 * (size_t)n, cudaMemcpyHostToDevice)); CK(cudaMemcpy(c, ha.data(), 4 * (size_t)n, cudaMemcpyHostToDevice));
    R.in.push_back(a); R.out.push_back(b); R.act.push_back(c); R.rew.push_back(d); R.done.push_back(e);
  }
  printf("n=%u ring=%d K=%d\n", n, ring, K);
  run_stream<8, true>("stream minb8 pdl", R, n, K, s);
  run_compute<4, 4, true>("compute-only scalar fr4 minb4 sincos/sub-step", R, n, K, s);
  run_compute<4, 4, false>("compute-only scalar fr4 minb4 angle-addition", R, n, K, s);
  run_compute2<4, 4, true>("compute-only packed fr4 minb4 sincos/sub-step", R, n, K, s);
  run_compute2<4, 4, false>("compute-only packed fr4 minb4 angle-addition", R, n, K, s);
  run_tma<4>("TMA packed fr4 (shipped)", R, n, K, s);
  run_tma<4>("TMA packed fr4 slots<=8", R, n, K, s, 8);
  run_tma<0>("TMA packed fr-runtime", R, n, K, s);
  run_tma<1>("TMA packed fr1", R, n, K, s);
  return 0;
}
