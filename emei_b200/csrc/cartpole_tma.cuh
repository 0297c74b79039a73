// float32 cart-pole / analytic inverted-pendulum step, TMA-staged.
//
// At BASELINE configs[1] (2^20 envs, 41 B/env-step) one SM's share of a step is 7 085 envs = 142 KB of inputs:
// it FITS in the SM's 227 KB of shared memory.  So the kernel is one persistent CTA per SM (1024 threads = four
// consumer groups of 256) that requests, at t = 0, one 1-D bulk copy (cp.async.bulk, the TMA engine) per 512-env
// chunk for as many chunks as the ring holds -- every input byte of the step is in flight within the first
// microsecond, HBM streams at full rate from the start, and no thread spends instructions or LDGSTS slots on
// address generation -- while the groups take their chunks as the mbarriers complete, advance TWO envs per thread
// with the packed f32x2 arithmetic of f32math.cuh and store the results.  Larger batches recycle the ring: every
// group owns a quarter of the slots and refills its own (empty mbarriers), which streams 2^26 envs at 0.97 of the
// measured HBM peak.  For a step this short (~10 us at 2^20) the ramp matters as much as the steady state:
// per-thread prefetch rings issue a slot's refill only after that slot's math, which left HBM idle during
// the compute of the first chunks (ncu: dram 18 %, issue 55 %, profiles/r01_kbench_cartpole_variants.txt).
// Batches below kSmallBatch take a plain one-env-per-thread kernel (launch latency is their whole cost).
//
// Chunk c = envs [512 c, 512 c + 512): thread t of a group owns envs 512 c + t and 512 c + 256 + t.
#pragma once
#include <type_traits>
#include "cartpole_f32.cuh"

namespace emei {

constexpr int kTmaGroups = 4;                                 // consumer groups of kBlock threads per CTA
constexpr int kTmaThreads = kTmaGroups * kBlock;              // 1024 threads: 8 warps per scheduler at <= 64 registers
constexpr uint32_t kChunk = 2 * kBlock;                       // envs per chunk
constexpr int kTmaSmemBudget = 208 * 1024;                    // ring bytes (of 227 KB per SM)
constexpr int kTmaMaxSlots = 32;
// The first ring-full (up to 16 chunks x 2 bulk copies, ~1 000 instructions of one thread) is requested by the first
// thread of the LAST consumer group: with 13.8 chunks per SM the groups own 4, 4, 3, 3 (or 4, 3, 3, 3) chunks, so the
// last group's warps have a chunk's worth of slack while group 0's are on the critical path of the CTA.
constexpr int kTmaProducerGroup = kTmaGroups - 1;

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive_u32(uint32_t bar) { asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory"); }
__device__ __forceinline__ void mbar_wait_u32(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  do {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
  } while (ok == 0);
}
__device__ __forceinline__ float4 lds128(uint32_t addr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
  return v;
}
template <class T>
__device__ __forceinline__ T lds_as(uint32_t addr) {  // one element of the staged action chunk
  if constexpr (sizeof(T) == 1) {
    uint32_t v;
    asm volatile("ld.shared.u8 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return static_cast<T>(v);
  } else if constexpr (sizeof(T) == 4) {
    uint32_t v;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    T r;
    memcpy(&r, &v, 4);
    return r;
  } else {
    unsigned long long v;
    asm volatile("ld.shared.b64 %0, [%1];" : "=l"(v) : "r"(addr) : "memory");
    T r;
    memcpy(&r, &v, 8);
    return r;
  }
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}
// 1-D bulk copy global -> shared (TMA engine); completes `bytes` on the mbarrier.  16-byte aligned, size % 16 == 0.
__device__ __forceinline__ void tma_load_1d(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
               "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// kTmaGroups consumer groups of kBlock threads per CTA, one CTA per SM.
// Chunk c = envs [512 c, 512 c + 512); warp w of a group owns the 64 contiguous envs 512 c + 64 w ..: lane l takes
// 64 w + l and 64 w + 32 + l.
template <bool IP, int AK, int FR, bool HAS_OBS>
__global__ void __launch_bounds__(kTmaThreads, 1)
    cartpole_step_f32_tma_kernel(const float4* state_in, float4* state_out, float4* obs_out,
                                 const void* __restrict__ action, float* __restrict__ reward, uint8_t* __restrict__ done,
                                 double* stats, uint32_t n, int n_slots, int flags, const CartPoleF32Consts k) {
  // flags: bit 0 = the action array is 16-byte aligned (staged by TMA); bit 1 = prefetch the first ring-full into L2 before
  // griddepcontrol.wait; bits 16.. = how many chunks of it to prefetch (0: all)
  const int action_via_tma = flags & 1;
  constexpr uint32_t producer_tid = kTmaProducerGroup * kBlock;
  using f32::f2;
  using ActT = typename ActionStorage<AK>::type;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  // layout: [n_slots] state chunks (8 KB each) | [n_slots] action chunks | full[n_slots] | empty[n_slots] | reduction scratch
  float4* s_state = reinterpret_cast<float4*>(smem_raw);
  ActT* s_act = reinterpret_cast<ActT*>(smem_raw + static_cast<size_t>(n_slots) * kChunk * sizeof(float4));
  uint64_t* full = reinterpret_cast<uint64_t*>(reinterpret_cast<unsigned char*>(s_act) + static_cast<size_t>(n_slots) * kChunk * sizeof(ActT));
  uint64_t* empty = full + n_slots;
  const uint32_t tid = threadIdx.x;
  const uint32_t n_chunks = (n + kChunk - 1) / kChunk;
  // this CTA's chunks: blockIdx.x, blockIdx.x + gridDim.x, ...   (local index j)
  const uint32_t my_chunks = blockIdx.x < n_chunks ? (n_chunks - blockIdx.x + gridDim.x - 1) / gridDim.x : 0;
  const ActT* act = static_cast<const ActT*>(action);

  if (tid == 0) {
    for (int s = 0; s < n_slots; ++s) {
      mbar_init(&full[s], 1);                    // one arrive.expect_tx by the producer; the bytes complete it
      mbar_init(&empty[s], kBlock / 32);         // one arrive per consumer warp of the group that drained the slot
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  pdl_trigger();  // let the next step kernel of the rollout be staged behind this one
  // L2 prefetch of this CTA's first ring-full BEFORE the grid dependency resolves.  A prefetch returns nothing to the SM and
  // L2 is the device's point of coherence, so it is architecturally invisible: if the previous kernel is still writing these
  // lines (the same batch stepped again) they are in L2 already and the prefetch is a hit; if they are cold (another batch,
  // a state set from the host) the DRAM reads start while the previous grid's stragglers drain -- the 1-2 us between
  // griddepcontrol.wait and the first chunk's landing (profiles/r02_c2_chunk_pipeline_trace.txt) shrink to an L2 hit.
  if ((flags & 2) && tid == kBlock) {  // a thread that neither initialises barriers nor issues the loads
    uint32_t first = my_chunks < static_cast<uint32_t>(n_slots) ? my_chunks : static_cast<uint32_t>(n_slots);
    const uint32_t depth = static_cast<uint32_t>((flags >> 16) & 0xff);
    if (depth != 0 && depth < first) first = depth;
    for (uint32_t j = 0; j < first; ++j) {
      const uint32_t base = (blockIdx.x + j * gridDim.x) * kChunk;
      const uint32_t cnt = n - base < kChunk ? n - base : kChunk;
      asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(state_in + base), "r"(cnt * 16u) : "memory");
      if (action_via_tma && cnt == kChunk)
        asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(act + base), "r"(kChunk * static_cast<uint32_t>(sizeof(ActT))) : "memory");
    }
  }
  __syncthreads();
  pdl_wait();     // the previous kernel in the stream (the step that wrote state_in) has completed

  float r_acc = 0.0f;
  unsigned d_cnt = 0;
  {
    // ------------------------------------------------------------------ four independent pipelines
    // Group g (256 threads) owns the CTA's local chunks g, g+4, ... and a private ring of n_slots / 4 slots.
    // The first thread of group kTmaProducerGroup requests the first ring-full of every group at t = 0; after that (batches whose share of an SM
    // exceeds the ring) thread 0 OF EACH GROUP refills, at the top of iteration m, the slot the group
    // read in iteration m - 1 -- by then all 8 warps of the group have long finished reading it, so the wait on
    // the empty barrier never blocks, and the request runs n_slots / 4 - 1 iterations ahead of its use.
    // (One producer thread for the whole CTA refilled only when ITS group came round and coupled the four groups
    // through the empty barriers: 96 G env-steps/s at 2^24 envs against 108 G at 2^20, where nothing is recycled.)
    // Everything that does not change from chunk to chunk is computed here once; the loop carries one running
    // env index and the slot / phase pair.  The body is compiled twice: FULL (every chunk but possibly the last
    // of the batch: no per-lane predicates) and the ragged tail.
    const uint32_t g = tid / kBlock, t = tid % kBlock;
    const uint32_t flip = ip_flip(IP, k.variant);
    const uint32_t spg = static_cast<uint32_t>(n_slots) / kTmaGroups;                      // slots per group (n_slots % kTmaGroups == 0)
    const uint32_t my_g = my_chunks > g ? (my_chunks - g + kTmaGroups - 1) / kTmaGroups : 0;  // this group's chunks
    const bool recycling = my_g > spg;  // group-uniform: the ring is reused
    const uint32_t slot0 = g * spg;
    auto issue = [&](uint32_t gg, uint32_t m, uint32_t sl) {  // chunk m of group gg into slot sl
      const uint32_t c = blockIdx.x + (gg + m * kTmaGroups) * gridDim.x;
      const uint32_t base = c * kChunk;
      const uint32_t cnt = n - base < kChunk ? n - base : kChunk;
      const bool act_tma = action_via_tma && cnt == kChunk;  // partial tail: consumers read their actions directly
      const uint32_t sbytes = cnt * static_cast<uint32_t>(sizeof(float4));
      const uint32_t abytes = act_tma ? kChunk * static_cast<uint32_t>(sizeof(ActT)) : 0u;
      mbar_expect_tx(&full[sl], sbytes + abytes);
      tma_load_1d(s_state + static_cast<size_t>(sl) * kChunk, state_in + base, sbytes, &full[sl]);
      if (act_tma) tma_load_1d(s_act + static_cast<size_t>(sl) * kChunk, act + base, abytes, &full[sl]);
    };
    // The first ring-full is requested by ONE thread in consumption order (local chunks 0, 1, 2, ...): bulk copies
    // issued together share the bandwidth, so four producers starting at once made every chunk of the ring
    // complete late (10.8 us per step at 2^20 envs instead of 9.7); issued in order, chunk 0 lands first.
    if (tid == producer_tid) {
      const uint32_t first = my_chunks < static_cast<uint32_t>(n_slots) ? my_chunks : static_cast<uint32_t>(n_slots);
      for (uint32_t j = 0; j < first; ++j) issue(j % kTmaGroups, j / kTmaGroups, (j % kTmaGroups) * spg + j / kTmaGroups);
    }
    // 32-bit shared-window addresses (the generic-pointer forms re-derive the window base per chunk)
    const uint32_t tw = (t >> 5) * 64u + (t & 31u);  // env A of this thread within a chunk; env B = tw + 32
    const uint32_t state_u32 = smem_u32(s_state) + tw * 16u, full_u32 = smem_u32(full), empty_u32 = smem_u32(empty);
    const uint32_t act_u32 = smem_u32(s_act) + tw * static_cast<uint32_t>(sizeof(ActT));
    const uint32_t i_step = kTmaGroups * gridDim.x * kChunk;
    uint32_t i = (blockIdx.x + g * gridDim.x) * kChunk + tw;  // env A of this thread in the current chunk; env B = i + 32
    uint32_t slot = slot0, phase = 0u;                      // slot / parity of the chunk consumed now
    uint32_t prev_slot = slot0, prev_phase = 0u;            // ... and of the previous iteration (the one to refill)

    auto body = [&](auto full_tag, auto recycle_tag) {
      constexpr bool FULL = decltype(full_tag)::value;
      constexpr bool RECYCLE = decltype(recycle_tag)::value;
      constexpr uint32_t kB = 32u;  // env B = env A + 32
      const bool live_a = FULL || i < n, live_b = FULL || i + kB < n;
      const bool act_tma = FULL && action_via_tma;  // partial tail: consumers read their actions directly
      mbar_wait_u32(full_u32 + slot * 8u, phase);
      const uint32_t sl = state_u32 + slot * (kChunk * 16u);
      float4 ya = live_a ? lds128(sl) : make_float4(0.f, 0.f, 0.f, 0.f);
      float4 yb = live_b ? lds128(sl + kB * 16u) : make_float4(0.f, 0.f, 0.f, 0.f);
      float aa = 0.f, ab = 0.f;
      if (act_tma) {
        const uint32_t al = act_u32 + slot * (kChunk * static_cast<uint32_t>(sizeof(ActT)));
        aa = static_cast<float>(lds_as<ActT>(al));
        ab = static_cast<float>(lds_as<ActT>(al + kB * static_cast<uint32_t>(sizeof(ActT))));
      } else {
        if (live_a) aa = static_cast<float>(__ldg(act + i));
        if (live_b) ab = static_cast<float>(__ldg(act + i + kB));
      }
      if constexpr (RECYCLE) {
        __syncwarp();
        if ((t & 31u) == 0) mbar_arrive_u32(empty_u32 + slot * 8u);  // this warp's reads of the slot are done
      }

      const float fa = action_to_f_mt<IP, AK>(aa, k), fb = action_to_f_mt<IP, AK>(ab, k);
      // ---- packed integration: [x, x_dot, theta, theta_dot] (cart-pole) / [x, theta, v, omega] (IP)
      f2 X = f32::f2_pack(ya.x, yb.x), V, TH, W = f32::f2_pack(ya.w, yb.w);
      if constexpr (!IP) {
        V = f32::f2_pack(ya.y, yb.y);
        TH = f32::f2_pack(ya.z, yb.z);
      } else {
        TH = f32::f2_pack(ya.y, yb.y);
        V = f32::f2_pack(ya.z, yb.z);
      }
      const f2 nf = f32::f2_pack(-fa, -fb);
      const float th0a = fabsf(IP ? ya.y : ya.z), th0b = fabsf(IP ? yb.y : yb.z);
      f32::LaneMax<f2> dmax;
      const f2 C = f32::cartpole_integrate<f2, FR>(X, V, TH, W, nf, flip, k.k, k.freq_rate, dmax);
      float4 na, nb;
      {
        float t0, t1;
        f32::f2_unpack(X, na.x, nb.x);
        f32::f2_unpack(W, na.w, nb.w);
        f32::f2_unpack(V, t0, t1);
        if constexpr (!IP) { na.y = t0; nb.y = t1; } else { na.z = t0; nb.z = t1; }
        f32::f2_unpack(TH, t0, t1);
        if constexpr (!IP) { na.z = t0; nb.z = t1; } else { na.y = t0; nb.y = t1; }
      }
      // cos of the reward angle from the integrator (IP: undo the flip of the hanging models)
      float ca, cb;
      f32::f2_unpack(C, ca, cb);
      if constexpr (IP) {
        ca = f32::u2f(f32::f2u(ca) ^ flip);
        cb = f32::u2f(f32::f2u(cb) ^ flip);
      }
      // the integrator's guard (f32math.cuh): otherwise (Inf, absurd angles or rates) redo that env from its
      // stored state with the libm path.  Cold: float32 theta is meaningless there.
      const bool ok_a = th0a <= f32::kSinCosSaneMax && dmax.a <= f32::kDeltaMax;
      const bool ok_b = th0b <= f32::kSinCosSaneMax && dmax.b <= f32::kDeltaMax;
      if (!(ok_a && ok_b)) {
        if (!ok_a && live_a) {
          na = integrate_libm<IP, FR>(state_in[i], fa, flip, k.k, k.freq_rate, &ca);
          if constexpr (IP) ca = f32::u2f(f32::f2u(ca) ^ flip);
        }
        if (!ok_b && live_b) {
          nb = integrate_libm<IP, FR>(state_in[i + kB], fb, flip, k.k, k.freq_rate, &cb);
          if constexpr (IP) cb = f32::u2f(f32::f2u(cb) ^ flip);
        }
      }
      float rew_a, rew_b;
      bool nd_a, nd_b;
      float4 oa, ob;
      cartpole_outcome<IP>(na, ca, k, rew_a, nd_a, oa);
      cartpole_outcome<IP>(nb, cb, k, rew_b, nd_b, ob);
      float4* so = state_out + i;
      float* ro = reward + i;
      uint8_t* dn = done + i;
      if (live_a) {
        so[0] = na;
        if constexpr (HAS_OBS) obs_out[i] = oa;
        ro[0] = rew_a;
        dn[0] = nd_a ? 0 : 1;
        r_acc += rew_a;
        d_cnt += nd_a ? 0u : 1u;
      }
      if (live_b) {
        so[kB] = nb;
        if constexpr (HAS_OBS) obs_out[i + kB] = ob;
        ro[kB] = rew_b;
        dn[kB] = nd_b ? 0 : 1;
        r_acc += rew_b;
        d_cnt += nd_b ? 0u : 1u;
      }
    };

    if (!recycling) {
      // the whole share of this group is in the ring (BASELINE configs[1]: 2^20 envs): no refill logic, no empty
      // barriers, one slot per chunk -- the loop carries the env index and the slot only
      for (uint32_t m = 0; m < my_g; ++m) {
        if (i - tw + kChunk <= n)
          body(std::true_type{}, std::false_type{});
        else
          body(std::false_type{}, std::false_type{});
        i += i_step;
        ++slot;
      }
    } else {
      for (uint32_t m = 0; m < my_g; ++m) {
        if (t == 0 && m >= 1 && m - 1 + spg < my_g) {  // refill the slot read one iteration ago
          mbar_wait(&empty[prev_slot], prev_phase);
          issue(g, m - 1 + spg, prev_slot);
        }
        if (i - tw + kChunk <= n)
          body(std::true_type{}, std::true_type{});
        else
          body(std::false_type{}, std::true_type{});
        i += i_step;
        prev_slot = slot;
        prev_phase = phase;
        if (++slot == slot0 + spg) {
          slot = slot0;
          phase ^= 1u;
        }
      }
    }
  }
  // ---- statistics: warp shuffles -> shared -> one atomic pair per CTA
  if (stats != nullptr) {  // uniform across the grid
    double* s_r = reinterpret_cast<double*>(empty + n_slots);
    unsigned* s_d = reinterpret_cast<unsigned*>(s_r + kTmaThreads / 32);
    const int lane = tid & 31, warp = tid >> 5;
    const double r = warp_sum(static_cast<double>(r_acc));
    const unsigned d = __reduce_add_sync(0xffffffffu, d_cnt);
    if (lane == 0) {
      s_r[warp] = r;
      s_d[warp] = d;
    }
    __syncthreads();
    if (warp == 0) {
      double rr = lane < kTmaThreads / 32 ? s_r[lane] : 0.0;
      unsigned dd = lane < kTmaThreads / 32 ? s_d[lane] : 0u;
      rr = warp_sum(rr);
      dd = __reduce_add_sync(0xffffffffu, dd);
      if (lane == 0) {
        atomicAdd(&stats[0], rr);
        atomicAdd(&stats[1], static_cast<double>(dd));  // exact: counts << 2^53
      }
    }
  }
}

// Small batches (n < kSmallBatch; BASELINE configs[0] is 4096 envs): launch latency is the whole cost, so the
// shortest dependency chain wins -- one env per thread, direct 128-bit loads, 128-thread CTAs spread over as many
// SMs as the batch allows, no staging.  Scalar form of the same arithmetic (bit-identical to the packed kernel).
constexpr int kSmallBlock = 128;
constexpr int64_t kSmallBatch = 8192;

template <bool IP, int AK, int FR, bool HAS_OBS>
__global__ void __launch_bounds__(kSmallBlock)
    cartpole_step_f32_small_kernel(const float4* __restrict__ state_in, float4* __restrict__ state_out,
                                   float4* __restrict__ obs_out, const void* __restrict__ action,
                                   float* __restrict__ reward, uint8_t* __restrict__ done, double* stats, uint32_t n,
                                   const CartPoleF32Consts k) {
  const uint32_t i = blockIdx.x * kSmallBlock + threadIdx.x;
  float rew = 0.f;
  bool notdone = true;
  pdl_trigger();
  // L2 prefetch of this thread's inputs before the grid dependency resolves (architecturally invisible: see the TMA kernel):
  // the loads after griddepcontrol.wait then hit L2 instead of paying the DRAM latency on the critical path of a 1.7 us launch
  if (i < n) {
    asm volatile("prefetch.global.L2 [%0];" ::"l"(state_in + i));
    if ((threadIdx.x & 15u) == 0)
      asm volatile("prefetch.global.L2 [%0];" ::"l"(static_cast<const char*>(action) + static_cast<size_t>(i) * sizeof(typename ActionStorage<AK>::type)));
  }
  pdl_wait();
  if (i < n) {
    float4 y = state_in[i];
    const float f_mt = action_to_f_mt<IP, AK>(load_action_f32<AK>(action, i), k);
    const uint32_t flip = ip_flip(IP, k.variant);
    float4 obs;
    cartpole_step_one<IP, FR>(y, f_mt, flip, k, rew, notdone, obs);
    state_out[i] = y;
    if constexpr (HAS_OBS) obs_out[i] = obs;
    reward[i] = rew;
    done[i] = notdone ? 0 : 1;
  }
  block_stats_accumulate_counts(stats, static_cast<double>(rew), notdone ? 0u : 1u);
}

// slots, dynamic shared memory bytes for an action element size
inline void tma_ring_shape(int action_bytes, int64_t chunks_per_cta, int* n_slots, size_t* smem_bytes) {
  const int slot_bytes = static_cast<int>(kChunk) * (16 + action_bytes);
  int s = kTmaSmemBudget / slot_bytes;
  if (s > kTmaMaxSlots) s = kTmaMaxSlots;
  if (s > chunks_per_cta) s = static_cast<int>(chunks_per_cta);
  s = (s + kTmaGroups - 1) / kTmaGroups * kTmaGroups;  // every consumer group owns n_slots / kTmaGroups slots
  while (s * slot_bytes > kTmaSmemBudget) s -= kTmaGroups;
  if (s < kTmaGroups) s = kTmaGroups;
  *n_slots = s;
  *smem_bytes = static_cast<size_t>(s) * slot_bytes + 2 * s * sizeof(uint64_t) + (kTmaThreads / 32) * (sizeof(double) + sizeof(unsigned)) + 16;
}

// opt in to > 48 KB of dynamic shared memory: the attribute is PER DEVICE, so it is set once per (kernel
// instantiation, device); a failure surfaces as the launch status of the call that needed it
template <auto Kernel>
inline cudaError_t tma_allow_smem() {
  static bool done[kMaxDevices] = {};
  const int d = current_device();
  if (!done[d]) {
    const cudaError_t e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
    done[d] = true;
  }
  return cudaSuccess;
}

template <bool IP, int FR>
inline void launch_cartpole_f32_tma(int ak, cudaStream_t s, const float* state_in, float* state_out, float* obs_out,
                                    const void* action, int action_bytes, float* reward, uint8_t* done, double* stats,
                                    int64_t n, const CartPoleF32Consts& k) {
  if (n < kSmallBatch) {
    const float4* in4 = reinterpret_cast<const float4*>(state_in);
    float4* out4 = reinterpret_cast<float4*>(state_out);
    float4* obs4 = reinterpret_cast<float4*>(obs_out);
    const int grid = grid_for(n, kSmallBlock);
    switch (ak) {
#define EMEI_AK(A)                                                                                                     \
  case A:                                                                                                              \
    if (obs4 != nullptr)                                                                                               \
      launch_pdl(cartpole_step_f32_small_kernel<IP, A, FR, true>, grid, kSmallBlock, s, in4, out4, obs4, action, reward, \
                 done, stats, static_cast<uint32_t>(n), k);                                                            \
    else                                                                                                               \
      launch_pdl(cartpole_step_f32_small_kernel<IP, A, FR, false>, grid, kSmallBlock, s, in4, out4, obs4, action, reward, \
                 done, stats, static_cast<uint32_t>(n), k);                                                            \
    break;
      EMEI_AK(EMEI_ACTION_DISCRETE_U8)
      EMEI_AK(EMEI_ACTION_DISCRETE_I32)
      EMEI_AK(EMEI_ACTION_DISCRETE_I64)
      EMEI_AK(EMEI_ACTION_CONTINUOUS_F32)
      EMEI_AK(EMEI_ACTION_CONTINUOUS_F64)
#undef EMEI_AK
    }
    return;
  }
  for (int64_t off = 0; off < n; off += kCartPoleMaxLaunch) {
    const int64_t m = n - off < kCartPoleMaxLaunch ? n - off : kCartPoleMaxLaunch;
    const int64_t chunks = (m + kChunk - 1) / kChunk;
    const int n_sm = sm_count();
    const int grid = static_cast<int>(chunks < n_sm ? chunks : n_sm);
    int n_slots;
    size_t smem;
    tma_ring_shape(action_bytes, (chunks + grid - 1) / grid, &n_slots, &smem);
    const float4* in4 = reinterpret_cast<const float4*>(state_in) + off;
    float4* out4 = reinterpret_cast<float4*>(state_out) + off;
    float4* obs4 = obs_out ? reinterpret_cast<float4*>(obs_out) + off : nullptr;
    const void* act = static_cast<const char*>(action) + off * action_bytes;
    // bit 1 + bits 16..: L2 prefetch of the first `depth` chunks before the grid dependency resolves.  Measured (kbench,
    // profiles/r02_kbench_c2_prefetch.txt): at 2^20 envs no prefetch 9.42 us, depth 1: 9.01, 3: 8.46, 4: 8.54, 6: 8.72, 8: 8.89,
    // the whole ring-full: 9.85 (the early CTAs' reads then compete with the previous grid's stragglers); at 2^22 envs
    // depth 6-8 is best (32.2 -> 29.9 us), at 2^18 depth 3 (4.70 -> 3.77 us).
    const int64_t per_cta = (chunks + grid - 1) / grid;
    const int depth = static_cast<int>(per_cta / 5 + 1 < 3 ? 3 : (per_cta / 5 + 1 > 8 ? 8 : per_cta / 5 + 1));
    const int act_tma = ((reinterpret_cast<uintptr_t>(act) & 15u) == 0 ? 1 : 0) | 2 | (depth << 16);
    switch (ak) {
#define EMEI_AK(A)                                                                                                  \
  case A:                                                                                                           \
    if (obs4 != nullptr) {                                                                                          \
      if (tma_allow_smem<cartpole_step_f32_tma_kernel<IP, A, FR, true>>() == cudaSuccess)                             \
        launch_pdl(cartpole_step_f32_tma_kernel<IP, A, FR, true>, grid, kTmaThreads, smem, s, in4, out4, obs4, act, \
                   reward + off, done + off, stats, static_cast<uint32_t>(m), n_slots, act_tma, k);                 \
    } else {                                                                                                        \
      if (tma_allow_smem<cartpole_step_f32_tma_kernel<IP, A, FR, false>>() == cudaSuccess)                            \
        launch_pdl(cartpole_step_f32_tma_kernel<IP, A, FR, false>, grid, kTmaThreads, smem, s, in4, out4, obs4, act, \
                   reward + off, done + off, stats, static_cast<uint32_t>(m), n_slots, act_tma, k);                 \
    }                                                                                                               \
    break;
      EMEI_AK(EMEI_ACTION_DISCRETE_U8)
      EMEI_AK(EMEI_ACTION_DISCRETE_I32)
      EMEI_AK(EMEI_ACTION_DISCRETE_I64)
      EMEI_AK(EMEI_ACTION_CONTINUOUS_F32)
      EMEI_AK(EMEI_ACTION_CONTINUOUS_F64)
#undef EMEI_AK
    }
  }
}

// R = float.  A template, so that the float64 translation unit, which sees this header too, instantiates none of the kernels.
template <typename R>
inline void cartpole_step_f32_tma_dispatch(const R* state_in, R* state_out, R* obs_out, const void* action, R* reward,
                                           uint8_t* done, double* stats, int64_t n, const emei_cartpole_params& p,
                                           cudaStream_t s) {
  const CartPoleF32Consts k = make_cartpole_f32_consts(p);
  const bool ip = p.variant > EMEI_CARTPOLE_SWINGUP;
  const int ab = action_kind_bytes(p.action_kind);
#define EMEI_GO(IPV, FRV) \
  launch_cartpole_f32_tma<IPV, FRV>(p.action_kind, s, state_in, state_out, obs_out, action, ab, reward, done, stats, n, k)
  if (!ip) {
    if (p.freq_rate == 1) EMEI_GO(false, 1);
    else if (p.freq_rate == 4) EMEI_GO(false, 4);
    else EMEI_GO(false, 0);
  } else {
    if (p.freq_rate == 1) EMEI_GO(true, 1);
    else if (p.freq_rate == 4) EMEI_GO(true, 4);
    else EMEI_GO(true, 0);
  }
#undef EMEI_GO
}

}  // namespace emei
