// device_util.cuh -- tunables and small device helpers (streaming loads/stores, mbarrier, TMA).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

#include "ekf_math.cuh"

namespace pkf_dev {
using namespace pkf;

// tunables (overridable with -D for experiments; the defaults are what ships)
#ifndef PKF_TMA_STEPS
#define PKF_TMA_STEPS 4
#endif
#ifndef PKF_TMA_STAGES
#define PKF_TMA_STAGES 2
#endif
#ifndef PKF_MIN_CTAS
#define PKF_MIN_CTAS 6
#endif
constexpr int kThreads = 128;                  // filters per CTA (4 warps)
constexpr int kMinCtasPerSm = PKF_MIN_CTAS;    // 6 CTAs/SM (24 warps) <=> <=80 registers per thread
constexpr int kTmaSteps = PKF_TMA_STEPS;       // TC: timesteps per TMA tile
constexpr int kTmaStages = PKF_TMA_STAGES;     // ring depth
constexpr int kChannels = 9;
// packed (two filters per thread) variant
#ifndef PKF_TMA2_STEPS
#define PKF_TMA2_STEPS 4
#endif
#ifndef PKF_TMA2_STAGES
#define PKF_TMA2_STAGES 2
#endif
#ifndef PKF_THREADS2
#define PKF_THREADS2 128          // 4 warps own a 256-filter tile (64 threads / 128 filters measured 1 % slower, burst and sustained)
#endif
#ifndef PKF_MIN_CTAS2
#define PKF_MIN_CTAS2 (384 / PKF_THREADS2)     // 12 warps per SM: <= 168 registers per thread, 3 x 73.7 KB of tiles
#endif
constexpr int kThreads2 = PKF_THREADS2;        // threads per CTA of the packed kernel
constexpr int kTile2 = 2 * kThreads2;          // filters per CTA (two per thread); TMA box width, <= 256
constexpr int kTma2Steps = PKF_TMA2_STEPS;
constexpr int kTma2Stages = PKF_TMA2_STAGES;
// PKF_FAST_TILE: the packed kernel runs complete tiles without a reflected-Wahba sample as one basic block
#ifndef PKF_FAST_TILE
#define PKF_FAST_TILE 1
#endif
// PKF_L2_PREFETCH: tiles of the packed kernel's ring are requested into L2 this many tiles beyond the ring's own depth
// (the ring holds the tile being processed and the next one; DRAM latency under load is about one tile's compute time)
#ifndef PKF_L2_PREFETCH
#define PKF_L2_PREFETCH 0
#endif
#ifndef PKF_AUTO_PACKED
#define PKF_AUTO_PACKED 1
#endif
constexpr bool kAutoPrefersPacked = PKF_AUTO_PACKED != 0;   // whether POSEKF_STAGE_AUTO picks the packed kernel

// ---------------------------------------------------------------------------------------------
// small device helpers
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ float ldg_stream(const float* p) {
  // streamed once: read-only path, do not keep in L1
  float v;
  asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(v) : "l"(p));
  return v;
}
__device__ __forceinline__ f32x2 ldg2_stream(const float* p) {
  float a, b;
  asm volatile("ld.global.nc.L1::no_allocate.v2.f32 {%0, %1}, [%2];" : "=f"(a), "=f"(b) : "l"(p));
  return f32x2(a, b);
}
__device__ __forceinline__ void stg_stream(float* p, float v) {
  asm volatile("st.global.cs.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}
__device__ __forceinline__ void stg_stream4(float4* p, float a, float b, float c, float d) {
  asm volatile("st.global.cs.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(p), "f"(a), "f"(b), "f"(c), "f"(d) : "memory");
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "WAIT_%=:\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
      "@p bra DONE_%=;\n"
      "bra WAIT_%=;\n"
      "DONE_%=:\n"
      "}\n" ::"r"(smem_u32(bar)),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];" ::"r"(
          smem_u32(dst)),
      "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}

// TMA prefetch of a tile into L2 only (no shared memory, no barrier): used one tile further ahead than the ring holds
__device__ __forceinline__ void tma_prefetch_l2_3d(const CUtensorMap* map, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.prefetch.tensor.3d.L2.global.tile [%0, {%1, %2, %3}];" ::"l"(map), "r"(c0), "r"(c1), "r"(c2) : "memory");
}

__device__ __forceinline__ f32x2 ld2(const float* p) {
  const float2 v = *reinterpret_cast<const float2*>(p);
  return f32x2(v.x, v.y);
}
__device__ __forceinline__ void st2(float* p, const f32x2& v) { *reinterpret_cast<float2*>(p) = make_float2(v.x, v.y); }

}  // namespace pkf_dev
