// Shared device-side plumbing of the tcgen05 kernels (gemm_tc.cu, gemm_ln.cu): mbarrier / TMA / UMMA / TMEM wrappers
// around the PTX, the K-major 128B-swizzle descriptors and the MUFU-based activations.  sm_100a only.
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <stdint.h>

#include "kernels.cuh"

namespace ds {

static constexpr int BM = 128;
static constexpr int BK = 64;
static constexpr int A_BYTES = BM * BK * 2;           // 16 KB
static constexpr uint64_t WAIT_TIMEOUT_CYCLES = 4000000000ull;   // ~2 s: a protocol bug traps instead of hanging

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a mis-programmed pipeline traps (the launch fails with an error) instead of hanging the GPU.
// SLEEP_NS > 0 (the single-lane TMA-producer / MMA-issuer roles, which are far off the critical path of an
// epilogue-bound kernel): back off between polls so that the spinning lane does not take issue slots from the
// epilogue warps of its SM sub-partition.
template <int SLEEP_NS = 0>
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity, int* err_flag, int code) {
  if (mbar_try_wait(bar, parity)) return;
  const unsigned long long t0 = clock64();
  unsigned int spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if constexpr (SLEEP_NS > 0) __nanosleep(SLEEP_NS);
    if ((++spins & 0x3FFu) == 0 && clock64() - t0 > WAIT_TIMEOUT_CYCLES) {     // clock read once per 1024 polls
      if (err_flag) atomicExch(err_flag, code);
      __threadfence_system();
      __trap();
    }
  }
}

__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ uint32_t cluster_nctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_nctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync_all() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}

__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// K-major, 128B-swizzled operand tile: rows of 128 bytes, 8-row swizzle atoms 1024 bytes apart.
__host__ __device__ constexpr uint64_t umma_desc_hi_sw128() {
  return ((uint64_t)1 << 16)                      // leading byte offset (unused for swizzled K-major)
         | ((uint64_t)(1024 >> 4) << 32)          // stride byte offset between 8-row groups
         | ((uint64_t)1 << 46)                    // descriptor version (Blackwell)
         | ((uint64_t)2 << 61);                   // SWIZZLE_128B
}
__device__ __forceinline__ uint64_t umma_desc(uint32_t smem_addr, uint64_t hi) {
  return hi | (uint64_t)((smem_addr & 0x3FFFFu) >> 4);   // start address in 16-byte units
}
// launch with the optional programmatic-stream-serialization attribute
template <typename... KArgs, typename... Args>
inline int tc_launch(void (*kern)(KArgs...), int grid, int threads, size_t smem, cudaStream_t s, bool pdl, Args&&... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(grid);
  cfg.blockDim = dim3(threads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  if (pdl) {
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
  }
  return (int)cudaLaunchKernelEx(&cfg, kern, KArgs(args)...);
}
// ---- warp-uniform issue --------------------------------------------------------------------------------------------
// The single-thread roles (TMA producer, MMA issuer) run their loops with the WHOLE warp active: control flow is
// warp-uniform, descriptors / barrier addresses / loop counters live in uniform registers, and one elected lane
// executes each tcgen05 / TMA instruction.  Inside an `if (lane == 0)` region the compiler cannot prove that a single
// thread is active and wraps every UTCHMMA / UTCBAR / UTMALDG in an ELECT + 5 x R2UR.BROADCAST + BRA.U.ANY waterfall
// (19 SASS instructions per MMA on the issuing thread; 4 MMAs + commit back to back in the uniform form).  The warp
// index must be taken through uniform_warp_idx() for this.  elect.sync picks the same lane for the same member mask
// every time, so the commits track that lane's MMAs.
__device__ __forceinline__ int uniform_warp_idx() { return __shfl_sync(0xffffffffu, int(threadIdx.x >> 5), 0); }

// D(tmem, fp32) (+)= A(smem, bf16) * B(smem, bf16)^T, M = 128, N from the instruction descriptor, K = 16
__device__ __forceinline__ void umma_issue_elect(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                 uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@e tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// completion of the MMAs issued so far -> one arrival on `bar`
__device__ __forceinline__ void umma_arrive_elect(uint32_t bar) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t}" ::"r"(bar)
      : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_elect(uint32_t bar, uint32_t bytes) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n\t}" ::"r"(bar), "r"(bytes)
      : "memory");
}
__device__ __forceinline__ void tma_load_2d_elect(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3}], [%4];\n\t}"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar)
      : "memory");
}

// ---- CTA pair (cta_group::2): one UMMA of M = 256 spans the two SMs of a cluster of 2 ------------------------------
// Each CTA keeps its own 128 rows of the M operand and HALF of the N operand's rows in its own shared memory (same
// offsets in both CTAs); the even ("leader") CTA issues the MMAs for the pair, each CTA's TMEM receives its 128 rows of
// D.  A shared::cta address used in the shared::cluster window carries the CTA's rank in bit 24, so clearing that bit
// addresses the leader's copy of a barrier (the convention of the TMA / commit instructions with .cta_group::2).
static constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;
// TMA load into THIS CTA's shared memory whose transaction bytes are counted on the LEADER's mbarrier
__device__ __forceinline__ void tma_load_2d_2sm_elect(uint32_t dst, const CUtensorMap* map, int c0, int c1, uint32_t bar) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes"
      " [%0], [%1, {%2, %3}], [%4];\n\t}"
      ::"r"(dst), "l"(map), "r"(c0), "r"(c1), "r"(bar & PEER_BIT_MASK)
      : "memory");
}
__device__ __forceinline__ void umma_issue_2sm_elect(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                                     uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p, e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "@e tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// completion of the pair's MMAs -> one arrival on the barrier at this offset in EVERY CTA of the mask
__device__ __forceinline__ void umma_arrive_2sm_mc_elect(uint32_t bar, uint16_t cta_mask) {
  asm volatile(
      "{\n\t.reg .pred e;\n\t"
      "elect.sync _|e, 0xffffffff;\n\t"
      "@e tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n\t}"
      ::"r"(bar), "h"(cta_mask)
      : "memory");
}
// arrive on the LEADER's copy of a barrier (from either CTA of the pair)
__device__ __forceinline__ void mbar_arrive_leader(uint32_t bar) {
  asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(bar & PEER_BIT_MASK) : "memory");
}

__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_ld32_issue(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
        "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
        "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
        "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// x * sigmoid(x) = h + h * tanh(h), h = x / 2  (one MUFU op; |rel err| ~ 2^-11, below the bf16 output ulp)
__device__ __forceinline__ float silu_from_half(float h) {      // argument is x / 2
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
  return fmaf(h, t, h);
}
__device__ __forceinline__ float silu_tanh(float x) { return silu_from_half(0.5f * x); }

// GELU in its tanh form (max |deviation| from the erf form ~3e-4, below the bf16 output ulp for |x| > 0.1):
// 0.5 x (1 + tanh(sqrt(2/pi) (x + 0.044715 x^3)))  -- throughput mode only; the fp32 parity path uses erff
__device__ __forceinline__ float gelu_tanh(float x) {
  float u = x * fmaf(0.0356774081f, x * x, 0.7978845608f), t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(u));
  float h = 0.5f * x;
  return fmaf(h, t, h);
}


}  // namespace ds
