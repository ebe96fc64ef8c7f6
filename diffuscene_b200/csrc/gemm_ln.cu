// k_gemm_ln: the tail of the reference's attention wrappers as ONE kernel,
//     out = LayerNorm_g( A[M, K] * W[C, K]^T + bias ) + residual
// i.e. `to_out = Sequential(Conv1d(hidden, dim, 1), LayerNorm(dim))` of LinearAttention / LinearAttentionCross
// (scene_synthesis/networks/denoise_net.py:214-217,234-235 and :268-271,296-297; LayerNorm :93-102: biased variance,
// eps 1e-5, gain only) followed by the `Residual` add of the un-normalised input (:39-45).  Unfused this was a GEMM
// launch (22 us at 4096 scenes) plus a LayerNorm launch (31 us) with a 50 MB activation written and re-read between
// them; fused, the projection never leaves TMEM.
//
// Shape: K = heads * dim_head = 128, C = 512.  That makes the WHOLE weight matrix 128 KB of bf16: every CTA loads it
// once into shared memory (TMA, 128B swizzle) and keeps it for all of its tiles, so the only streamed operand is the
// 128 x 128 activation tile (32 KB per tile).  One persistent CTA per SM, 576 threads:
//   warp 0       TMA producer (weights once, then the A ring)
//   warp 1       MMA issuer: per tile 2 k-blocks x 4 x 2 tcgen05.mma (M = 128, N = 256, K = 16) into ONE 128 x 512 fp32
//                accumulator that fills TMEM (512 columns) -- no second buffer, the MMAs of the next tile start when
//                the last epilogue warp has drained this one (they are 1/5 of the tile time)
//   warps 2-17   epilogue, four warps per TMEM lane quadrant, each owning 128 of the 512 columns; a thread owns ONE
//                token row, so the LayerNorm statistics are in-thread sums over columns plus a 4-way exchange through
//                shared memory (one 128-thread named barrier per quadrant):
//                  pass 1  tcgen05.ld, sum / sum of squares of (acc + bias)
//                  pass 2  tcgen05.ld again, (acc + bias - mean) * rstd * g, + residual, bf16, coalesced store
//                residual loads and output stores go through a per-warp XOR-swizzled 32 x 32 staging block so that
//                every global access is a coalesced 8-row x 64-byte instruction (same scheme as k_gemm_tc).
// Roof: HBM -- 12 MB in + 50 MB residual + 50 MB out per launch at 4096 bedroom scenes = 17 us at the measured copy
// bandwidth; the epilogue's instruction stream (about 10 issue slots per element) is of the same order.
#include <stdio.h>
#include <string.h>

#include "kernels.cuh"
#include "tc_common.cuh"

namespace ds {

namespace {

constexpr int LN_C = 512;                 // output channels = LayerNorm width
constexpr int LN_KMAX = 128;              // weights stay resident: C x K x 2 B = 128 KB
constexpr int LN_EPI_W = 16;
constexpr int LN_THREADS = 64 + LN_EPI_W * 32;
constexpr int LN_STAGES = 3;              // A ring: 3 x 16 KB (a tile needs 2)
constexpr int LN_W_BYTES = LN_C * LN_KMAX * 2;                 // 131072
constexpr int LN_A_OFF = LN_W_BYTES;
constexpr int LN_BAR_OFF = LN_A_OFF + LN_STAGES * A_BYTES;     // barriers: full[4] empty[4] wfull tfull tempty + tmem slot
constexpr int LN_CONST_OFF = LN_BAR_OFF + 128;                 // bias[512] g[512] floats
constexpr int LN_PART_OFF = LN_CONST_OFF + 2 * LN_C * 4;       // [4 column groups][128 rows] float2
constexpr int LN_STG_OFF = ((LN_PART_OFF + 4 * BM * 8 + 1023) / 1024) * 1024;
constexpr int LN_SMEM = 1024 + LN_STG_OFF + LN_EPI_W * 2048;
static_assert(LN_SMEM <= 232448, "shared memory budget exceeded");
// instruction descriptor: D = f32, A = B = bf16, K-major both, N = 256, M = 128
constexpr uint32_t LN_IDESC = (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(256 >> 3) << 17) | (uint32_t(BM >> 4) << 24);

struct LnEpi {
  const float* bias;       // [C] or nullptr
  const float* g;          // [C] LayerNorm gain
  bf16* d; int ldd;
  const bf16* res; int ldres;      // residual added after the norm, or nullptr
  int M, kblocks;
  uint64_t desc_hi;
};

__global__ void __launch_bounds__(LN_THREADS, 1)
k_gemm_ln(const __grid_constant__ CUtensorMap tm_a, const __grid_constant__ CUtensorMap tm_w, LnEpi epi, int* err_flag) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* const base_ptr = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t bar_base = base + LN_BAR_OFF;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (LN_STAGES + s); };
  const uint32_t wfull_bar = bar_base + 8u * (2 * LN_STAGES);
  const uint32_t tfull_bar = bar_base + 8u * (2 * LN_STAGES + 1);
  const uint32_t tempty_bar = bar_base + 8u * (2 * LN_STAGES + 2);
  const uint32_t tmem_slot = bar_base + 8u * (2 * LN_STAGES + 3);
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(base_ptr + LN_BAR_OFF + 8 * (2 * LN_STAGES + 3));
  float* const bias_s = reinterpret_cast<float*>(base_ptr + LN_CONST_OFF);
  float* const g_s = bias_s + LN_C;
  float2* const part = reinterpret_cast<float2*>(base_ptr + LN_PART_OFF);

  const int warp = uniform_warp_idx(), lane = threadIdx.x & 31;
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");     // PDL: the next kernel's prologue may overlap our tail
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_a);
    tma_prefetch_desc(&tm_w);
    for (int s = 0; s < LN_STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(wfull_bar, 1);
    mbar_init(tfull_bar, 1);
    mbar_init(tempty_bar, LN_EPI_W);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "n"(512) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  asm volatile("griddepcontrol.wait;" ::: "memory");      // nothing above touched memory written by earlier kernels

  const int num_tiles = (epi.M + BM - 1) / BM;
  const int kblocks = epi.kblocks;

  if (warp == 0) {
    // TMA producer: the whole warp walks the loop, one elected lane issues (see tc_common.cuh)
    // the whole weight matrix, once: per k-block two boxes of 256 rows x 64 columns -> [512 rows][128 B] slabs
    mbar_expect_tx_elect(wfull_bar, uint32_t(kblocks * LN_C * BK * 2));
    for (int kb = 0; kb < kblocks; ++kb) {
      tma_load_2d_elect(base + uint32_t(kb * LN_C * BK * 2), &tm_w, kb * BK, 0, wfull_bar);
      tma_load_2d_elect(base + uint32_t(kb * LN_C * BK * 2 + 256 * BK * 2), &tm_w, kb * BK, 256, wfull_bar);
    }
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      for (int kb = 0; kb < kblocks; ++kb) {
        mbar_wait(empty_bar(stage), phase ^ 1u, err_flag, 11);
        mbar_expect_tx_elect(full_bar(stage), A_BYTES);
        tma_load_2d_elect(base + LN_A_OFF + stage * A_BYTES, &tm_a, kb * BK, tile * BM, full_bar(stage));
        if (++stage == LN_STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // MMA issuer
    mbar_wait(wfull_bar, 0, err_flag, 12);
    int stage = 0;
    uint32_t phase = 0, tphase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      mbar_wait(tempty_bar, tphase ^ 1u, err_flag, 13);      // the epilogue has drained the accumulator
      tphase ^= 1u;
      tc_fence_after();
      for (int kb = 0; kb < kblocks; ++kb) {
        mbar_wait(full_bar(stage), phase, err_flag, 14);
        tc_fence_after();
        const uint64_t adesc = umma_desc(base + LN_A_OFF + stage * A_BYTES, epi.desc_hi);
        const uint64_t b0 = umma_desc(base + uint32_t(kb * LN_C * BK * 2), epi.desc_hi);
        const uint64_t b1 = umma_desc(base + uint32_t(kb * LN_C * BK * 2 + 256 * BK * 2), epi.desc_hi);
#pragma unroll
        for (int k = 0; k < BK / 16; ++k) {
          umma_issue_elect(tmem_base, adesc + uint64_t(2 * k), b0 + uint64_t(2 * k), LN_IDESC, (kb | k) != 0);
          umma_issue_elect(tmem_base + 256u, adesc + uint64_t(2 * k), b1 + uint64_t(2 * k), LN_IDESC, (kb | k) != 0);
        }
        umma_arrive_elect(empty_bar(stage));
        if (++stage == LN_STAGES) { stage = 0; phase ^= 1u; }
      }
      umma_arrive_elect(tfull_bar);
    }
  } else {
    // ---------------- epilogue warps ----------------
    const int q = warp & 3;                        // TMEM lane quadrant
    const int cgp = (warp - 2) >> 2;               // which 128 columns
    const int etid = threadIdx.x - 64;
    const int row_in_tile = q * 32 + lane;
    for (int n = etid; n < LN_C; n += LN_EPI_W * 32) {
      bias_s[n] = epi.bias ? __ldg(epi.bias + n) : 0.f;
      g_s[n] = __ldg(epi.g + n);
    }
    asm volatile("bar.sync 1, %0;" ::"n"(LN_EPI_W * 32) : "memory");
    const uint32_t stg = base + uint32_t(LN_STG_OFF) + uint32_t((warp - 2) * 2048);
    const int co_r = lane >> 2, co_p = lane & 3;
    uint32_t own_a[4], co_a[4];
#pragma unroll
    for (int g4 = 0; g4 < 4; ++g4) {
      own_a[g4] = stg + uint32_t(lane * 64) + ((uint32_t(g4) ^ uint32_t((lane >> 1) & 3)) << 4);
      const int r = g4 * 8 + co_r;
      co_a[g4] = stg + uint32_t(r * 64) + ((uint32_t(co_p) ^ uint32_t((r >> 1) & 3)) << 4);
    }
    auto sts128 = [](uint32_t a, const uint4& v) {
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
    };
    auto lds128 = [](uint32_t a) {
      uint4 v;
      asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
      return v;
    };
    const int nbase = cgp * 128;
    const uint32_t taddr0 = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(nbase);
    uint32_t tphase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int m0 = tile * BM;
      bool ok4[4];
      bf16* dp4[4];
      const bf16* rp4[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = m0 + q * 32 + i * 8 + co_r;
        ok4[i] = r < epi.M;
        dp4[i] = epi.d + (int64_t)r * epi.ldd + nbase + co_p * 8;
        rp4[i] = epi.res ? epi.res + (int64_t)r * epi.ldres + nbase + co_p * 8 : nullptr;
      }
      if (epi.res) {      // this warp's residual block (32 rows x 256 B) towards L2 while the MMAs run
        const int r = m0 + row_in_tile;
        if (r < epi.M) {
          const char* rp = reinterpret_cast<const char*>(epi.res + (int64_t)r * epi.ldres + nbase);
          asm volatile("prefetch.global.L2 [%0];" ::"l"(rp));
          asm volatile("prefetch.global.L2 [%0];" ::"l"(rp + 128));
        }
      }
      mbar_wait(tfull_bar, tphase, err_flag, 15);
      tphase ^= 1u;
      tc_fence_after();
      // ---- pass 1: statistics of (acc + bias) over this warp's 128 columns
      {
        uint32_t ra[32];
        float s = 0.f, ss = 0.f;
        auto acc = [&](const uint32_t (&r)[32], int c) {
          const float4* b4 = reinterpret_cast<const float4*>(bias_s + nbase + c * 32);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 bb = b4[j];
            const float v0 = __uint_as_float(r[4 * j]) + bb.x, v1 = __uint_as_float(r[4 * j + 1]) + bb.y;
            const float v2 = __uint_as_float(r[4 * j + 2]) + bb.z, v3 = __uint_as_float(r[4 * j + 3]) + bb.w;
            s += (v0 + v1) + (v2 + v3);
            ss = fmaf(v0, v0, ss); ss = fmaf(v1, v1, ss); ss = fmaf(v2, v2, ss); ss = fmaf(v3, v3, ss);
          }
        };
        // (one TMEM buffer in flight: 4 warps per SM sub-partition hide the load latency; a second buffer spills)
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          tmem_ld32(taddr0 + uint32_t(c * 32), ra);
          acc(ra, c);
        }
        part[cgp * BM + row_in_tile] = make_float2(s, ss);
      }
      asm volatile("bar.sync %0, 128;" ::"r"(2 + q) : "memory");      // the four warps of this lane quadrant
      float mean, rstd;
      {
        float s = 0.f, ss = 0.f;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
          const float2 p2 = part[c * BM + row_in_tile];
          s += p2.x;
          ss += p2.y;
        }
        mean = s * (1.0f / LN_C);
        const float var = fmaxf(ss * (1.0f / LN_C) - mean * mean, 0.f);
        rstd = rsqrtf(var + 1e-5f);
      }
      const float nmr = -mean * rstd;
      // ---- pass 2: normalise, gain, residual, coalesced store
      uint32_t ra[32];
      uint4 rga[4], rgb[4];
      auto fetch_res = [&](uint4 (&rg)[4], int c) {
        if (epi.res) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            rg[i] = make_uint4(0u, 0u, 0u, 0u);
            if (ok4[i]) rg[i] = __ldg(reinterpret_cast<const uint4*>(rp4[i] + c * 32));
          }
        }
      };
      auto finish = [&](const uint32_t (&r)[32], int c, const uint4 (&rcur)[4], uint4 (&rnext)[4]) {
        if (c + 1 < 4) fetch_res(rnext, c + 1);
        float v[32];
        const float4* b4 = reinterpret_cast<const float4*>(bias_s + nbase + c * 32);
        const float4* g4 = reinterpret_cast<const float4*>(g_s + nbase + c * 32);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const float4 bb = b4[j], gg = g4[j];
          // ((acc + b) - mean) * rstd * g  =  fma(acc + b, rstd, -mean * rstd) * g
          v[4 * j] = fmaf(__uint_as_float(r[4 * j]) + bb.x, rstd, nmr) * gg.x;
          v[4 * j + 1] = fmaf(__uint_as_float(r[4 * j + 1]) + bb.y, rstd, nmr) * gg.y;
          v[4 * j + 2] = fmaf(__uint_as_float(r[4 * j + 2]) + bb.z, rstd, nmr) * gg.z;
          v[4 * j + 3] = fmaf(__uint_as_float(r[4 * j + 3]) + bb.w, rstd, nmr) * gg.w;
        }
        if (epi.res) {
#pragma unroll
          for (int i = 0; i < 4; ++i) sts128(co_a[i], rcur[i]);
          __syncwarp();
#pragma unroll
          for (int g8 = 0; g8 < 4; ++g8) {
            const uint4 rv = lds128(own_a[g8]);
            const uint32_t w4[4] = {rv.x, rv.y, rv.z, rv.w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              v[g8 * 8 + e * 2] += __uint_as_float(w4[e] << 16);
              v[g8 * 8 + e * 2 + 1] += __uint_as_float(w4[e] & 0xffff0000u);
            }
          }
          __syncwarp();
        }
#pragma unroll
        for (int g8 = 0; g8 < 4; ++g8) {
          uint4 o;
          __nv_bfloat162* h2 = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
          for (int e = 0; e < 4; ++e) h2[e] = __floats2bfloat162_rn(v[g8 * 8 + e * 2], v[g8 * 8 + e * 2 + 1]);
          sts128(own_a[g8], o);
        }
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const uint4 o = lds128(co_a[i]);
          if (ok4[i]) *reinterpret_cast<uint4*>(dp4[i] + c * 32) = o;
        }
        __syncwarp();
      };
      fetch_res(rga, 0);
      tmem_ld32(taddr0, ra);
      finish(ra, 0, rga, rgb);
      tmem_ld32(taddr0 + 32u, ra);
      finish(ra, 1, rgb, rga);
      tmem_ld32(taddr0 + 64u, ra);
      finish(ra, 2, rga, rgb);
      tmem_ld32(taddr0 + 96u, ra);
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar);      // accumulator drained: the next tile's MMAs may start
      finish(ra, 3, rgb, rga);
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(512) : "memory");
  }
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
struct LnGemmPlan {
  CUtensorMap tm_a, tm_w;
  LnEpi epi;
  int num_sms;
};

bool tc_encode_2d(CUtensorMap* map, const void* base, uint64_t inner, uint64_t rows, uint64_t pitch_elems,
                  uint32_t box_rows, char* err, int err_len);      // gemm_tc.cu
int* tc_error_flag_dev();                                          // gemm_tc.cu
int tc_num_sms();

bool ln_gemm_supported(int N, int K) { return N == LN_C && K > 0 && K % BK == 0 && K <= LN_KMAX; }

LnGemmPlan* ln_plan_create(const GemmArgs& g, int rows_capacity, char* err, int err_len) {
  if (!tc_runtime_available(err, err_len)) return nullptr;
  if (!ln_gemm_supported(g.N, g.k0) || g.a1 || !g.gamma) {
    if (err) snprintf(err, err_len, "fused GEMM + LayerNorm needs N = %d, K %% 64 == 0, K <= %d, one operand, a gain vector", LN_C, LN_KMAX);
    return nullptr;
  }
  if ((g.lda0 % 8) || (g.ldw % 8) || (g.ldd % 8) || (g.res && (g.ldres % 8)) || ((uintptr_t)g.a0 % 16) ||
      ((uintptr_t)g.w % 16) || ((uintptr_t)g.d % 16) || (g.res && ((uintptr_t)g.res % 16))) {
    if (err) snprintf(err, err_len, "fused GEMM + LayerNorm needs 16-byte aligned operands and pitches");
    return nullptr;
  }
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(k_gemm_ln, cudaFuncAttributeMaxDynamicSharedMemorySize, LN_SMEM);
    attr_set = true;
  }
  LnGemmPlan* p = new LnGemmPlan();
  memset(p, 0, sizeof(*p));
  bool ok = tc_encode_2d(&p->tm_a, g.a0, g.k0, rows_capacity, g.lda0, BM, err, err_len);
  if (ok) ok = tc_encode_2d(&p->tm_w, g.w, g.k0, g.N, g.ldw, 256, err, err_len);
  if (!ok) {
    delete p;
    return nullptr;
  }
  p->epi.bias = g.bias;
  p->epi.g = g.gamma;
  p->epi.d = (bf16*)g.d;
  p->epi.ldd = g.ldd;
  p->epi.res = (const bf16*)g.res;
  p->epi.ldres = g.ldres;
  p->epi.M = g.M;
  p->epi.kblocks = g.k0 / BK;
  p->epi.desc_hi = umma_desc_hi_sw128();
  p->num_sms = tc_num_sms();
  return p;
}
void ln_plan_destroy(LnGemmPlan* p) { delete p; }

int launch_gemm_ln(const LnGemmPlan* p, int M, cudaStream_t s) {
  LnEpi epi = p->epi;
  epi.M = M;
  const int tiles = (M + BM - 1) / BM;
  if (tiles == 0) return 0;
  const int grid = tiles < p->num_sms ? tiles : p->num_sms;
  return tc_launch(k_gemm_ln, grid, LN_THREADS, LN_SMEM, s, pdl_enabled(M), p->tm_a, p->tm_w, epi, tc_error_flag_dev());
}

}  // namespace ds
