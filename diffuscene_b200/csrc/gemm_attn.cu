// k_ln_qkv_attn: the head of the reference's linear-attention wrapper as ONE kernel,
//     o[tokens, 128] = LinearAttentionCore( to_qkv( LayerNorm_g(x) ) )
// i.e. `Residual(PreNorm(dim, LinearAttention(dim)))` up to (not including) `to_out`
// (scene_synthesis/networks/denoise_net.py:104-112 PreNorm, :93-102 LayerNorm, :208-233 LinearAttention: qkv = Conv1d(dim,
// 3 * 128, 1, bias=False); q = softmax over the 32 head channels * 32^-1/2; k = softmax over the tokens;
// context = k v^T; out = context^T q).  Unfused this was three launches (LayerNorm 25 us, to_qkv GEMM 36 us, core 21 us
// at 4096 bedroom scenes) with a 50 MB and a 38 MB activation written and re-read in between; k_gemm_ln (gemm_ln.cu)
// is the other half of the wrapper.
//
// The LayerNorm never materialises.  Its gain is folded into the weights when they are packed
// (W'[n][k] = W[n][k] g[k], ds_commit_weights), and with cs[n] = sum_k W'[n][k]:
//     to_qkv(LN(x))[row][n] = rstd[row] * ( (x W'^T)[row][n] - mean[row] * cs[n] )
// so the MMAs run on the raw bf16 x (no extra rounding of a normalised copy) and the per-row statistics are applied
// to the fp32 accumulator.  The statistics are computed by the epilogue warps from global memory (the same lines the
// TMA loads are pulling through L2) while the MMAs run.
//
// Tile = SPT whole scenes (10 scenes = 120 token rows for N = 12; UMMA M = 128).  One persistent CTA per SM, 576 threads:
//   warp 0      TMA producer: per k-block the 128 x 64 x tile and the 384 x 64 W' slab (2 stages x 64 KB)
//   warp 1      MMA issuer: 2 x tcgen05.mma per k16 step (N = 256 -> TMEM columns 0..255, N = 128 -> 256..383)
//   warps 2-17  (a) row statistics of the tile (overlaps the MMAs); (b) accumulator -> normalise -> bf16 q | k | v rows
//               in shared memory ([row][392] bf16: 784-byte rows are conflict-free for ldmatrix and for the 16-byte
//               row-owner stores), after which TMEM is released and the next tile's MMAs start; (c) the attention core,
//               one warp per (scene, head), on mma.sync with operands straight from that shared-memory block
//               (k is soft-maxed in place; rows of the neighbouring scene inside a 16-token MMA tile are masked out of
//               the v fragments), o written to global memory as packed bf16 pairs.
// Roof: the 512 KB of operands per tile come from L2 (210 MB per launch at 4096 scenes, ~20 us at the L2 -> SM limit);
// HBM traffic is x in (50 MB) + o out (12.6 MB).
#include <stdio.h>
#include <string.h>

#include "kernels.cuh"
#include "tc_common.cuh"

namespace ds {

namespace {

constexpr int AT_NQ = 384;                          // q | k | v channels
constexpr int AT_STAGES = 2;
constexpr int AT_W_BYTES = AT_NQ * BK * 2;          // 49152
constexpr int AT_STAGE_BYTES = A_BYTES + AT_W_BYTES;                 // 65536
constexpr int AT_EPI_W = 16;
constexpr int AT_THREADS = 64 + AT_EPI_W * 32;
constexpr int AT_LDS = 392;                         // staging row pitch in bf16 (784 B)
constexpr int AT_BAR_OFF = AT_STAGES * AT_STAGE_BYTES;               // full[2] empty[2] tfull tempty + tmem slot
constexpr int AT_CS_OFF = AT_BAR_OFF + 64;                           // cs[384] floats
constexpr int AT_STAT_OFF = AT_CS_OFF + AT_NQ * 4;                   // (mean, rstd)[128]
constexpr int AT_STG_OFF = AT_STAT_OFF + 128 * 8;
constexpr uint32_t AT_IDESC_256 = (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(256 >> 3) << 17) | (uint32_t(BM >> 4) << 24);
constexpr uint32_t AT_IDESC_128 = (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(128 >> 3) << 17) | (uint32_t(BM >> 4) << 24);

template <int NOBJ>
struct AtCfg {
  // scenes per tile: 10 x 12 = 120 rows; for N = 21 five scenes (105 rows): six would not leave shared memory for the
  // 11 masked tail rows of the last scene's second 16-token MMA step
  static constexpr int SPT = (NOBJ == 12) ? 10 : (NOBJ == 21 ? 5 : 128 / NOBJ);
  static constexpr int ROWS = SPT * NOBJ;                            // token rows per tile (<= 128)
  static constexpr int NT = (NOBJ + 15) / 16 * 16;                   // tokens of a scene rounded up to MMA tiles
  static constexpr int STG_ROWS = ROWS + (NT - NOBJ);                // + zeroed tail rows read (masked) by the last scene
  static constexpr int SMEM = 1024 + AT_STG_OFF + STG_ROWS * AT_LDS * 2;
  static_assert(SMEM <= 232448, "shared memory budget exceeded");
};

struct AtEpi {
  const bf16* x; int ldx;           // the un-normalised input (statistics)
  const float* cs;                  // [384] column sums of the gain-folded, bf16-rounded weights
  bf16* o; int ldo;                 // [M, 128]
  int M, kblocks;
  uint64_t desc_hi;
};

__device__ __forceinline__ float at_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ void at_mma(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void at_ldsm_x4_t(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr));
}
__device__ __forceinline__ uint32_t at_pack(float lo, float hi) {
  __nv_bfloat162 h2 = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h2);
}
__device__ __forceinline__ float at_quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}
__device__ __forceinline__ float at_quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  return v + __shfl_xor_sync(0xffffffffu, v, 2);
}

// One (scene, head) of the linear-attention core on one warp.  sbase: shared-memory bf16 pointer to the scene's first
// row, columns [q | k | v] x 128, row pitch AT_LDS; head h uses columns h*32 .. h*32+31 of each third.
template <int NOBJ>
__device__ __forceinline__ void linattn_core(bf16* sbase, int h, bf16* out, int ld_out, int lane) {
  constexpr int NT = AtCfg<NOBJ>::NT, MT = NT / 16;
  const int g = lane >> 2, t = lane & 3;
  const float LOG2E = 1.4426950408889634f;
  bf16* qb = sbase + h * 32;
  bf16* kb = sbase + 128 + h * 32;
  const uint32_t k_a = smem_u32(kb), v_a = smem_u32(sbase + 256 + h * 32);
  // ---- k~: softmax over the scene's tokens, one lane per channel, written back in place
  {
    float kv[NOBJ];
    float kmax = -INFINITY;
#pragma unroll
    for (int r = 0; r < NOBJ; ++r) {
      kv[r] = __bfloat162float(kb[r * AT_LDS + lane]);
      kmax = fmaxf(kmax, kv[r]);
    }
    float ksum = 0.f;
    const float moff = -kmax * LOG2E;
#pragma unroll
    for (int r = 0; r < NOBJ; ++r) {
      kv[r] = at_exp2(fmaf(kv[r], LOG2E, moff));
      ksum += kv[r];
    }
    const float kinv = __fdividef(1.0f, ksum);
#pragma unroll
    for (int r = 0; r < NOBJ; ++r) kb[r * AT_LDS + lane] = __float2bfloat16_rn(kv[r] * kinv);
  }
  // ---- q~ in MMA fragment layout: softmax over the 32 channels of a token = 8 local values + the quad
  uint32_t qa[MT][2][4];
#pragma unroll
  for (int mq = 0; mq < MT; ++mq) {
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
      const int tk = 16 * mq + 8 * hf + g;
      const bool ok = tk < NOBJ;
      const uint32_t* qp = reinterpret_cast<const uint32_t*>(qb + (ok ? tk : 0) * AT_LDS + 2 * t);
      float v[8];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t raw = qp[4 * j];                      // channels 8j + 2t, 8j + 2t + 1
        v[2 * j] = __uint_as_float(raw << 16);
        v[2 * j + 1] = __uint_as_float(raw & 0xffff0000u);
      }
      float m = fmaxf(fmaxf(fmaxf(v[0], v[1]), fmaxf(v[2], v[3])), fmaxf(fmaxf(v[4], v[5]), fmaxf(v[6], v[7])));
      m = at_quad_max(m);
      const float moff = -m * LOG2E;
      float ssum = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        v[j] = at_exp2(fmaf(v[j], LOG2E, moff));
        ssum += v[j];
      }
      ssum = at_quad_sum(ssum);
      const float sc = ok ? __fdividef(0.17677669529663687f, ssum) : 0.f;      // 32^-1/2 / sum
      qa[mq][0][hf] = at_pack(v[0] * sc, v[1] * sc);
      qa[mq][0][2 + hf] = at_pack(v[2] * sc, v[3] * sc);
      qa[mq][1][hf] = at_pack(v[4] * sc, v[5] * sc);
      qa[mq][1][2 + hf] = at_pack(v[6] * sc, v[7] * sc);
    }
  }
  __syncwarp();
  // ---- ctx^T[e][d] = sum_tok v[tok][e] k~[tok][d]: M = e (2 tiles), N = d (4 tiles), K = tokens (MT steps of 16)
  float c[2][4][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) c[mt][nt][i] = 0.f;
  const int mi = lane >> 3, mr = lane & 7;
#pragma unroll
  for (int kt = 0; kt < MT; ++kt) {
    uint32_t a[2][4], b[2][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
      at_ldsm_x4_t(a[mt], v_a + uint32_t(((16 * kt + 8 * (mi >> 1) + mr) * AT_LDS + 16 * mt + 8 * (mi & 1)) * 2));
#pragma unroll
    for (int np = 0; np < 2; ++np)
      at_ldsm_x4_t(b[np], k_a + uint32_t(((16 * kt + 8 * (mi & 1) + mr) * AT_LDS + 8 * (2 * np + (mi >> 1))) * 2));
    // tokens >= NOBJ of this 16-token step are rows of the NEXT scene (or the zeroed tail): drop them from the v operand.
    // A fragment of m16n8k16: a0 / a1 hold k = 2t, 2t + 1; a2 / a3 hold k = 2t + 8, 2t + 9
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      const int k0 = 16 * kt + 2 * t, k1 = k0 + 8;
      const uint32_t m0 = (k0 + 1 < NOBJ) ? 0xffffffffu : (k0 < NOBJ ? 0x0000ffffu : 0u);
      const uint32_t m1 = (k1 + 1 < NOBJ) ? 0xffffffffu : (k1 < NOBJ ? 0x0000ffffu : 0u);
      a[mt][0] &= m0; a[mt][1] &= m0; a[mt][2] &= m1; a[mt][3] &= m1;
    }
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) at_mma(c[mt][nt], a[mt], b[nt >> 1][2 * (nt & 1)], b[nt >> 1][2 * (nt & 1) + 1]);
  }
  // ---- out[tok][e] = sum_d q~[tok][d] ctx[d][e]: M = tokens, N = e (4 tiles of 8), K = d (2 steps)
  uint32_t cb[4][2][2];
#pragma unroll
  for (int eb = 0; eb < 4; ++eb)
#pragma unroll
    for (int ks2 = 0; ks2 < 2; ++ks2) {
      const int i0 = (eb & 1) * 2;
      cb[eb][ks2][0] = at_pack(c[eb >> 1][2 * ks2][i0], c[eb >> 1][2 * ks2][i0 + 1]);
      cb[eb][ks2][1] = at_pack(c[eb >> 1][2 * ks2 + 1][i0], c[eb >> 1][2 * ks2 + 1][i0 + 1]);
    }
#pragma unroll
  for (int mq = 0; mq < MT; ++mq) {
#pragma unroll
    for (int eb = 0; eb < 4; ++eb) {
      float o[4] = {0.f, 0.f, 0.f, 0.f};
      at_mma(o, qa[mq][0], cb[eb][0][0], cb[eb][0][1]);
      at_mma(o, qa[mq][1], cb[eb][1][0], cb[eb][1][1]);
      const int tk0 = 16 * mq + g, tk1 = tk0 + 8;
      bf16* op = out + (int64_t)tk0 * ld_out + h * 32 + 8 * eb + 2 * t;
      if (tk0 < NOBJ) *reinterpret_cast<uint32_t*>(op) = at_pack(o[0], o[1]);
      if (tk1 < NOBJ) *reinterpret_cast<uint32_t*>(op + (int64_t)8 * ld_out) = at_pack(o[2], o[3]);
    }
  }
}

template <int NOBJ>
__global__ void __launch_bounds__(AT_THREADS, 1)
k_ln_qkv_attn(const __grid_constant__ CUtensorMap tm_x, const __grid_constant__ CUtensorMap tm_w, AtEpi epi, int* err_flag) {
  using Cfg = AtCfg<NOBJ>;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* const base_ptr = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t bar_base = base + AT_BAR_OFF;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (AT_STAGES + s); };
  const uint32_t tfull_bar = bar_base + 8u * (2 * AT_STAGES);
  const uint32_t tempty_bar = bar_base + 8u * (2 * AT_STAGES + 1);
  const uint32_t tmem_slot = bar_base + 8u * (2 * AT_STAGES + 2);
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(base_ptr + AT_BAR_OFF + 8 * (2 * AT_STAGES + 2));
  float* const cs_s = reinterpret_cast<float*>(base_ptr + AT_CS_OFF);
  float2* const stat_s = reinterpret_cast<float2*>(base_ptr + AT_STAT_OFF);
  bf16* const stg = reinterpret_cast<bf16*>(base_ptr + AT_STG_OFF);

  const int warp = uniform_warp_idx(), lane = threadIdx.x & 31;
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");     // PDL: the next kernel's prologue may overlap our tail
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_x);
    tma_prefetch_desc(&tm_w);
    for (int s = 0; s < AT_STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    mbar_init(tfull_bar, 1);
    mbar_init(tempty_bar, AT_EPI_W);
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

  const int n_scenes = epi.M / NOBJ;
  const int num_tiles = (n_scenes + Cfg::SPT - 1) / Cfg::SPT;
  const int kblocks = epi.kblocks;

  if (warp == 0) {
    // TMA producer: the whole warp walks the loop, one elected lane issues (see tc_common.cuh)
    int stage = 0;
    uint32_t phase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int m0 = tile * Cfg::ROWS;
      for (int kb = 0; kb < kblocks; ++kb) {
        mbar_wait(empty_bar(stage), phase ^ 1u, err_flag, 21);
        mbar_expect_tx_elect(full_bar(stage), AT_STAGE_BYTES);
        const uint32_t sa = base + stage * AT_STAGE_BYTES;
        tma_load_2d_elect(sa, &tm_x, kb * BK, m0, full_bar(stage));
#pragma unroll
        for (int r3 = 0; r3 < 3; ++r3)      // W' slab: three boxes of 128 rows -> [384 rows][128 B]
          tma_load_2d_elect(sa + A_BYTES + r3 * 128 * BK * 2, &tm_w, kb * BK, r3 * 128, full_bar(stage));
        if (++stage == AT_STAGES) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // MMA issuer
    int stage = 0;
    uint32_t phase = 0, tphase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      mbar_wait(tempty_bar, tphase ^ 1u, err_flag, 22);
      tphase ^= 1u;
      tc_fence_after();
      for (int kb = 0; kb < kblocks; ++kb) {
        mbar_wait(full_bar(stage), phase, err_flag, 23);
        tc_fence_after();
        const uint32_t sa = base + stage * AT_STAGE_BYTES;
        const uint64_t adesc = umma_desc(sa, epi.desc_hi);
        const uint64_t b0 = umma_desc(sa + A_BYTES, epi.desc_hi);
        const uint64_t b1 = umma_desc(sa + A_BYTES + 256 * BK * 2, epi.desc_hi);
#pragma unroll
        for (int k = 0; k < BK / 16; ++k) {
          umma_issue_elect(tmem_base, adesc + uint64_t(2 * k), b0 + uint64_t(2 * k), AT_IDESC_256, (kb | k) != 0);
          umma_issue_elect(tmem_base + 256u, adesc + uint64_t(2 * k), b1 + uint64_t(2 * k), AT_IDESC_128, (kb | k) != 0);
        }
        umma_arrive_elect(empty_bar(stage));
        if (++stage == AT_STAGES) { stage = 0; phase ^= 1u; }
      }
      umma_arrive_elect(tfull_bar);
    }
  } else {
    // ---------------- epilogue / core warps ----------------
    const int ew = warp - 2;                     // 0..15
    const int q = warp & 3;                      // TMEM lane quadrant of this warp
    const int part = ew >> 2;                    // which 96 of the 384 columns
    const int etid = threadIdx.x - 64;
    auto epi_bar = []() { asm volatile("bar.sync 1, %0;" ::"n"(AT_EPI_W * 32) : "memory"); };
    for (int n = etid; n < AT_NQ; n += AT_EPI_W * 32) cs_s[n] = __ldg(epi.cs + n);
    // zero the staging tail once (rows ROWS .. STG_ROWS-1: finite operands for the masked MMA lanes of the last scene)
    for (int i = etid; i < (Cfg::STG_ROWS - Cfg::ROWS) * AT_LDS / 2; i += AT_EPI_W * 32)
      reinterpret_cast<uint32_t*>(stg + Cfg::ROWS * AT_LDS)[i] = 0u;
    const int row_in_tile = q * 32 + lane;
    uint32_t tphase = 0;
    for (int tile = blockIdx.x; tile < num_tiles; tile += gridDim.x) {
      const int m0 = tile * Cfg::ROWS;
      const int rows_here = min(Cfg::ROWS, epi.M - m0);
      // ---- (a) LayerNorm statistics of this tile's rows, 8 rows per warp, coalesced 1 KB row reads; the loads of four
      //      rows are in flight together (one L2 round trip per batch instead of one per row)
#pragma unroll
      for (int rb = 0; rb < 8; rb += 4) {
        uint4 u[4][2];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int r = ew * 8 + rb + j;
          u[j][0] = u[j][1] = make_uint4(0u, 0u, 0u, 0u);
          if (r < rows_here) {
            const uint4* rp = reinterpret_cast<const uint4*>(epi.x + (int64_t)(m0 + r) * epi.ldx) + lane * 2;
            u[j][0] = __ldg(rp);
            u[j][1] = __ldg(rp + 1);
          }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          float s = 0.f, ss = 0.f;
#pragma unroll
          for (int i = 0; i < 2; ++i) {
            const uint32_t w4[4] = {u[j][i].x, u[j][i].y, u[j][i].z, u[j][i].w};
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              const float a = __uint_as_float(w4[e] << 16), b = __uint_as_float(w4[e] & 0xffff0000u);
              s += a + b;
              ss = fmaf(a, a, ss);
              ss = fmaf(b, b, ss);
            }
          }
          s = warp_sum(s);
          ss = warp_sum(ss);
          if (lane == 0) {
            const float mean = s * (1.0f / 512.0f);
            const float var = fmaxf(ss * (1.0f / 512.0f) - mean * mean, 0.f);
            stat_s[ew * 8 + rb + j] = make_float2(mean, rsqrtf(var + 1e-5f));
          }
        }
      }
      epi_bar();                                  // statistics visible; every warp has left the previous tile's core
      // ---- (b) accumulator -> q | k | v rows in shared memory
      mbar_wait(tfull_bar, tphase, err_flag, 24);
      tphase ^= 1u;
      tc_fence_after();
      {
        const float2 st = stat_s[row_in_tile];
        const float nmr = -st.x * st.y;           // -mean * rstd
        bf16* rowp = stg + row_in_tile * AT_LDS + part * 96;
        uint32_t ra[32];
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          tmem_ld32(tmem_base + (uint32_t(q * 32) << 16) + uint32_t(part * 96 + c * 32), ra);
          if (row_in_tile < Cfg::ROWS) {
            const float* csp = cs_s + part * 96 + c * 32;
#pragma unroll
            for (int g8 = 0; g8 < 4; ++g8) {
              uint4 o;
              uint32_t* ow = reinterpret_cast<uint32_t*>(&o);
#pragma unroll
              for (int e = 0; e < 4; ++e) {
                const int j = g8 * 8 + e * 2;
                // rstd * (acc - mean * cs) = fma(acc, rstd, (-mean * rstd) * cs)
                ow[e] = at_pack(fmaf(__uint_as_float(ra[j]), st.y, nmr * csp[j]), fmaf(__uint_as_float(ra[j + 1]), st.y, nmr * csp[j + 1]));
              }
              *reinterpret_cast<uint4*>(rowp + c * 32 + g8 * 8) = o;
            }
          }
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(tempty_bar);     // accumulator drained: the next tile's MMAs run under the core
      epi_bar();                                  // all q | k | v rows are in place
      // ---- (c) attention core: (scene, head) tasks round-robin over the 16 warps
      const int scenes_here = rows_here / NOBJ;
      for (int task = ew; task < scenes_here * 4; task += AT_EPI_W) {
        const int sc = task >> 2, h = task & 3;
        linattn_core<NOBJ>(stg + sc * NOBJ * AT_LDS, h, epi.o + (int64_t)(m0 + sc * NOBJ) * epi.ldo, epi.ldo, lane);
      }
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
struct AttnQkvPlan {
  CUtensorMap tm_x, tm_w;
  AtEpi epi;
  int n_obj, num_sms;
};

bool tc_encode_2d(CUtensorMap* map, const void* base, uint64_t inner, uint64_t rows, uint64_t pitch_elems,
                  uint32_t box_rows, char* err, int err_len);      // gemm_tc.cu
int* tc_error_flag_dev();
int tc_num_sms();

bool attn_qkv_supported(int n_obj, int C) { return (n_obj == 12 || n_obj == 21) && C == 512; }

// x [rows, 512] bf16; w [384, 512] bf16 = to_qkv weights with the LayerNorm gain folded into the columns;
// cs [384] fp32 = row sums of those (bf16-rounded) weights; o [rows, 128] bf16
AttnQkvPlan* attn_qkv_plan_create(const void* x, int ldx, const void* w, int ldw, const float* cs, void* o, int ldo,
                                  int n_obj, int K, int rows_capacity, char* err, int err_len) {
  if (!tc_runtime_available(err, err_len)) return nullptr;
  if (!attn_qkv_supported(n_obj, K) || (ldx % 8) || (ldw % 8) || (ldo % 2)) {
    if (err) snprintf(err, err_len, "fused LN + to_qkv + linear attention needs n_obj in {12, 21}, C = 512, aligned pitches");
    return nullptr;
  }
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(k_ln_qkv_attn<12>, cudaFuncAttributeMaxDynamicSharedMemorySize, AtCfg<12>::SMEM);
    cudaFuncSetAttribute(k_ln_qkv_attn<21>, cudaFuncAttributeMaxDynamicSharedMemorySize, AtCfg<21>::SMEM);
    attr_set = true;
  }
  AttnQkvPlan* p = new AttnQkvPlan();
  memset(p, 0, sizeof(*p));
  bool ok = tc_encode_2d(&p->tm_x, x, K, rows_capacity, ldx, BM, err, err_len);
  if (ok) ok = tc_encode_2d(&p->tm_w, w, K, AT_NQ, ldw, 128, err, err_len);      // 128-row boxes, three per k-block
  if (!ok) {
    delete p;
    return nullptr;
  }
  p->epi.x = (const bf16*)x;
  p->epi.ldx = ldx;
  p->epi.cs = cs;
  p->epi.o = (bf16*)o;
  p->epi.ldo = ldo;
  p->epi.kblocks = K / BK;
  p->epi.desc_hi = umma_desc_hi_sw128();
  p->n_obj = n_obj;
  p->num_sms = tc_num_sms();
  return p;
}
void attn_qkv_plan_destroy(AttnQkvPlan* p) { delete p; }

int launch_ln_qkv_attn(const AttnQkvPlan* p, int M, cudaStream_t s) {
  AtEpi epi = p->epi;
  epi.M = M;
  const int n_scenes = M / p->n_obj;
  const int spt = p->n_obj == 21 ? AtCfg<21>::SPT : AtCfg<12>::SPT;
  const int tiles = (n_scenes + spt - 1) / spt;
  if (tiles == 0) return 0;
  const int grid = tiles < p->num_sms ? tiles : p->num_sms;
  const bool pdl = pdl_enabled(M);
  if (p->n_obj == 21)
    return tc_launch(k_ln_qkv_attn<21>, grid, AT_THREADS, AtCfg<21>::SMEM, s, pdl, p->tm_x, p->tm_w, epi, tc_error_flag_dev());
  return tc_launch(k_ln_qkv_attn<12>, grid, AT_THREADS, AtCfg<12>::SMEM, s, pdl, p->tm_x, p->tm_w, epi, tc_error_flag_dev());
}

}  // namespace ds
