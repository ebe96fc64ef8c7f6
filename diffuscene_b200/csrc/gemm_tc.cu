// tcgen05 tensor-core GEMMs for sm_100a:  D[M,N] = act([A0|A1][M,K] * W[N,K]^T + bias) (+ residual)
// bf16 operands, fp32 accumulation in TMEM, bf16 output.  Two kernels share the TMA / mbarrier / TMEM plumbing:
//   k_gemm_tc<BN, GN>   rows of D on the TMEM lanes (activations = M operand), described right below;
//   k_gemm_gnt<NOBJ>    output CHANNELS on the TMEM lanes (weights = M operand, whole scenes = N operand), the
//                       kernel of the fused conv + GroupNorm + FiLM + SiLU blocks -- see its own header further down.
//
// This kernel carries every 1x1-conv / linear layer of the denoiser in throughput mode (reference:
// F.conv1d / nn.Linear calls of scene_synthesis/networks/denoise_net.py:91,183,214-217,244-245,487-502).
//
// Structure (one persistent CTA per SM, 320 threads):
//   warp 0      TMA producer: cp.async.bulk.tensor 2-D tiles (128B swizzle) of A (128 x 64) and W (BN x 64)
//               into a STAGES-deep shared-memory ring, completion on mbarriers
//   warp 1      MMA issuer: one elected thread issues tcgen05.mma (M=128, N=BN, K=16) x 4 per k-block,
//               accumulating into one of two TMEM buffers; tcgen05.commit releases smem slots / signals
//               the epilogue.  Both single-thread roles run their loops warp-uniformly and elect the issuing
//               lane inside the PTX wrapper (tc_common.cuh): descriptors live in uniform registers and the
//               four UTCHMMA of a k-block issue back to back.
//   TWO = true  the CTA-pair instantiation (cluster of 2, tcgen05.mma.cta_group::2, M = 256): each CTA loads its
//               own token tile and half of the weight tile, the even CTA issues for both, commits are multicast
//               to both CTAs' barriers, both epilogues release the leader's TMEM-empty barrier.  Chosen by
//               shape at plan creation (K >= 1024 or N >= 2048), a separate instantiation because a kernel
//               that contains cta_group::2 instructions cannot be launched without a cluster.
//   warps 2-9   epilogue (two warps per TMEM lane quadrant, each owning half of the tile's columns):
//               tcgen05.ld (32 lanes x 32 columns) -> epilogue math -> bf16 -> HBM; double-buffered TMEM
//               lets the epilogue of tile i overlap the MMAs of tile i+1.  Two epilogues:
//                 plain  bias / GELU|SiLU / residual
//                 GN     the whole `Block` of the reference (denoise_net.py:160-176) after the conv:
//                        bias -> GroupNorm(8) statistics per (scene, group) reduced across the rows of a
//                        scene through shared memory -> affine -> FiLM -> SiLU (-> + residual).  M tiles
//                        are whole scenes (120 of 128 rows for N=12, 126 for N=21), N tiles are 4 whole
//                        groups, so the statistics never leave the CTA.
// Both operands are K-major (activations [rows, K], weights [N, K] exactly as PyTorch stores them), so no
// transposes exist anywhere in the data path.  A "virtual concat" [A0|A1] (the U-Net skip connections,
// denoise_net.py:562,566,573) is served by switching tensor maps inside the k loop.
#include <cuda.h>
#include <type_traits>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include "kernels.cuh"
#include "tc_common.cuh"

namespace ds {

static constexpr int EPI_WARPS = 8;
static constexpr int TC_THREADS = 64 + EPI_WARPS * 32;
struct TcEpi {
  const float* bias;
  bf16* d; int ldd;
  const bf16* res; int ldres;
  int act;
  int M, N;
  int kb0, kb1;          // k-blocks taken from A0 and from A1
  uint64_t desc_hi;      // constant (non-address) bits of the shared-memory matrix descriptors
  uint32_t idesc;        // tcgen05 instruction descriptor
  int tile_rows;         // rows advanced per M tile (128, or whole scenes for the GN epilogue)
  // GroupNorm epilogue
  int n_obj;             // rows per scene
  int C;                 // channel count of the FiLM table rows ([scale(C) | shift(C)])
  const float* gamma;
  const float* beta;
  FilmRef film;
  int film_uniform;      // FILM_TIME only: t[] holds one value for the whole launch (sampling loop)
  int plain;             // channels-on-lanes kernel without GroupNorm: bias, activation, residual only
  float* d32;            // row-major plain kernel: fp32 output accumulated with atomics (split-K weight-gradient GEMMs)
  int ksplit;            // ... number of K splits (work units = tiles x ksplit)
  unsigned long long* trace;   // optional [grid][8] cycle counters (bring-up / profiling aid), else nullptr
};
// trace slots: 0 producer wait-empty, 1 producer total, 2 mma wait-tmem-empty, 3 mma wait-full, 4 mma total,
//              5 epilogue(warp 2) wait-tmem-full, 6 epilogue total, 7 tiles processed

__device__ __forceinline__ void epi_bar_sync() { asm volatile("bar.sync 1, %0;" ::"n"(EPI_WARPS * 32) : "memory"); }

template <int BN, bool GN>
struct TcCfg {
  static constexpr int B_BYTES = BN * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = GN ? 3 : ((BN == 256) ? 4 : 6);   // GN: 3 x 48 KB leaves room for its tables
  static constexpr int TMEM_COLS = 2 * BN;                      // two accumulator buffers (256 or 512 columns)
  // epilogue scratch: per-column constants (bias, gamma, beta, -) + GroupNorm partials and statistics
  // per-column constants for ALL N columns of the GEMM, staged once per CTA:
  //   GN: float4 (bias, gamma, beta, -) for N <= 512;  plain: float bias for N <= 4096
  static constexpr int CHAN_MAX_N = GN ? 512 : 4096;
  // GN: bias[N] floats | (gamma, beta)[N] float2 | batch-uniform FiLM (scale+1, shift)[N] float2  = 20 B / column
  static constexpr int CHAN_BYTES = GN ? CHAN_MAX_N * 20 : CHAN_MAX_N * 4;
  static constexpr int PART_BYTES = GN ? BM * 4 * 8 : 0;
  static constexpr int SPT_FAST = 10;                    // folded-coefficient fast path: <= 10 scenes per tile
  static constexpr int AB_BYTES = BN * SPT_FAST * 8;     // folded (A, B) coefficients [column][scene]
  static constexpr int STAGING_BYTES = EPI_WARPS * 32 * 64;   // per epilogue warp: 32 rows x 32 bf16, 64B-swizzled
  // second region: coefficient double-buffer (per-scene FiLM prefetch) OR the per-object FiLM table (context blocks)
  static constexpr int AUX_BYTES = 32000;
  static constexpr int OBJ_MAX = AUX_BYTES / (BN * 4);   // objects per scene supported by the packed table (31)
  static constexpr int GN_BYTES = GN ? PART_BYTES + 512 + AB_BYTES + AUX_BYTES : 0;
  static constexpr int SCRATCH_OFF = STAGES * STAGE_BYTES + 256;          // barriers occupy the 256 bytes before it
  static constexpr int STAGING_OFF = ((SCRATCH_OFF + CHAN_BYTES + GN_BYTES + 1023) / 1024) * 1024;   // swizzle-atom aligned
  static constexpr int SMEM_BYTES = 1024 /*align slack*/ + STAGING_OFF + STAGING_BYTES;
  static_assert(SMEM_BYTES <= 232448, "shared memory budget exceeded");
  static_assert(!GN || AUX_BYTES >= AB_BYTES, "aux region doubles as the second coefficient buffer");
  // instruction descriptor: D=f32, A=B=bf16, both K-major, N>>3 at bit 17, M>>4 at bit 24
  static constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(BN >> 3) << 17) |
                                    (uint32_t(BM >> 4) << 24);
  // CTA pair (cta_group::2): M = 256 = the two CTAs' token tiles, N = BN (half of the weight tile's rows in each CTA)
  static constexpr uint32_t IDESC_2SM = (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(BN >> 3) << 17) |
                                        (uint32_t((2 * BM) >> 4) << 24);
  static constexpr int STAGE_BYTES_2SM = A_BYTES + B_BYTES / 2;
  static constexpr int STAGE_TX_2SM = 2 * STAGE_BYTES_2SM;
  static constexpr int MAX_STAGES = 6;       // barrier slots reserved behind the ring
  static constexpr int STAGES_2SM = (STAGES * STAGE_BYTES) / STAGE_BYTES_2SM < MAX_STAGES ? (STAGES * STAGE_BYTES) / STAGE_BYTES_2SM : MAX_STAGES;
  static_assert(STAGES <= MAX_STAGES && STAGE_BYTES_2SM % 1024 == 0, "ring geometry");
};

// TWO: the CTA-pair instantiation (see k_gemm_gnt): one tcgen05.mma.cta_group::2 of M = 256 covers the two consecutive
// token tiles of a cluster of 2; each CTA loads its own token tile and HALF of the weight tile, the even CTA issues.
// Per CTA and k-block 32 KB instead of 48 KB come from L2 for the same MMA work (BN = 256) and the ring holds 6 stages.
template <int BN, bool GN, bool TWO = false>
// 10 warps occupy 12 warp slots of the register file (allocation is per 4 warps): 65536 / (12 * 32) = 170 registers
__global__ void __launch_bounds__(TC_THREADS, 1)
k_gemm_tc(const __grid_constant__ CUtensorMap tm_a0, const __grid_constant__ CUtensorMap tm_a1,
          const __grid_constant__ CUtensorMap tm_w, TcEpi epi, int* err_flag) {
  using Cfg = TcCfg<BN, GN>;
  static_assert(!GN || BN == 256, "the GroupNorm epilogue owns 4 groups of 64 channels per tile");
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* const base_ptr = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t bar_base = base + Cfg::STAGES * Cfg::STAGE_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (Cfg::MAX_STAGES + s); };
  auto tfull_bar = [&](int b) { return bar_base + 8u * (2 * Cfg::MAX_STAGES + b); };
  auto tempty_bar = [&](int b) { return bar_base + 8u * (2 * Cfg::MAX_STAGES + 2 + b); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * Cfg::MAX_STAGES + 4);
  uint8_t* const scratch = base_ptr + Cfg::SCRATCH_OFF;
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(base_ptr + (tmem_slot - base));
  float* const bias_s = reinterpret_cast<float*>(scratch);          // [N] bias (both epilogues)
  float2* const gb_s = reinterpret_cast<float2*>(scratch + Cfg::CHAN_MAX_N * 4);     // GN: [N] (gamma, beta)
  float2* const film_u = reinterpret_cast<float2*>(scratch + Cfg::CHAN_MAX_N * 12);  // GN: [N] uniform-t FiLM
  float2* const part = reinterpret_cast<float2*>(scratch + Cfg::CHAN_BYTES);            // [128 rows][4 groups]
  float2* const stat = reinterpret_cast<float2*>(scratch + Cfg::CHAN_BYTES + Cfg::PART_BYTES);   // [scene][4]
  float2* const coef = reinterpret_cast<float2*>(scratch + Cfg::CHAN_BYTES + Cfg::PART_BYTES + 512);   // [col][scene]
  uint8_t* const aux = scratch + Cfg::CHAN_BYTES + Cfg::PART_BYTES + 512 + (GN ? Cfg::AB_BYTES : 0);
  uint32_t* const film_o = reinterpret_cast<uint32_t*>(aux);       // [col][obj] packed bf16x2 (scale + 1, shift)

  const int warp = uniform_warp_idx(), lane = threadIdx.x & 31;
  // programmatic dependent launch: let the next kernel's CTAs be scheduled as SMs drain (its prologue overlaps
  // our tail); our own dependent work starts only after griddepcontrol.wait below
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  // cluster: 1 CTA, or the CTA pair (TWO), whose CTAs work on the 2 consecutive M tiles of the same N tile
  const uint32_t cs = cluster_nctarank();
  const uint32_t crank = cluster_ctarank();

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_a0);
    tma_prefetch_desc(&tm_a1);
    tma_prefetch_desc(&tm_w);
    // CTA pair: full[] and tempty[] are used in the leader only (its own expect_tx covers both CTAs' bytes; 2 x 8
    // epilogue warps arrive on its tempty), empty[] / tfull[] get one arrival each from the leader's multicast commits
    for (int s = 0; s < Cfg::MAX_STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(tfull_bar(b), 1);
      mbar_init(tempty_bar(b), TWO ? 2 * EPI_WARPS : EPI_WARPS);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {
    if constexpr (TWO) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot),
                   "n"(Cfg::TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot),
                   "n"(Cfg::TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  constexpr int nst = TWO ? Cfg::STAGES_2SM : Cfg::STAGES;
  constexpr uint32_t stb = TWO ? uint32_t(Cfg::STAGE_BYTES_2SM) : uint32_t(Cfg::STAGE_BYTES);
  tc_fence_before();
  __syncthreads();
  if (cs > 1) cluster_sync_all();        // peers' barriers are initialised before anyone signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  // everything above touched no activation memory; from here on we read / write buffers of earlier kernels
  asm volatile("griddepcontrol.wait;" ::: "memory");

  const int num_m = (epi.M + epi.tile_rows - 1) / epi.tile_rows;
  const int num_n = epi.N / BN;
  const int num_mg = (num_m + int(cs) - 1) / int(cs);          // groups of CS consecutive M tiles
  const int ksplit = epi.ksplit > 1 ? epi.ksplit : 1;
  const int tiles_mn = num_mg * num_n;
  const int total = tiles_mn * ksplit;                          // work units: (cluster tile, K split)
  const int cluster_id = blockIdx.x / cs, num_clusters = gridDim.x / cs;
  const int kblocks = epi.kb0 + epi.kb1;
  const int kb_per = (kblocks + ksplit - 1) / ksplit;

  if (warp == 0) {
    // TMA producer: the whole warp walks the loop, one elected lane issues (see tc_common.cuh)
    int stage = 0;
    uint32_t phase = 0;
    unsigned long long tw = 0, tstart = clock64();
    for (int unit = cluster_id; unit < total; unit += num_clusters) {
      const int tile = unit % tiles_mn, kb_lo = (unit / tiles_mn) * kb_per, kb_hi = min(kblocks, kb_lo + kb_per);
      const int n_idx = tile % num_n, m_idx = (tile / num_n) * int(cs) + int(crank);   // N fastest: neighbours share A in L2
      const int m0 = m_idx * epi.tile_rows;
      for (int kb = kb_lo; kb < kb_hi; ++kb) {
        unsigned long long t0 = epi.trace ? clock64() : 0;
        mbar_wait(empty_bar(stage), phase ^ 1u, err_flag, 1);
        if (epi.trace) tw += clock64() - t0;
        const uint32_t sa = base + stage * stb;
        if constexpr (TWO) {      // CTA pair: own token tile + own half of the weight tile, bytes counted on the leader
          if (crank == 0) mbar_expect_tx_elect(full_bar(stage), Cfg::STAGE_TX_2SM);
          if (kb < epi.kb0) tma_load_2d_2sm_elect(sa, &tm_a0, kb * BK, m0, full_bar(stage));
          else tma_load_2d_2sm_elect(sa, &tm_a1, (kb - epi.kb0) * BK, m0, full_bar(stage));
          tma_load_2d_2sm_elect(sa + A_BYTES, &tm_w, kb * BK, n_idx * BN + int(crank) * (BN / 2), full_bar(stage));
        } else {
          mbar_expect_tx_elect(full_bar(stage), Cfg::STAGE_BYTES);
          if (kb < epi.kb0) tma_load_2d_elect(sa, &tm_a0, kb * BK, m0, full_bar(stage));
          else tma_load_2d_elect(sa, &tm_a1, (kb - epi.kb0) * BK, m0, full_bar(stage));
          tma_load_2d_elect(sa + A_BYTES, &tm_w, kb * BK, n_idx * BN, full_bar(stage));
        }
        if (++stage == nst) { stage = 0; phase ^= 1u; }
      }
    }
    if (epi.trace && lane == 0) {
      epi.trace[blockIdx.x * 8 + 0] = tw;
      epi.trace[blockIdx.x * 8 + 1] = clock64() - tstart;
    }
  } else if (warp == 1) {
    // MMA issuer (CTA pair: the even CTA issues for both)
    if (!TWO || crank == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int ab = 0;
      uint32_t aphase = 0;
      unsigned long long tw_te = 0, tw_f = 0, tstart = clock64();
      for (int unit = cluster_id; unit < total; unit += num_clusters) {
        const int kb_lo = (unit / tiles_mn) * kb_per, kb_hi = min(kblocks, kb_lo + kb_per);
        unsigned long long t0 = epi.trace ? clock64() : 0;
        mbar_wait(tempty_bar(ab), aphase ^ 1u, err_flag, 2);
        if (epi.trace) tw_te += clock64() - t0;
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + uint32_t(ab * BN);
        for (int kb = kb_lo; kb < kb_hi; ++kb) {
          t0 = epi.trace ? clock64() : 0;
          mbar_wait(full_bar(stage), phase, err_flag, 3);
          if (epi.trace) tw_f += clock64() - t0;
          tc_fence_after();
          const uint32_t sa = base + stage * stb;
          const uint64_t adesc = umma_desc(sa, epi.desc_hi);
          const uint64_t bdesc = umma_desc(sa + A_BYTES, epi.desc_hi);
          // advance 16 elements (32 bytes) along K inside the 128-byte swizzle row: +2 in 16-byte units
          if constexpr (TWO) {
#pragma unroll
            for (int k = 0; k < BK / 16; ++k)
              umma_issue_2sm_elect(d_tmem, adesc + uint64_t(2 * k), bdesc + uint64_t(2 * k), Cfg::IDESC_2SM, ((kb - kb_lo) | k) != 0);
            umma_arrive_2sm_mc_elect(empty_bar(stage), 3);     // the slot is free in BOTH CTAs
          } else {
#pragma unroll
            for (int k = 0; k < BK / 16; ++k)
              umma_issue_elect(d_tmem, adesc + uint64_t(2 * k), bdesc + uint64_t(2 * k), epi.idesc, ((kb - kb_lo) | k) != 0);
            umma_arrive_elect(empty_bar(stage));     // smem slot reusable once these MMAs have read it
          }
          if (++stage == nst) { stage = 0; phase ^= 1u; }
        }
        if constexpr (TWO) umma_arrive_2sm_mc_elect(tfull_bar(ab), 3);     // both CTAs' halves are complete
        else umma_arrive_elect(tfull_bar(ab));               // accumulator complete -> epilogue
        if (++ab == 2) { ab = 0; aphase ^= 1u; }
      }
      if (epi.trace && lane == 0) {
        epi.trace[blockIdx.x * 8 + 2] = tw_te;
        epi.trace[blockIdx.x * 8 + 3] = tw_f;
        epi.trace[blockIdx.x * 8 + 4] = clock64() - tstart;
      }
    }
  } else {
    // ---------------- epilogue warps ----------------
    const int q = warp & 3;                        // TMEM lane quadrant this warp may access
    const int hh = (warp - 2) >> 2;                // which half of the tile's columns this warp owns
    const int etid = threadIdx.x - 64;             // 0..255
    const int row_in_tile = q * 32 + lane;
    constexpr int HALF = BN / 2;
    constexpr int CHUNKS = HALF / 32;
    int ab = 0;
    uint32_t aphase = 0;
    // GN: row -> (scene slot, row in scene); constant per thread
    const int sc_local = GN ? row_in_tile / epi.n_obj : 0;
    const int r_in_scene = GN ? row_in_tile - sc_local * epi.n_obj : 0;
    const int scenes_per_tile = GN ? epi.tile_rows / epi.n_obj : 0;
    // stage the per-column constants once per CTA
    // film_uniform: every scene of the launch has the same timestep (the sampling loop), so the per-scene FiLM row
    // is one row for the whole kernel and is staged here instead of being fetched per tile
    const bool film_uni = GN && epi.film.mode == FILM_TIME && epi.film_uniform;
    // per-object FiLM (context blocks with a batch-shared condition): constant over tiles -> packed table in smem,
    // (re)built whenever this CTA moves to another N tile (never, when the grid size is even)
    const bool film_obj = GN && epi.film.mode == FILM_OBJECT && epi.n_obj <= Cfg::OBJ_MAX;
    int film_obj_n = -1;
    const float* fr_u = film_uni ? epi.film.base + (int64_t)__ldg(epi.film.t) * epi.film.row_stride : nullptr;
    for (int n = etid; n < epi.N; n += EPI_WARPS * 32) {
      bias_s[n] = epi.bias ? __ldg(epi.bias + n) : 0.f;
      if constexpr (GN) {
        gb_s[n] = make_float2(__ldg(epi.gamma + n), __ldg(epi.beta + n));
        film_u[n] = film_uni ? make_float2(__ldg(fr_u + n) + 1.0f, __ldg(fr_u + epi.C + n)) : make_float2(1.0f, 0.0f);
      }
    }
    epi_bar_sync();
    // Global traffic goes through a per-warp 32 x 32 (bf16) staging block in shared memory (16-byte pieces
    // XOR-swizzled by (row/2)%4) so that BOTH the residual loads and the output stores are coalesced: one warp
    // instruction moves 8 rows x 64 contiguous bytes.  Two views of the block:
    //   row-owner view  lane = row, pieces g = 0..3            (own_a[g])
    //   coalesced view  instruction i: row 8i + lane/4, piece lane%4   (co_a[i])
    const uint32_t stg = base + uint32_t(Cfg::STAGING_OFF) + uint32_t((warp - 2) * 2048);
    const int co_r = lane >> 2, co_p = lane & 3;
    uint32_t own_a[4], co_a[4];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      own_a[g] = stg + uint32_t(lane * 64) + ((uint32_t(g) ^ uint32_t((lane >> 1) & 3)) << 4);
      const int r = g * 8 + co_r;
      co_a[g] = stg + uint32_t(r * 64) + ((uint32_t(co_p) ^ uint32_t((r >> 1) & 3)) << 4);
    }
    const int rows_q = min(32, max(0, epi.tile_rows - q * 32));          // rows of this quadrant inside a tile
    auto sts128 = [](uint32_t a, const uint4& v) {
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
    };
    auto lds128 = [](uint32_t a) {
      uint4 v;
      asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
      return v;
    };
    unsigned long long tw_tf = 0, tstart = clock64(), ntiles = 0;
    int tile_par = 0;
    for (int unit = cluster_id; unit < total; unit += num_clusters) {
      const int tile = unit % tiles_mn;
      const int n_idx = tile % num_n, m_idx = (tile / num_n) * int(cs) + int(crank);   // N fastest: neighbours share A in L2
      const int m0 = m_idx * epi.tile_rows;
      const int m = m0 + row_in_tile;
      const bool row_ok = row_in_tile < epi.tile_rows && m < epi.M;
      float2* const cf = (tile_par && !film_obj) ? reinterpret_cast<float2*>(aux) : coef;   // this tile's coefficient table
      tile_par ^= 1;
      if (epi.res && row_ok) {
        // pull this row's residual segment (HALF bf16 = 1-2 cache lines) towards L2 while the MMAs run
        const char* rp = reinterpret_cast<const char*>(epi.res + (int64_t)m * epi.ldres + n_idx * BN + hh * HALF);
#pragma unroll
        for (int b = 0; b < HALF * 2; b += 128) asm volatile("prefetch.global.L2 [%0];" ::"l"(rp + b));
      }
      if (film_obj && film_obj_n != n_idx) {
        epi_bar_sync();                          // nobody still reads the previous table
        for (int i = etid; i < BN * epi.n_obj; i += EPI_WARPS * 32) {
          const int col = i % BN, ob = i / BN;
          const float* fr = epi.film.base + (int64_t)ob * epi.film.row_stride + n_idx * BN + col;
          __nv_bfloat162 h2 = __floats2bfloat162_rn(0.5f * (__ldg(fr) + 1.0f), 0.5f * __ldg(fr + epi.C));   // halved: see SiLU
          film_o[col * epi.n_obj + ob] = *reinterpret_cast<uint32_t*>(&h2);
        }
        film_obj_n = n_idx;                      // visible to the readers after the barriers of the statistics pass
      }
      if constexpr (GN) {
        // While the MMAs of this tile are still running: fetch the per-scene FiLM (scale + 1, shift) of this
        // thread's column for every scene of the tile -- all loads independent, two round trips in total -- and
        // park them in the (double-buffered) coefficient table, where the same thread folds them in later.
        const int col = etid, n = n_idx * BN + col;
        const int n_scenes_total = epi.M / epi.n_obj;
        if (epi.film.mode == FILM_TIME && !film_uni) {
          int tt[Cfg::SPT_FAST];
#pragma unroll
          for (int sc = 0; sc < Cfg::SPT_FAST; ++sc) {
            const int scene_g = m_idx * scenes_per_tile + sc;
            tt[sc] = (sc < scenes_per_tile && scene_g < n_scenes_total) ? __ldg(epi.film.t + scene_g) : -1;
          }
          float2 fv[Cfg::SPT_FAST];
#pragma unroll
          for (int sc = 0; sc < Cfg::SPT_FAST; ++sc) {
            fv[sc] = make_float2(1.0f, 0.0f);
            if (tt[sc] >= 0) {
              const float* fr = epi.film.base + (int64_t)tt[sc] * epi.film.row_stride;
              fv[sc] = make_float2(__ldg(fr + n) + 1.0f, __ldg(fr + epi.C + n));
            }
          }
#pragma unroll
          for (int sc = 0; sc < Cfg::SPT_FAST; ++sc)
            if (sc < scenes_per_tile) cf[col * Cfg::SPT_FAST + sc] = fv[sc];
        }
      }
      unsigned long long t0 = epi.trace ? clock64() : 0;
      mbar_wait(tfull_bar(ab), aphase, err_flag, 4);
      if (epi.trace) { tw_tf += clock64() - t0; ++ntiles; }
      tc_fence_after();
      const uint32_t taddr0 = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(ab * BN + hh * HALF);

      const int nbase = n_idx * BN + hh * HALF;     // first global column this warp owns in this tile
      // ---- shared pieces of both epilogues -------------------------------------------------------------------
      // per-tile addresses of the coalesced view (4 instructions x 8 rows): predicate, output / residual pointers
      bool ok4[4];
      bf16* dp4[4];
      const bf16* rp4[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int r = i * 8 + co_r;
        ok4[i] = r < rows_q && m0 + q * 32 + r < epi.M;
        dp4[i] = epi.d + (int64_t)(m0 + q * 32 + r) * epi.ldd + nbase + co_p * 8;
        rp4[i] = epi.res ? epi.res + (int64_t)(m0 + q * 32 + r) * epi.ldres + nbase + co_p * 8 : nullptr;
      }
      // coalesced residual fetch for chunk c (issued one chunk ahead of its use)
      auto fetch_res = [&](uint4 (&rg)[4], int c) {
        if (epi.res) {
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            rg[i] = make_uint4(0u, 0u, 0u, 0u);
            // plain (coherent) load, not __ldg: the backward GEMMs accumulate in place (res == d), every address is
            // read and later written by the same lane
            if (ok4[i]) rg[i] = *reinterpret_cast<const uint4*>(rp4[i] + c * 32);
          }
        }
      };
      // v (this lane's row, 32 columns of chunk c) += residual; -> bf16 -> coalesced store
      auto emit = [&](float (&v)[32], const uint4 (&rg)[4], int c) {
        if (epi.res) {
#pragma unroll
          for (int i = 0; i < 4; ++i) sts128(co_a[i], rg[i]);
          __syncwarp();
#pragma unroll
          for (int g = 0; g < 4; ++g) {
            const uint4 rv = lds128(own_a[g]);
            const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&rv);
#pragma unroll
            for (int e = 0; e < 4; ++e) {
              float2 f = __bfloat1622float2(h2[e]);
              v[g * 8 + e * 2] += f.x;
              v[g * 8 + e * 2 + 1] += f.y;
            }
          }
          __syncwarp();
        }
#pragma unroll
        for (int g = 0; g < 4; ++g) {
          uint4 o;
          __nv_bfloat162* h2 = reinterpret_cast<__nv_bfloat162*>(&o);
#pragma unroll
          for (int e = 0; e < 4; ++e) h2[e] = __floats2bfloat162_rn(v[g * 8 + e * 2], v[g * 8 + e * 2 + 1]);
          sts128(own_a[g], o);
        }
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const uint4 o = lds128(co_a[i]);
          if (ok4[i]) *reinterpret_cast<uint4*>(dp4[i] + c * 32) = o;
        }
        __syncwarp();
      };
      auto release_tmem = [&]() {
        tc_fence_before();
        __syncwarp();
        // accumulator buffer free: the next tile's MMAs may start (CTA pair: counted on the leader's barrier)
        if (lane == 0) { if constexpr (TWO) mbar_arrive_leader(tempty_bar(ab)); else mbar_arrive(tempty_bar(ab)); }
        if (++ab == 2) { ab = 0; aphase ^= 1u; }
      };

      if constexpr (GN) {
        // ---- pass 1: per-row partial (sum, sum of squares) of the two 64-channel groups this warp owns;
        //      TMEM loads are software-pipelined (next chunk in flight while this one is reduced)
        {
          uint32_t ra[32], rb[32];
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
          tmem_ld32_issue(taddr0, ra);
          tmem_ld_wait();
          tmem_ld32_issue(taddr0 + 32u, rb);
          acc(ra, 0);
          tmem_ld_wait();
          tmem_ld32_issue(taddr0 + 64u, ra);
          acc(rb, 1);
          part[row_in_tile * 4 + hh * 2] = make_float2(s, ss);
          s = 0.f; ss = 0.f;
          tmem_ld_wait();
          tmem_ld32_issue(taddr0 + 96u, rb);
          acc(ra, 2);
          tmem_ld_wait();
          acc(rb, 3);
          part[row_in_tile * 4 + hh * 2 + 1] = make_float2(s, ss);
        }
        epi_bar_sync();
        if (etid < scenes_per_tile * 4) {
          const int sc = etid >> 2, g = etid & 3;
          float s = 0.f, ss = 0.f;
          for (int r = 0; r < epi.n_obj; ++r) {
            float2 p2 = part[(sc * epi.n_obj + r) * 4 + g];
            s += p2.x;
            ss += p2.y;
          }
          const float inv = 1.0f / float(epi.n_obj * 64);
          const float mean = s * inv;
          const float var = fmaxf(ss * inv - mean * mean, 0.f);
          stat[etid] = make_float2(mean, rsqrtf(var + 1e-5f));
        }
        epi_bar_sync();
        // fold bias, statistics, affine and per-scene FiLM into y = acc * A + B per (column, scene)
        {
          const int col = etid;                      // 256 epilogue threads <-> 256 tile columns
          const int n = n_idx * BN + col;
          const float2 gb = gb_s[n];
          const float bias = bias_s[n];
          const bool per_scene = epi.film.mode == FILM_TIME && !film_uni;
          // with the per-object table the halving lives in that table; the generic per-row path halves at the end
          const float half_scale = (film_obj || epi.film.mode == FILM_TOKEN || (epi.film.mode == FILM_OBJECT && !film_obj)) ? 1.0f : 0.5f;
          const float2 fu = film_u[n];                                // (1, 0) unless the timestep is batch-uniform
#pragma unroll
          for (int sc = 0; sc < Cfg::SPT_FAST; ++sc) {
            if (sc < scenes_per_tile) {
              const float2 st = stat[sc * 4 + (col >> 6)];
              const float2 f = per_scene ? cf[col * Cfg::SPT_FAST + sc] : fu;   // per-scene rows parked at tile start
              const float a = st.y * gb.x;
              const float b = fmaf(bias - st.x, a, gb.y);
              // `half_scale`: the table produces y / 2 directly (SiLU's tanh form wants x / 2)
              cf[col * Cfg::SPT_FAST + sc] = make_float2(a * f.x * half_scale, fmaf(b, f.x, f.y) * half_scale);
            }
          }
        }
        epi_bar_sync();

        // ---- pass 2: re-read the accumulator, one FMA + SiLU per element, residual, coalesced store
        const float* frow = nullptr;                  // per-object / per-token FiLM rows (context blocks)
        if (row_ok && !film_obj && (epi.film.mode == FILM_OBJECT || epi.film.mode == FILM_TOKEN))
          frow = epi.film.base + (int64_t)(epi.film.mode == FILM_OBJECT ? r_in_scene : m) * epi.film.row_stride;
        const uint32_t* fo = film_o + (hh * HALF) * epi.n_obj + r_in_scene;
        const float2* cb = cf + (hh * HALF) * Cfg::SPT_FAST + (row_in_tile < epi.tile_rows ? sc_local : 0);
        uint32_t ra[32], rb[32];
        uint4 rga[4], rgb[4];
        auto finish = [&](const uint32_t (&r)[32], int c, const uint4 (&rcur)[4], uint4 (&rnext)[4]) {
          if (c + 1 < CHUNKS) fetch_res(rnext, c + 1);
          float v[32];
          const float2* cc = cb + c * 32 * Cfg::SPT_FAST;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const float2 k2 = cc[j * Cfg::SPT_FAST];
            v[j] = fmaf(__uint_as_float(r[j]), k2.x, k2.y);
          }
          if (film_obj) {
            const uint32_t* fc = fo + c * 32 * epi.n_obj;
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const uint32_t pkd = fc[j * epi.n_obj];
              const float2 f = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&pkd));
              v[j] = fmaf(v[j], f.x, f.y);
            }
          } else if (frow) {
            const int n0 = nbase + c * 32;
#pragma unroll
            for (int j = 0; j < 32; ++j)
              v[j] = 0.5f * fmaf(v[j], __ldg(frow + n0 + j) + 1.0f, __ldg(frow + epi.C + n0 + j));
          }
#pragma unroll
          for (int j = 0; j < 32; ++j) v[j] = silu_from_half(v[j]);
          emit(v, rcur, c);
        };
        fetch_res(rga, 0);
        tmem_ld32_issue(taddr0, ra);
        tmem_ld_wait();
        tmem_ld32_issue(taddr0 + 32u, rb);
        finish(ra, 0, rga, rgb);
        tmem_ld_wait();
        tmem_ld32_issue(taddr0 + 64u, ra);
        finish(rb, 1, rgb, rga);
        tmem_ld_wait();
        tmem_ld32_issue(taddr0 + 96u, rb);
        finish(ra, 2, rga, rgb);
        tmem_ld_wait();
        release_tmem();
        finish(rb, 3, rgb, rga);
      } else {
        // ---- plain epilogue: bias, activation, residual (TMEM loads software-pipelined)
        uint32_t ra[32], rb[32];
        uint4 rga[4], rgb[4];
        auto finish = [&](const uint32_t (&r)[32], int c, const uint4 (&rcur)[4], uint4 (&rnext)[4]) {
          if (epi.d32) {      // split-K partial sums: fp32 atomics straight from the accumulator (this lane's row)
            if (row_ok) {
              float* op = epi.d32 + (int64_t)m * epi.ldd + nbase + c * 32;      // 16-byte aligned (ldd, nbase multiples of 4)
#pragma unroll
              for (int j = 0; j < 32; j += 4)      // vector reduction: 4 floats per L2 atomic transaction
                asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(op + j), "f"(__uint_as_float(r[j])),
                             "f"(__uint_as_float(r[j + 1])), "f"(__uint_as_float(r[j + 2])), "f"(__uint_as_float(r[j + 3]))
                             : "memory");
            }
            return;
          }
          if (c + 1 < CHUNKS) fetch_res(rnext, c + 1);
          float v[32];
          const float4* b4 = reinterpret_cast<const float4*>(bias_s + nbase + c * 32);
#pragma unroll
          for (int j = 0; j < 8; ++j) {
            const float4 bb = b4[j];
            v[4 * j] = __uint_as_float(r[4 * j]) + bb.x;
            v[4 * j + 1] = __uint_as_float(r[4 * j + 1]) + bb.y;
            v[4 * j + 2] = __uint_as_float(r[4 * j + 2]) + bb.z;
            v[4 * j + 3] = __uint_as_float(r[4 * j + 3]) + bb.w;
          }
          if (epi.act == ACT_GELU) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = gelu_tanh(v[j]);
          } else if (epi.act == ACT_SILU) {
#pragma unroll
            for (int j = 0; j < 32; ++j) v[j] = silu_tanh(v[j]);
          }
          emit(v, rcur, c);
        };
        fetch_res(rga, 0);
        tmem_ld32_issue(taddr0, ra);
        tmem_ld_wait();
#pragma unroll
        for (int c = 0; c < CHUNKS; c += 2) {
          if (c + 1 < CHUNKS) tmem_ld32_issue(taddr0 + uint32_t((c + 1) * 32), rb);
          else release_tmem();
          finish(ra, c, rga, rgb);
          if (c + 1 < CHUNKS) {
            tmem_ld_wait();
            if (c + 2 < CHUNKS) tmem_ld32_issue(taddr0 + uint32_t((c + 2) * 32), ra);
            else release_tmem();
            finish(rb, c + 1, rgb, rga);
            if (c + 2 < CHUNKS) tmem_ld_wait();
          }
        }
      }
    }
    if (epi.trace && warp == 2 && lane == 0) {
      epi.trace[blockIdx.x * 8 + 5] = tw_tf;
      epi.trace[blockIdx.x * 8 + 6] = clock64() - tstart;
      epi.trace[blockIdx.x * 8 + 7] = ntiles;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (cs > 1) cluster_sync_all();        // no CTA leaves while peers may still write its smem / barriers
  if (warp == 1) {
    tc_fence_after();
    if constexpr (TWO) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(Cfg::TMEM_COLS) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(Cfg::TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// GNT: the fused conv + GroupNorm + FiLM + SiLU (+ residual) GEMM with the OUTPUT CHANNELS on the TMEM lanes
// ------------------------------------------------------------------------------------------------
// D^T[channel, token] = W[channel, K] * X[token, K]^T : the weight tile (128 channels) is the M operand, a run of
// whole scenes (SC scenes = TOK tokens) is the N operand.  An epilogue thread therefore owns ONE channel and walks
// over tokens, which removes everything that made the row-major epilogue expensive:
//   * bias, gamma, beta and the (batch-uniform) FiLM pair of the channel live in registers -- no per-element
//     shared-memory coefficient loads, no per-tile coefficient table;
//   * the conv bias never has to be added per element: the statistics of (acc + b) follow from sum(acc) and
//     sum(acc^2) of the channel over the 12 tokens of a scene;
//   * a scene is 12 consecutive TMEM columns, so the normalisation constants are per-(thread, scene) scalars.
// The price is a transposed store: values are packed as (token j, token j+1) pairs and written with
// stmatrix.trans into a [token][32 channel] staging block (ldmatrix.trans for the residual), which needs the
// lanes of a warp to hold the channels in the order 8 (lane % 4) + lane / 4.  The host stores the weight rows of
// these convs in exactly that order inside every block of 32 (ds_commit_weights), so the shuffle costs nothing.
// GroupNorm statistics: per-(scene, channel) partials -> shared memory -> 8 threads per (scene, group) reduce.
template <int NOBJ, bool PAIR = true>
struct GntCfg {
  // scenes per tile: 16 for N = 12 (UMMA N = 192), 12 for N = 21 (252 -> 256)
  static constexpr int SC = (NOBJ == 12) ? 16 : 256 / NOBJ;
  static constexpr int TOK = SC * NOBJ;                         // tokens per tile (192 / 252)
  static constexpr int UN = (TOK + 15) / 16 * 16;               // UMMA N = TMA box rows of the activation tile
  static constexpr int EPI_W = 16;                              // epilogue warps: 4 per TMEM lane quadrant
  static constexpr int NP = EPI_W / 4;                          // each quadrant's warps split the scenes NP ways
  static constexpr int SPP = SC / NP;                           // scenes per warp and tile
  static constexpr int THREADS = 64 + EPI_W * 32;
  static constexpr int B_BYTES = UN * BK * 2;
  static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
  static constexpr int STAGES = (UN <= 192) ? 4 : 3;
  static constexpr int ACC_STRIDE = 256;                        // TMEM columns between the two accumulators
  static constexpr int TMEM_COLS = 512;
  static constexpr int CHAN_MAX_N = 512;
  static constexpr int CHAN_BYTES = CHAN_MAX_N * 20;            // bias | (gamma, beta) | uniform FiLM
  // PAIR: [tile parity][warp pair][scene][S, SS of both warps] floats;  else (sum, sum of squares) per (scene, channel)
  // and (mean, rstd) per (scene, group of the tile), reduced behind two CTA-wide barriers
  static constexpr int RED_BYTES = PAIR ? 2 * 8 * 4 * 4 * 4 : SC * 128 * 8;
  static constexpr int STAT_BYTES = PAIR ? 0 : SC * 2 * 8;
  // a scene is moved as NPAIR (token 2i, token 2i + 1) pairs; an odd scene pads its last pair with a dummy token
  static constexpr int NPAIR = (NOBJ + 1) / 2;
  static constexpr int NG4 = NPAIR / 4;                         // full ldmatrix / stmatrix .x4 groups (8 tokens each)
  static constexpr int REM = NPAIR % 4;                         // 0, 2 (-> .x2) or 3 (-> .x4 with a zero pair)
  static constexpr int PKN = 4 * NG4 + (REM == 0 ? 0 : (REM <= 2 ? 2 : 4));
  static constexpr int PIECES = NOBJ * 4;                       // 16-byte pieces of a [token][32 channel] block
  static constexpr int PROUNDS = (PIECES + 31) / 32;
  static constexpr int STG_ROWS = 8 * (NG4 + 1);                // ldmatrix row addresses stay inside the block
  static constexpr int STG_BYTES = STG_ROWS * 64;               // one [token][32 channel] bf16 block
  static constexpr int SCRATCH_OFF = STAGES * STAGE_BYTES + 256;
  static constexpr int RED_OFF = SCRATCH_OFF + CHAN_BYTES;
  static constexpr int STAT_OFF = RED_OFF + RED_BYTES;
  static constexpr int STG_OFF = (STAT_OFF + STAT_BYTES + 127) / 128 * 128;
  static constexpr int SMEM_BYTES = 1024 + STG_OFF + EPI_W * 2 * STG_BYTES;
  static_assert(SC % NP == 0, "scenes must split evenly over the warps of a quadrant");
  static_assert(STAGE_BYTES % 1024 == 0, "stages must stay swizzle-atom aligned");
  static_assert(SMEM_BYTES <= 232448, "shared memory budget exceeded");
  static_assert(NOBJ == 12 || NOBJ == 21, "TMEM load shapes are written out for N = 12 and N = 21");
  static_assert(REM != 1, "a single trailing pair would need an .x1 matrix");
  static_assert(UN <= 256 && 2 * UN <= TMEM_COLS + (ACC_STRIDE - UN), "accumulators must fit TMEM");
  static constexpr uint32_t IDESC = (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(UN >> 3) << 17) |
                                    (uint32_t(BM >> 4) << 24);
  // CTA pair (cta_group::2): M = 256 = the two CTAs' channel tiles, N = the whole token tile (half of its rows in each
  // CTA's shared memory)
  static constexpr uint32_t IDESC_2SM = (1u << 4) | (1u << 7) | (1u << 10) | (uint32_t(UN >> 3) << 17) |
                                        (uint32_t((2 * BM) >> 4) << 24);
  static constexpr int STAGE_BYTES_2SM = A_BYTES + B_BYTES / 2;       // per CTA of a pair
  static constexpr int STAGE_TX_2SM = 2 * STAGE_BYTES_2SM;            // bytes both CTAs land per stage (leader's barrier)
  static constexpr int STAGES_2SM = (STAGES * STAGE_BYTES) / STAGE_BYTES_2SM < 6 ? (STAGES * STAGE_BYTES) / STAGE_BYTES_2SM : 6;
  static constexpr int MAX_STAGES = 6;                                // barrier slots reserved (256 bytes behind the ring)
  static_assert(STAGE_BYTES_2SM % 1024 == 0, "pair stages must stay swizzle-atom aligned");
  static_assert(8 * (2 * MAX_STAGES + 5) <= 256, "barrier block");
  static_assert(UN % 16 == 0, "each CTA of a pair holds UN / 2 rows of the token tile (whole 8-row swizzle atoms)");
};

__device__ __forceinline__ void tmem_ld12_issue(uint32_t taddr, uint32_t (&r)[12]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11])
               : "r"(taddr + 8u)
               : "memory");
}
__device__ __forceinline__ void tmem_ld21_issue(uint32_t taddr, uint32_t (&r)[21]) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
                 "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
               : "r"(taddr)
               : "memory");
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x4.b32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19])
               : "r"(taddr + 16u)
               : "memory");
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(r[20]) : "r"(taddr + 20u) : "memory");
}
__device__ __forceinline__ void tmem_ld21_wait(uint32_t (&r)[21]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                 "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20])
               :
               : "memory");
}
// wait for the loads above; the registers are listed as read-write so that the compiler cannot move or copy
// them between the (asynchronous) issue and this point
__device__ __forceinline__ void tmem_ld12_wait(uint32_t (&r)[12]) {
  asm volatile("tcgen05.wait::ld.sync.aligned;"
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                 "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11])
               :
               : "memory");
}
// one scene's columns of the accumulator (N consecutive TMEM columns) -> N registers
__device__ __forceinline__ void tmem_ld_scene_issue(uint32_t taddr, uint32_t (&r)[12]) { tmem_ld12_issue(taddr, r); }
__device__ __forceinline__ void tmem_ld_scene_issue(uint32_t taddr, uint32_t (&r)[21]) { tmem_ld21_issue(taddr, r); }
__device__ __forceinline__ void tmem_ld_scene_wait(uint32_t (&r)[12]) { tmem_ld12_wait(r); }
__device__ __forceinline__ void tmem_ld_scene_wait(uint32_t (&r)[21]) { tmem_ld21_wait(r); }
__device__ __forceinline__ void ldsm_x4_t(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(addr) : "memory");
}
__device__ __forceinline__ void ldsm_x2_t(uint32_t (&r)[2], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.trans.shared.b16 {%0, %1}, [%2];"
               : "=r"(r[0]), "=r"(r[1]) : "r"(addr) : "memory");
}
__device__ __forceinline__ void stsm_x4_t(uint32_t addr, uint32_t r0, uint32_t r1, uint32_t r2, uint32_t r3) {
  asm volatile("stmatrix.sync.aligned.m8n8.x4.trans.shared.b16 [%0], {%1, %2, %3, %4};"
               ::"r"(addr), "r"(r0), "r"(r1), "r"(r2), "r"(r3) : "memory");
}
__device__ __forceinline__ void stsm_x2_t(uint32_t addr, uint32_t r0, uint32_t r1) {
  asm volatile("stmatrix.sync.aligned.m8n8.x2.trans.shared.b16 [%0], {%1, %2};" ::"r"(addr), "r"(r0), "r"(r1) : "memory");
}

// TWO: the CTA-pair instantiation (cta_group::2 instructions; must be launched with a cluster of 2 -- the driver
// refuses a plain launch of a kernel that contains them, so the single-CTA path is a separate instantiation)
template <int NOBJ, bool PAIR, bool TWO = false>
// 18 warps = 5 on the fullest SM sub-partition: 16384 / (5 * 32) = 102 registers per thread at most
__global__ void __maxnreg__(96)
k_gemm_gnt(const __grid_constant__ CUtensorMap tm_w, const __grid_constant__ CUtensorMap tm_x0,
           const __grid_constant__ CUtensorMap tm_x1, TcEpi epi, int* err_flag) {
  using Cfg = GntCfg<NOBJ, PAIR>;
  static_assert(!PAIR || Cfg::SPP <= 4, "the warp-pair statistics exchange packs at most 4 scenes per warp");
  extern __shared__ uint8_t smem_raw[];
  const uint32_t base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* const base_ptr = smem_raw + (base - smem_u32(smem_raw));
  const uint32_t bar_base = base + Cfg::STAGES * Cfg::STAGE_BYTES;
  auto full_bar = [&](int s) { return bar_base + 8u * s; };
  auto empty_bar = [&](int s) { return bar_base + 8u * (Cfg::MAX_STAGES + s); };
  auto tfull_bar = [&](int b) { return bar_base + 8u * (2 * Cfg::MAX_STAGES + b); };
  auto tempty_bar = [&](int b) { return bar_base + 8u * (2 * Cfg::MAX_STAGES + 2 + b); };
  const uint32_t tmem_slot = bar_base + 8u * (2 * Cfg::MAX_STAGES + 4);
  volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(base_ptr + (tmem_slot - base));
  float* const bias_s = reinterpret_cast<float*>(base_ptr + Cfg::SCRATCH_OFF);
  float2* const gb_s = reinterpret_cast<float2*>(base_ptr + Cfg::SCRATCH_OFF + Cfg::CHAN_MAX_N * 4);
  float2* const film_u = reinterpret_cast<float2*>(base_ptr + Cfg::SCRATCH_OFF + Cfg::CHAN_MAX_N * 12);
  // GroupNorm partial sums exchanged between the TWO warps that share a (scene range, group):
  // [tile parity][pair 0..7][scene 0..3][S_q0, SS_q0, S_q1, SS_q1]
  float* const red2 = reinterpret_cast<float*>(base_ptr + Cfg::RED_OFF);
  float2* const red = reinterpret_cast<float2*>(base_ptr + Cfg::RED_OFF);        // !PAIR layout
  float2* const stat = reinterpret_cast<float2*>(base_ptr + Cfg::STAT_OFF);

  const int warp = uniform_warp_idx(), lane = threadIdx.x & 31;
  asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  const uint32_t cs = cluster_nctarank();
  const uint32_t crank = cluster_ctarank();
  // CTA pair (TWO, cluster of 2): ONE tcgen05.mma.cta_group::2 of M = 256 covers both CTAs' channel tiles
  // of the same token tile.  Each CTA loads its own weight tile and HALF of the token tile (224 KB instead of 320 KB
  // from L2 per tile pair-half, and the tensor core reads 7 KB instead of 10 KB of shared memory per MMA and SM); the
  // even CTA issues the MMAs for the pair, and every pipeline barrier that gates them lives in that CTA:
  //   full[s]    leader only: 1 arrival (its own producer, expect_tx = both CTAs' bytes); the peer's TMA completes on it
  //   empty[s]   both CTAs: 1 arrival each from the leader's multicast commit
  //   tfull[b]   both CTAs: 1 arrival each from the leader's multicast commit
  //   tempty[b]  leader only: 2 x 16 arrivals (the epilogue warps of both CTAs)
  // operand ring geometry: the CTA pair stages only half of the token tile per CTA, so the same shared memory holds
  // more (smaller) stages
  constexpr int nst = TWO ? Cfg::STAGES_2SM : Cfg::STAGES;
  constexpr uint32_t stb = TWO ? uint32_t(Cfg::STAGE_BYTES_2SM) : uint32_t(Cfg::STAGE_BYTES);
  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tm_w);
    tma_prefetch_desc(&tm_x0);
    tma_prefetch_desc(&tm_x1);
    for (int s = 0; s < Cfg::MAX_STAGES; ++s) {
      mbar_init(full_bar(s), 1);
      mbar_init(empty_bar(s), 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(tfull_bar(b), 1);
      mbar_init(tempty_bar(b), TWO ? 2 * Cfg::EPI_W : Cfg::EPI_W);
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  }
  if (warp == 1) {
    if constexpr (TWO) {       // collective over the pair: warp 1 of both CTAs
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot),
                   "n"(Cfg::TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot),
                   "n"(Cfg::TMEM_COLS)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if (cs > 1) cluster_sync_all();        // peers' barriers are initialised before anyone signals them
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot_ptr;
  asm volatile("griddepcontrol.wait;" ::: "memory");

  const int n_scenes_total = epi.M / NOBJ;
  const int num_tt = (n_scenes_total + Cfg::SC - 1) / Cfg::SC;     // token tiles
  const int num_ct = epi.N / BM;                                    // channel tiles
  // work units: (token tile, group of CS channel tiles); the CTAs of a pair walk the same unit sequence and
  // CTA `crank` takes channel tile group * CS + crank.  CS == 1: unit == tile, exactly the single-CTA schedule.
  const int cgn = num_ct / int(cs);
  const int total = num_tt * cgn;
  const int unit0 = int(blockIdx.x) / int(cs), unit_step = int(gridDim.x) / int(cs);
  const int kblocks = epi.kb0 + epi.kb1;

  if (warp == 0) {
    // TMA producer: the whole warp walks the loop, one elected lane issues (see tc_common.cuh)
    int stage = 0;
    uint32_t phase = 0;
    unsigned long long tw = 0, tstart = clock64();
    for (int tile = unit0; tile < total; tile += unit_step) {
      const int ct = (tile % cgn) * int(cs) + int(crank), tt = tile / cgn;   // channel tiles fastest: neighbours share X
      const int m0 = tt * Cfg::TOK;
      for (int kb = 0; kb < kblocks; ++kb) {
        unsigned long long t0 = epi.trace ? clock64() : 0;
        mbar_wait(empty_bar(stage), phase ^ 1u, err_flag, 1);
        if (epi.trace) tw += clock64() - t0;
        const uint32_t sa = base + stage * stb;
        const CUtensorMap* tmx = kb < epi.kb0 ? &tm_x0 : &tm_x1;
        const int kx = (kb < epi.kb0 ? kb : kb - epi.kb0) * BK;
        if constexpr (TWO) {      // CTA pair: own weight tile + own half of the token tile, bytes counted on the leader's barrier
          if (crank == 0) mbar_expect_tx_elect(full_bar(stage), Cfg::STAGE_TX_2SM);
          tma_load_2d_2sm_elect(sa, &tm_w, kb * BK, ct * BM, full_bar(stage));
          tma_load_2d_2sm_elect(sa + A_BYTES, tmx, kx, m0 + int(crank) * (Cfg::UN / 2), full_bar(stage));
        } else {
          mbar_expect_tx_elect(full_bar(stage), Cfg::STAGE_BYTES);
          tma_load_2d_elect(sa, &tm_w, kb * BK, ct * BM, full_bar(stage));
          tma_load_2d_elect(sa + A_BYTES, tmx, kx, m0, full_bar(stage));
        }
        if (++stage == nst) { stage = 0; phase ^= 1u; }
      }
    }
    if (epi.trace && lane == 0) {
      epi.trace[blockIdx.x * 8 + 0] = tw;
      epi.trace[blockIdx.x * 8 + 1] = clock64() - tstart;
    }
  } else if (warp == 1) {
    // MMA issuer (CTA pair: the even CTA issues for both)
    if (!TWO || crank == 0) {
      int stage = 0;
      uint32_t phase = 0;
      int ab = 0;
      uint32_t aphase = 0;
      unsigned long long tw_te = 0, tw_f = 0, tstart = clock64();
      for (int tile = unit0; tile < total; tile += unit_step) {
        unsigned long long t0 = epi.trace ? clock64() : 0;
        mbar_wait(tempty_bar(ab), aphase ^ 1u, err_flag, 2);
        if (epi.trace) tw_te += clock64() - t0;
        tc_fence_after();
        const uint32_t d_tmem = tmem_base + uint32_t(ab * Cfg::ACC_STRIDE);
        for (int kb = 0; kb < kblocks; ++kb) {
          t0 = epi.trace ? clock64() : 0;
          mbar_wait(full_bar(stage), phase, err_flag, 3);
          if (epi.trace) tw_f += clock64() - t0;
          tc_fence_after();
          const uint32_t sa = base + stage * stb;
          const uint64_t adesc = umma_desc(sa, epi.desc_hi);                // weights: the M operand
          const uint64_t bdesc = umma_desc(sa + A_BYTES, epi.desc_hi);      // activations: the N operand
          if constexpr (TWO) {
#pragma unroll
            for (int k = 0; k < BK / 16; ++k)
              umma_issue_2sm_elect(d_tmem, adesc + uint64_t(2 * k), bdesc + uint64_t(2 * k), Cfg::IDESC_2SM, (kb | k) != 0);
            umma_arrive_2sm_mc_elect(empty_bar(stage), 3);     // the slot is free in BOTH CTAs
          } else {
#pragma unroll
            for (int k = 0; k < BK / 16; ++k)
              umma_issue_elect(d_tmem, adesc + uint64_t(2 * k), bdesc + uint64_t(2 * k), Cfg::IDESC, (kb | k) != 0);
            umma_arrive_elect(empty_bar(stage));     // smem slot reusable once these MMAs have read it
          }
          if (++stage == nst) { stage = 0; phase ^= 1u; }
        }
        if constexpr (TWO) umma_arrive_2sm_mc_elect(tfull_bar(ab), 3);     // both CTAs' halves of the accumulator are complete
        else umma_arrive_elect(tfull_bar(ab));
        if (++ab == 2) { ab = 0; aphase ^= 1u; }
      }
      if (epi.trace && lane == 0) {
        epi.trace[blockIdx.x * 8 + 2] = tw_te;
        epi.trace[blockIdx.x * 8 + 3] = tw_f;
        epi.trace[blockIdx.x * 8 + 4] = clock64() - tstart;
      }
    }
  } else {
    // ---------------- epilogue warps ----------------
    auto epi_bar = []() { asm volatile("bar.sync 1, %0;" ::"n"(Cfg::EPI_W * 32) : "memory"); };
    const int q = warp & 3;                          // TMEM lane quadrant
    const int part = (warp - 2) >> 2;                // which scenes of the tile
    const int etid = threadIdx.x - 64;
    const int chl = 32 * q + 8 * (lane & 3) + (lane >> 2);      // channel (inside the tile) on this thread's lane
    const int pr = part * 2 + (q >> 1);                         // warp pair sharing a (scene range, 64-channel group)
    const bool film_uni = epi.film.mode == FILM_TIME && epi.film_uniform;
    const bool per_scene_t = epi.film.mode == FILM_TIME && !film_uni;
    const float* fr_u = film_uni ? epi.film.base + (int64_t)__ldg(epi.film.t) * epi.film.row_stride : nullptr;
    if (!epi.plain) {      // per-channel tables of the GroupNorm epilogue (N <= 512); plain GEMMs read their bias directly
      for (int n = etid; n < epi.N; n += Cfg::EPI_W * 32) {
        bias_s[n] = epi.bias ? __ldg(epi.bias + n) : 0.f;
        gb_s[n] = make_float2(__ldg(epi.gamma + n), __ldg(epi.beta + n));
        film_u[n] = film_uni ? make_float2(__ldg(fr_u + n) + 1.0f, __ldg(fr_u + epi.C + n)) : make_float2(1.0f, 0.0f);
      }
      epi_bar();
    }
    // staging blocks of this warp: [token][32 channels] bf16, 64 B rows
    const uint32_t stg_in = base + uint32_t(Cfg::STG_OFF) + uint32_t((warp - 2) * 2 * Cfg::STG_BYTES);
    const uint32_t stg_out = stg_in + uint32_t(Cfg::STG_BYTES);
    // ldmatrix / stmatrix row address of this lane: matrix lane / 8 holds tokens 2 (lane / 8) + {0, 1}; its row
    // (lane % 8) = 2 * chunk + e is the 16-byte chunk `chunk` (8 channels) of token 2 (lane / 8) + e
    const uint32_t mrow = uint32_t((2 * (lane >> 3) + (lane & 1)) * 64 + ((lane & 7) >> 1) * 16);
    auto sts128 = [](uint32_t a, const uint4& v) {
      asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
    };
    auto lds128 = [](uint32_t a) {
      uint4 v;
      asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a) : "memory");
      return v;
    };
    // coalesced view of a staging block: 16-byte piece `lane` and (for 12 tokens) `lane + 32` of its 48 pieces
    const int cr0 = lane >> 2, cp0 = lane & 3;
    constexpr bool OBJ_IN_REGS = NOBJ <= 12;         // per-object FiLM pairs of a channel held in registers
    const int s_begin = part * Cfg::SPP;
    // tile walk without divisions: (ct, tt) advance by a constant step with carry
    const int step_cg = unit_step % cgn, step_tt = unit_step / cgn;
    int ab = 0;
    uint32_t aphase = 0;
    unsigned long long tw_tf = 0, tstart = clock64(), ntiles = 0;

    // The tile loop is instantiated per (FiLM mode, residual) so that the per-scene loop carries no mode branches:
    //   FM 0: scene-constant FiLM (none / batch-uniform timestep)   FM 1: per-object FiLM (context blocks)
    //   FM 2: per-token FiLM                                        FM 3: per-scene timestep FiLM
    //   FM 4: no GroupNorm at all (plain GEMM: bias, GELU / SiLU, residual) -- no statistics pass, no barriers
    auto run_tiles = [&](auto fm_tag, auto res_tag) {
      constexpr int FM = decltype(fm_tag)::value;
      constexpr bool RES = decltype(res_tag)::value;
      int cg = unit0 % cgn, tt = unit0 / cgn;
      int tile_par = 0;
      for (int tile = unit0; tile < total; tile += unit_step, tile_par ^= 1) {
        const int ct = cg * int(cs) + int(crank);
        const int ch = ct * BM + chl;
        float bias;
        float2 gb = make_float2(1.0f, 0.0f);
        if constexpr (FM == 4) {
          bias = epi.bias ? __ldg(epi.bias + ch) : 0.f;
        } else {
          bias = bias_s[ch];
          gb = gb_s[ch];
        }
        // scene-constant part of y/2 = (acc + bias - mean) * rstd * P + Q  (FM 1, 2: plain affine, FiLM per element)
        float P = gb.x, Q = gb.y;
        if constexpr (FM == 0) {
          const float2 fu = film_u[ch];
          P = 0.5f * gb.x * fu.x;
          Q = 0.5f * fmaf(gb.y, fu.x, fu.y);
        }
        float Fo[(FM == 1 && OBJ_IN_REGS) ? NOBJ : 1], Go[(FM == 1 && OBJ_IN_REGS) ? NOBJ : 1];   // per-object FiLM
        if constexpr (FM == 1 && OBJ_IN_REGS) {
#pragma unroll
          for (int j = 0; j < NOBJ; ++j) {
            const float* fr = epi.film.base + (int64_t)j * epi.film.row_stride + ch;
            Fo[j] = 0.5f * (__ldg(fr) + 1.0f);
            Go[j] = 0.5f * __ldg(fr + epi.C);
          }
        }
        const int scene0 = tt * Cfg::SC + s_begin;                 // first scene of this warp in this tile
        const int n_live = n_scenes_total - scene0;                // scenes si < n_live exist
        const int col0 = ct * BM + 32 * q + cp0 * 8;
        // piece pointers of scene 0 (rows cr0 + 8 r of the [token][32 channel] block, r = 0..PROUNDS-1); + NOBJ rows per scene
        bf16* dp = epi.d + ((int64_t)scene0 * NOBJ + cr0) * epi.ldd + col0;
        const bf16* rp = RES ? epi.res + ((int64_t)scene0 * NOBJ + cr0) * epi.ldres + col0 : nullptr;
        const int64_t d_step = (int64_t)NOBJ * epi.ldd, r_step = (int64_t)NOBJ * epi.ldres;
        const int64_t d_hi = (int64_t)8 * epi.ldd, r_hi = (int64_t)8 * epi.ldres;
        // residual: software-pipelined one scene ahead; the first fetch is issued before the accumulator is complete
        uint4 rg[Cfg::PROUNDS];
#pragma unroll
        for (int r = 0; r < Cfg::PROUNDS; ++r) rg[r] = make_uint4(0u, 0u, 0u, 0u);
        auto fetch_res = [&]() {
#pragma unroll
          for (int r = 0; r < Cfg::PROUNDS; ++r)
            if (lane + 32 * r < Cfg::PIECES) rg[r] = __ldg(reinterpret_cast<const uint4*>(rp + r * r_hi));
        };
        if constexpr (RES) {
          if (0 < n_live) fetch_res();
        }
        unsigned long long t0 = epi.trace ? clock64() : 0;
        mbar_wait(tfull_bar(ab), aphase, err_flag, 4);
        if (epi.trace) { tw_tf += clock64() - t0; ++ntiles; }
        tc_fence_after();
        const uint32_t taddr = tmem_base + (uint32_t(q * 32) << 16) + uint32_t(ab * Cfg::ACC_STRIDE + s_begin * NOBJ);

        float* const r2 = red2 + ((tile_par * 8 + pr) * 16);
        if constexpr (PAIR) {
        // ---- pass 1: per-(scene, channel) sums of acc and acc^2 over the scene's tokens (bias folded analytically),
        //      reduced over the 32 channels of this warp with a butterfly reduce-scatter (9 shuffles for the 8 values
        //      {sum, sum of squares} x <= 4 scenes), then exchanged with the ONE other warp that holds the rest of the
        //      64-channel group through shared memory and a 64-thread named barrier: no CTA-wide barrier, the 8 warp
        //      pairs of a tile run decoupled from each other
        if constexpr (FM != 4) {
          float v8[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) v8[i] = 0.f;
          uint32_t va[NOBJ];
          tmem_ld_scene_issue(taddr, va);
#pragma unroll
          for (int si = 0; si < Cfg::SPP; ++si) {
            tmem_ld_scene_wait(va);
            float v[NOBJ];
#pragma unroll
            for (int j = 0; j < NOBJ; ++j) v[j] = __uint_as_float(va[j]);
            if (si + 1 < Cfg::SPP) tmem_ld_scene_issue(taddr + uint32_t((si + 1) * NOBJ), va);
            float s1 = 0.f, s2 = 0.f;
#pragma unroll
            for (int j = 0; j < NOBJ; ++j) {
              s1 += v[j];
              s2 = fmaf(v[j], v[j], s2);
            }
            v8[si] = fmaf(float(NOBJ), bias, s1);
            v8[4 + si] = fmaf(bias, fmaf(float(NOBJ), bias, 2.0f * s1), s2);
          }
          {
            const bool up = (lane & 16) != 0;
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float send = up ? v8[i] : v8[i + 4], keep = up ? v8[i + 4] : v8[i];
              v8[i] = keep + __shfl_xor_sync(0xffffffffu, send, 16);
            }
          }
          {
            const bool up = (lane & 8) != 0;
#pragma unroll
            for (int i = 0; i < 2; ++i) {
              const float send = up ? v8[i] : v8[i + 2], keep = up ? v8[i + 2] : v8[i];
              v8[i] = keep + __shfl_xor_sync(0xffffffffu, send, 8);
            }
          }
          {
            const bool up = (lane & 4) != 0;
            const float send = up ? v8[0] : v8[1], keep = up ? v8[1] : v8[0];
            v8[0] = keep + __shfl_xor_sync(0xffffffffu, send, 4);
          }
          v8[0] += __shfl_xor_sync(0xffffffffu, v8[0], 2);
          v8[0] += __shfl_xor_sync(0xffffffffu, v8[0], 1);
          // lane l holds the warp total of value l >> 2: scene (l >> 2) & 3, sum (l < 16) or sum of squares (l >= 16)
          if ((lane & 3) == 0) r2[((lane >> 2) & 3) * 4 + (q & 1) * 2 + (lane >> 4)] = v8[0];
          asm volatile("bar.sync %0, 64;" ::"r"(2 + pr) : "memory");
        }

        } else {
        // ---- pass 1: per-(scene, channel) sums of acc and acc^2 over the scene's tokens, bias folded analytically
        if constexpr (FM != 4) {
          uint32_t va[NOBJ];
          tmem_ld_scene_issue(taddr, va);
          float2* rdst = red + s_begin * 128 + 32 * q + lane;
#pragma unroll
          for (int si = 0; si < Cfg::SPP; ++si) {
            tmem_ld_scene_wait(va);
            float v[NOBJ];
#pragma unroll
            for (int j = 0; j < NOBJ; ++j) v[j] = __uint_as_float(va[j]);
            if (si + 1 < Cfg::SPP) tmem_ld_scene_issue(taddr + uint32_t((si + 1) * NOBJ), va);
            float s1 = 0.f, s2 = 0.f;
#pragma unroll
            for (int j = 0; j < NOBJ; ++j) {
              s1 += v[j];
              s2 = fmaf(v[j], v[j], s2);
            }
            const float S = fmaf(float(NOBJ), bias, s1);
            const float SS = fmaf(bias, fmaf(float(NOBJ), bias, 2.0f * s1), s2);
            rdst[si * 128] = make_float2(S, SS);
          }
        }
        if constexpr (FM != 4) epi_bar();
        if (FM != 4 && etid < Cfg::SC * 2 * 8) {                  // 8 threads per (scene, group): whole warps by construction
          const int pid = etid >> 3, sub = etid & 7;
          const float2* rsrc = red + (pid >> 1) * 128 + (pid & 1) * 64 + sub;
          float s = 0.f, ss = 0.f;
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const float2 p2 = rsrc[8 * i];
            s += p2.x;
            ss += p2.y;
          }
#pragma unroll
          for (int o = 1; o < 8; o <<= 1) {
            s += __shfl_xor_sync(0xffffffffu, s, o);
            ss += __shfl_xor_sync(0xffffffffu, ss, o);
          }
          if (sub == 0) {
            const float inv = 1.0f / float(NOBJ * 64);
            const float mean = s * inv;
            const float var = fmaxf(ss * inv - mean * mean, 0.f);
            stat[pid] = make_float2(mean, rsqrtf(var + 1e-5f));
          }
        }
        if constexpr (FM != 4) epi_bar();

        }
        // ---- pass 2: normalise + FiLM + SiLU (+ residual) per scene, transposed store through the staging blocks
        uint32_t va[NOBJ];
        tmem_ld_scene_issue(taddr, va);
#pragma unroll 1
        for (int si = 0; si < Cfg::SPP; ++si) {
          const bool live = si < n_live;
          float Ps = P, Qs = Q;
          if constexpr (FM == 3) {
            if (live) {
              const float* fr = epi.film.base + (int64_t)__ldg(epi.film.t + scene0 + si) * epi.film.row_stride + ch;
              const float fx = __ldg(fr) + 1.0f, fy = __ldg(fr + epi.C);
              Ps = 0.5f * gb.x * fx;
              Qs = 0.5f * fmaf(gb.y, fx, fy);
            }
          }
          float a = 1.0f, b = bias;
          if constexpr (FM != 4) {
            if constexpr (PAIR) {
              const float4 t4 = reinterpret_cast<const float4*>(r2)[si];
              const float inv = 1.0f / float(NOBJ * 64);
              const float mean = (t4.x + t4.z) * inv;
              const float var = fmaxf((t4.y + t4.w) * inv - mean * mean, 0.f);
              a = rsqrtf(var + 1e-5f) * Ps;
              b = fmaf(bias - mean, a, Qs);
            } else {
              const float2 st = (stat + s_begin * 2 + (q >> 1))[2 * si];
              a = st.y * Ps;
              b = fmaf(bias - st.x, a, Qs);
            }
          }
          float y[2 * Cfg::PKN];                      // tokens >= NOBJ: padding of the last pair(s), never stored
#pragma unroll
          for (int j = NOBJ; j < 2 * Cfg::PKN; ++j) y[j] = 0.f;
          tmem_ld_scene_wait(va);
#pragma unroll
          for (int j = 0; j < NOBJ; ++j) y[j] = FM == 4 ? __uint_as_float(va[j]) + b : fmaf(__uint_as_float(va[j]), a, b);
          if (si + 1 < Cfg::SPP) tmem_ld_scene_issue(taddr + uint32_t((si + 1) * NOBJ), va);
          else {
            tc_fence_before();
            __syncwarp();
            // accumulator drained: the next tile's MMAs may start (CTA pair: counted on the leader's barrier)
            if (lane == 0) { if constexpr (TWO) mbar_arrive_leader(tempty_bar(ab)); else mbar_arrive(tempty_bar(ab)); }
          }
          if constexpr (FM == 1) {
            if constexpr (OBJ_IN_REGS) {
#pragma unroll
              for (int j = 0; j < NOBJ; ++j) y[j] = fmaf(y[j], Fo[j], Go[j]);
            } else {
#pragma unroll
              for (int j = 0; j < NOBJ; ++j) {
                const float* fr = epi.film.base + (int64_t)j * epi.film.row_stride + ch;
                y[j] = 0.5f * fmaf(y[j], __ldg(fr) + 1.0f, __ldg(fr + epi.C));
              }
            }
          }
          if constexpr (FM == 2) {
            if (live) {
#pragma unroll
              for (int j = 0; j < NOBJ; ++j) {
                const float* fr = epi.film.base + ((int64_t)(scene0 + si) * NOBJ + j) * epi.film.row_stride + ch;
                y[j] = 0.5f * fmaf(y[j], __ldg(fr) + 1.0f, __ldg(fr + epi.C));
              }
            }
          }
          if constexpr (FM == 4) {
            if (epi.act == ACT_GELU) {
#pragma unroll
              for (int j = 0; j < NOBJ; ++j) y[j] = gelu_tanh(y[j]);
            } else if (epi.act == ACT_SILU) {
#pragma unroll
              for (int j = 0; j < NOBJ; ++j) y[j] = silu_tanh(y[j]);
            }
          } else {
#pragma unroll
            for (int j = 0; j < NOBJ; ++j) y[j] = silu_from_half(y[j]);
          }
          if constexpr (RES) {
#pragma unroll
            for (int r = 0; r < Cfg::PROUNDS; ++r)
              if (lane + 32 * r < Cfg::PIECES) sts128(stg_in + uint32_t((lane + 32 * r) * 16), rg[r]);
            rp += r_step;
            if (si + 1 < Cfg::SPP && si + 1 < n_live) fetch_res();       // next scene's rows land while this one is finished
            __syncwarp();
            uint32_t rr[Cfg::PKN];
#pragma unroll
            for (int g8 = 0; g8 < Cfg::NG4; ++g8) {
              uint32_t r4[4];
              ldsm_x4_t(r4, stg_in + uint32_t(g8 * 512) + mrow);
              rr[4 * g8] = r4[0]; rr[4 * g8 + 1] = r4[1]; rr[4 * g8 + 2] = r4[2]; rr[4 * g8 + 3] = r4[3];
            }
            if constexpr (Cfg::REM == 2) {
              uint32_t r2[2];
              ldsm_x2_t(r2, stg_in + uint32_t(Cfg::NG4 * 512) + mrow);      // lanes 0-15 address the 4 trailing tokens
              rr[4 * Cfg::NG4] = r2[0]; rr[4 * Cfg::NG4 + 1] = r2[1];
            } else if constexpr (Cfg::REM == 3) {
              uint32_t r4[4];
              ldsm_x4_t(r4, stg_in + uint32_t(Cfg::NG4 * 512) + mrow);
              rr[4 * Cfg::NG4] = r4[0]; rr[4 * Cfg::NG4 + 1] = r4[1]; rr[4 * Cfg::NG4 + 2] = r4[2]; rr[4 * Cfg::NG4 + 3] = r4[3];
            }
#pragma unroll
            for (int i = 0; i < Cfg::NPAIR; ++i) {
              y[2 * i] += __uint_as_float(rr[i] << 16);
              y[2 * i + 1] += __uint_as_float(rr[i] & 0xffff0000u);
            }
          }
          uint32_t pk[Cfg::PKN];
#pragma unroll
          for (int i = 0; i < Cfg::PKN; ++i) {
            __nv_bfloat162 h2 = __floats2bfloat162_rn(y[2 * i], y[2 * i + 1]);
            pk[i] = *reinterpret_cast<uint32_t*>(&h2);
          }
#pragma unroll
          for (int g8 = 0; g8 < Cfg::NG4; ++g8)
            stsm_x4_t(stg_out + uint32_t(g8 * 512) + mrow, pk[4 * g8], pk[4 * g8 + 1], pk[4 * g8 + 2], pk[4 * g8 + 3]);
          if constexpr (Cfg::REM == 2)
            stsm_x2_t(stg_out + uint32_t(Cfg::NG4 * 512) + mrow, pk[4 * Cfg::NG4], pk[4 * Cfg::NG4 + 1]);
          else if constexpr (Cfg::REM == 3)
            stsm_x4_t(stg_out + uint32_t(Cfg::NG4 * 512) + mrow, pk[4 * Cfg::NG4], pk[4 * Cfg::NG4 + 1], pk[4 * Cfg::NG4 + 2],
                      pk[4 * Cfg::NG4 + 3]);
          __syncwarp();
          if (live) {
#pragma unroll
            for (int r = 0; r < Cfg::PROUNDS; ++r)
              if (lane + 32 * r < Cfg::PIECES) {
                const uint4 o = lds128(stg_out + uint32_t((lane + 32 * r) * 16));
                *reinterpret_cast<uint4*>(dp + r * d_hi) = o;
              }
          }
          dp += d_step;
          __syncwarp();
        }
        if (++ab == 2) { ab = 0; aphase ^= 1u; }
        cg += step_cg;
        tt += step_tt;
        if (cg >= cgn) { cg -= cgn; ++tt; }
      }
    };
    using I0 = std::integral_constant<int, 0>;
    using I1 = std::integral_constant<int, 1>;
    using I2 = std::integral_constant<int, 2>;
    using I3 = std::integral_constant<int, 3>;
    using I4 = std::integral_constant<int, 4>;
    const int fm = epi.plain ? 4 : (epi.film.mode == FILM_OBJECT ? 1 : (epi.film.mode == FILM_TOKEN ? 2 : (per_scene_t ? 3 : 0)));
    if (fm == 4) {
      if (epi.res) run_tiles(I4{}, std::true_type{});
      else run_tiles(I4{}, std::false_type{});
    } else if (epi.res) {
      if (fm == 0) run_tiles(I0{}, std::true_type{});
      else if (fm == 1) run_tiles(I1{}, std::true_type{});
      else if (fm == 2) run_tiles(I2{}, std::true_type{});
      else run_tiles(I3{}, std::true_type{});
    } else {
      if (fm == 0) run_tiles(I0{}, std::false_type{});
      else if (fm == 1) run_tiles(I1{}, std::false_type{});
      else if (fm == 2) run_tiles(I2{}, std::false_type{});
      else run_tiles(I3{}, std::false_type{});
    }
    if (epi.trace && warp == 2 && lane == 0) {
      epi.trace[blockIdx.x * 8 + 5] = tw_tf;
      epi.trace[blockIdx.x * 8 + 6] = clock64() - tstart;
      epi.trace[blockIdx.x * 8 + 7] = ntiles;
    }
  }

  tc_fence_before();
  __syncthreads();
  if (cs > 1) cluster_sync_all();        // no CTA leaves while peers may still write its smem / barriers
  if (warp == 1) {
    tc_fence_after();
    if constexpr (TWO) asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(Cfg::TMEM_COLS) : "memory");
    else asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "n"(Cfg::TMEM_COLS) : "memory");
  }
}

// ------------------------------------------------------------------------------------------------
// host side: tensor maps + launch
// ------------------------------------------------------------------------------------------------
struct TcGemmPlan {
  CUtensorMap tm_a0, tm_a1, tm_w;
  TcEpi epi;
  int bn;
  bool gn;
  bool gnt;          // GroupNorm epilogue, channels-on-lanes variant (weights stored in the permuted row order)
  int num_sms;
  int cluster;       // CTAs per cluster: 1, or 2 for the CTA pair (TWO instantiations)
};

typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
static PFN_encodeTiled g_encode = nullptr;
static int g_num_sms = 0;
static int* g_err_flag = nullptr;       // pinned host memory, device-visible

bool tc_runtime_available(char* err, int err_len) {
  if (g_encode) return true;
  void* fn = nullptr;
  cudaDriverEntryPointQueryResult qres;
  cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres);
  if (e != cudaSuccess || qres != cudaDriverEntryPointSuccess || !fn) {
    if (err) snprintf(err, err_len, "cuTensorMapEncodeTiled unavailable (%s)", cudaGetErrorString(e));
    return false;
  }
  int dev = 0;
  cudaGetDevice(&dev);
  cudaDeviceProp prop;
  cudaGetDeviceProperties(&prop, dev);
  if (prop.major != 10) {
    if (err) snprintf(err, err_len, "tcgen05 GEMM needs sm_100 (found sm_%d%d)", prop.major, prop.minor);
    return false;
  }
  g_num_sms = prop.multiProcessorCount;
  if (!g_err_flag) {
    cudaHostAlloc((void**)&g_err_flag, sizeof(int), cudaHostAllocMapped);
    *g_err_flag = 0;
  }
  cudaFuncSetAttribute(k_gemm_tc<128, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<128, false>::SMEM_BYTES);
  cudaFuncSetAttribute(k_gemm_tc<256, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<256, false>::SMEM_BYTES);
  cudaFuncSetAttribute(k_gemm_tc<256, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<256, true>::SMEM_BYTES);
  cudaFuncSetAttribute(k_gemm_tc<256, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, TcCfg<256, false>::SMEM_BYTES);
  cudaFuncSetAttribute(k_gemm_gnt<12, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, GntCfg<12, true>::SMEM_BYTES);
  cudaFuncSetAttribute(k_gemm_gnt<21, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, GntCfg<21, true>::SMEM_BYTES);
  cudaFuncSetAttribute(k_gemm_gnt<12, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, GntCfg<12, true>::SMEM_BYTES);
  cudaFuncSetAttribute(k_gemm_gnt<21, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, GntCfg<21, false>::SMEM_BYTES);
  g_encode = (PFN_encodeTiled)fn;
  return true;
}

static bool encode_2d(CUtensorMap* map, const void* base, uint64_t inner, uint64_t rows, uint64_t pitch_elems,
                      uint32_t box_rows, char* err, int err_len, uint32_t box_cols = BK,
                      CUtensorMapSwizzle swz = CU_TENSOR_MAP_SWIZZLE_128B) {
  cuuint64_t dims[2] = {inner, rows};
  cuuint64_t strides[1] = {pitch_elems * 2};
  cuuint32_t box[2] = {box_cols, box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = g_encode(map, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    if (err) snprintf(err, err_len, "cuTensorMapEncodeTiled failed (%d): inner=%llu rows=%llu pitch=%llu box=%u",
                      (int)r, (unsigned long long)inner, (unsigned long long)rows, (unsigned long long)pitch_elems,
                      box_rows);
    return false;
  }
  return true;
}

TcGemmPlan* tc_plan_create(const GemmArgs& g, int rows_capacity, char* err, int err_len) {
  if (!tc_runtime_available(err, err_len)) return nullptr;
  const int K = g.k0 + g.k1;
  if (g.k0 % BK || g.k1 % BK || g.N % 128 || K == 0) {
    if (err) snprintf(err, err_len, "tcgen05 GEMM needs K%%64==0 and N%%128==0 (k0=%d k1=%d N=%d)", g.k0, g.k1, g.N);
    return nullptr;
  }
  if ((g.lda0 % 8) || (g.a1 && (g.lda1 % 8)) || (g.ldw % 8) || (g.ldd % 8) || (g.res && (g.ldres % 8)) ||
      ((uintptr_t)g.a0 % 16) || ((uintptr_t)g.w % 16) || ((uintptr_t)g.d % 16) || (g.a1 && ((uintptr_t)g.a1 % 16)) ||
      (g.res && ((uintptr_t)g.res % 16))) {
    if (err) snprintf(err, err_len, "tcgen05 GEMM needs 16-byte aligned operands and pitches");
    return nullptr;
  }
  const bool plain_t = g.gn == 3;                 // channels-on-lanes kernel, no GroupNorm
  const bool gn = g.gn != 0 && !plain_t;
  const bool gnt = g.gn == 2 || plain_t;
  if (g.gn == 2 && !tc_gnt_supported(g.n_obj, g.N)) {
    if (err) snprintf(err, err_len, "channels-on-lanes GroupNorm GEMM needs n_obj in {12, 21} and N %% 128 == 0, N <= 512");
    return nullptr;
  }
  if (plain_t && !tc_gnt_plain_supported(g.n_obj, g.N)) {
    if (err) snprintf(err, err_len, "channels-on-lanes GEMM needs n_obj in {12, 21} and N %% 128 == 0");
    return nullptr;
  }
  if (gn && (g.N % 256 || g.N > TcCfg<256, true>::CHAN_MAX_N || g.n_obj < 1 || g.n_obj > 128 || !g.gamma || !g.beta)) {
    if (err) snprintf(err, err_len, "fused GroupNorm epilogue needs N%%256==0, N<=512, 1<=n_obj<=128, gamma/beta");
    return nullptr;
  }
  if (!gn && !plain_t && g.N > TcCfg<256, false>::CHAN_MAX_N) {
    if (err) snprintf(err, err_len, "tcgen05 GEMM supports N <= 4096 (N=%d)", g.N);
    return nullptr;
  }
  TcGemmPlan* p = new TcGemmPlan();
  memset(p, 0, sizeof(*p));
  // BN = 256 halves the A re-reads; keep 128 when N is not a multiple of 256
  p->bn = (g.N % 256 == 0) ? 256 : 128;
  p->gn = gn;
  p->gnt = gnt;
  p->num_sms = g_num_sms;
  // CTA pair (cta_group::2, a cluster of 2): one M = 256 MMA spans two CTAs, each of which loads half of the operand
  // they share.  Channels-on-lanes kernel: K >= 1024 and an even channel-tile count -- measured on B200
  // (profiles/round2_probe_2cta.txt): the K = 1024 skip convs gain 15 % (66.3 -> 56.6 us), the K = 512 blocks do not
  // (39.2 us either way; with a residual the pair's lock-step costs 3 us).
  // Row-major plain kernel, 128 x 256 tiles: K >= 1024 or N >= 2048.  Same box, 4096 scenes
  // (profiles/round2_probe_tc2.txt): 512 x 1024 51.0 -> 45.1 us, encoder K = 3072 128.3 -> 119.6 us, dec.l0 N = 3072
  // 143.3 -> 137.1 us, but 512 x 512 31.2 -> 34.2 us and enc.l1 (N = 1024, K = 512) 51.4 -> 52.5 us; whole sample
  // +1.4 % with the pair on every K >= 256 launch.  All 111 GPU tests ran green with the pair on every K >= 256 launch
  // (a superset).
  const bool two = gnt ? K >= 1024 && (g.N / BM) % 2 == 0
                       : !gn && !g.no_pair && p->bn == 256 && (K >= 1024 || g.N >= 2048);
  p->cluster = two ? 2 : 1;
  const int gnt_un = g.n_obj == 21 ? GntCfg<21>::UN : GntCfg<12>::UN;
  const int gnt_tok = g.n_obj == 21 ? GntCfg<21>::TOK : GntCfg<12>::TOK;
  const uint32_t act_box = gnt ? uint32_t(gnt_un / p->cluster) : uint32_t(BM);     // rows of one activation load
  bool ok = encode_2d(&p->tm_a0, g.a0, g.k0, rows_capacity, g.lda0, act_box, err, err_len);
  if (ok && g.a1) ok = encode_2d(&p->tm_a1, g.a1, g.k1, rows_capacity, g.lda1, act_box, err, err_len);
  if (ok && !g.a1) p->tm_a1 = p->tm_a0;
  if (ok) ok = encode_2d(&p->tm_w, g.w, K, g.N, g.ldw, gnt ? BM : p->bn / p->cluster, err, err_len);
  const int tile_rows = gnt ? gnt_tok : (gn ? (BM / g.n_obj) * g.n_obj : BM);
  if (gn && !gnt && tile_rows / g.n_obj > TcCfg<256, true>::SPT_FAST) {
    if (err) snprintf(err, err_len, "fused GroupNorm epilogue supports at most %d scenes per 128-row tile (n_obj=%d)",
                      TcCfg<256, true>::SPT_FAST, g.n_obj);
    ok = false;
  }
  if (!ok) {
    delete p;
    return nullptr;
  }
  p->epi.bias = g.bias;
  p->epi.d = (bf16*)g.d;
  p->epi.ldd = g.ldd;
  p->epi.res = (const bf16*)g.res;
  p->epi.ldres = g.ldres;
  p->epi.act = g.act;
  p->epi.M = g.M;
  p->epi.N = g.N;
  p->epi.kb0 = g.k0 / BK;
  p->epi.kb1 = g.k1 / BK;
  p->epi.desc_hi = umma_desc_hi_sw128();
  p->epi.idesc = p->bn == 256 ? TcCfg<256, false>::IDESC : TcCfg<128, false>::IDESC;
  p->epi.tile_rows = tile_rows;
  p->epi.n_obj = g.n_obj;
  p->epi.C = g.film_C;
  p->epi.gamma = g.gamma;
  p->epi.beta = g.beta;
  p->epi.film = g.film;
  p->epi.plain = plain_t ? 1 : 0;
  p->epi.d32 = nullptr;
  p->epi.ksplit = 1;
  return p;
}
void tc_plan_destroy(TcGemmPlan* p) { delete p; }
void tc_plan_set_film(TcGemmPlan* p, const FilmRef& f) { p->epi.film = f; }
void tc_plan_set_trace(TcGemmPlan* p, unsigned long long* trace) { p->epi.trace = trace; }
void tc_plan_set_uniform_t(TcGemmPlan* p, int uniform) { p->epi.film_uniform = uniform; }
// split-K mode of the plain row-major kernel: D (fp32, pitch ldd floats) += A W^T, partial sums added with atomics
void tc_plan_set_atomic_out(TcGemmPlan* p, float* d32, int ldd, int ksplit) {
  p->epi.d32 = d32;
  p->epi.ldd = ldd;
  p->epi.ksplit = ksplit < 1 ? 1 : ksplit;
}
void tc_plan_set_residual(TcGemmPlan* p, const void* res) { p->epi.res = (const bf16*)res; }
int tc_plan_tiles(const TcGemmPlan* p, int M) {
  const int num_m = (M + p->epi.tile_rows - 1) / p->epi.tile_rows;
  return ((num_m + p->cluster - 1) / p->cluster) * (p->epi.N / p->bn);
}

template <int BN, bool GN, bool TWO = false>
static int launch_one(const TcGemmPlan* p, const TcEpi& epi, int total_ct, int* flag_dev, cudaStream_t s) {
  const int cs = p->cluster;
  int max_cl = p->num_sms / cs;
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3(TC_THREADS);
  cfg.dynamicSmemBytes = TcCfg<BN, GN>::SMEM_BYTES;
  cfg.stream = s;
  cudaLaunchAttribute attr[2];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = cs;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  // off by default at the throughput batch: with the 576-thread channels-on-lanes kernels in the step program PDL
  // measured 1.5 % SLOWER (the chip is power-capped; early-resident CTAs polling their barriers cost clock)
  const bool pdl = pdl_enabled(epi.M);
  if (pdl) {      // may start while the previous kernel in the stream drains (it waits at griddepcontrol.wait)
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.numAttrs = 2;
  }
  if constexpr (TWO) {
    static int cached = 0;      // co-resident CTA pairs
    if (!cached) {
      cfg.gridDim = dim3(max_cl * cs);
      int n = 0;
      cached = (cudaOccupancyMaxActiveClusters(&n, k_gemm_tc<BN, GN, TWO>, &cfg) == cudaSuccess && n > 0) ? n : max_cl;
    }
    if (cached < max_cl) max_cl = cached;
  }
  const int ncl = total_ct < max_cl ? total_ct : max_cl;
  cfg.gridDim = dim3(ncl * cs);
  return (int)cudaLaunchKernelEx(&cfg, k_gemm_tc<BN, GN, TWO>, p->tm_a0, p->tm_a1, p->tm_w, epi, flag_dev);
}

// object counts the channels-on-lanes kernel is instantiated for
static bool gnt_nobj_ok(int n_obj) { return n_obj == 12 || n_obj == 21; }
bool tc_gnt_plain_supported(int n_obj, int N) { return gnt_nobj_ok(n_obj) && N % BM == 0; }
bool tc_gnt_supported(int n_obj, int N) { return gnt_nobj_ok(n_obj) && N % BM == 0 && N <= GntCfg<12, true>::CHAN_MAX_N; }

template <int NOBJ, bool PAIR, bool TWO = false>
static int launch_gnt(const TcGemmPlan* p, const TcEpi& epi, int* flag_dev, cudaStream_t s) {
  using Cfg = GntCfg<NOBJ, PAIR>;
  const int n_scenes = epi.M / NOBJ;
  const int cs = p->cluster;
  const int total = ((n_scenes + Cfg::SC - 1) / Cfg::SC) * (epi.N / BM / cs);      // work units per cluster
  if (total == 0) return 0;
  cudaLaunchConfig_t cfg = {};
  cfg.blockDim = dim3(Cfg::THREADS);
  cfg.dynamicSmemBytes = Cfg::SMEM_BYTES;
  cfg.stream = s;
  cudaLaunchAttribute attr[2];
  int na = 0;
  const bool pdl = pdl_enabled(epi.M);
  if (pdl) {
    attr[na].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[na].val.programmaticStreamSerializationAllowed = 1;
    ++na;
  }
  int max_cl = p->num_sms / cs;
  if (cs > 1) {
    attr[na].id = cudaLaunchAttributeClusterDimension;
    attr[na].val.clusterDim.x = cs;
    attr[na].val.clusterDim.y = 1;
    attr[na].val.clusterDim.z = 1;
    ++na;
    static int cached = 0;
    if (!cached) {
      cfg.attrs = attr;
      cfg.numAttrs = na;
      cfg.gridDim = dim3(max_cl * cs);
      int n = 0;
      cached = (cudaOccupancyMaxActiveClusters(&n, k_gemm_gnt<NOBJ, PAIR, TWO>, &cfg) == cudaSuccess && n > 0) ? n : max_cl;
    }
    if (cached < max_cl) max_cl = cached;
  }
  cfg.attrs = na ? attr : nullptr;
  cfg.numAttrs = na;
  cfg.gridDim = dim3((total < max_cl ? total : max_cl) * cs);
  return (int)cudaLaunchKernelEx(&cfg, k_gemm_gnt<NOBJ, PAIR, TWO>, p->tm_w, p->tm_a0, p->tm_a1, epi, flag_dev);
}

int launch_gemm_tc(const TcGemmPlan* p, int M, cudaStream_t s) {
  TcEpi epi = p->epi;
  epi.M = M;
  if (p->gnt) {
    int* fd = nullptr;
    cudaHostGetDevicePointer((void**)&fd, g_err_flag, 0);
    // GroupNorm statistics exchange: warp-pair local (PAIR, named 64-thread barriers) rather than two CTA-wide
    // barriers.  No difference while the MMA issue was the slow side (profiles/round2_gnt_ab.txt: 39.3 / 43.2 / 66.3
    // us vs 40.0 / 43.2 / 66.0 us); with the warp-uniform issue the residual blocks gain (41.5 -> 40.1 us) and the
    // whole sample 1.1 % (900.5 -> 910.8 scenes/s, profiles/round2_probe_l2pf.txt).  The N = 21 CTA pair keeps the
    // CTA-wide barriers.
    if (p->cluster == 2)
      return epi.n_obj == 21 ? launch_gnt<21, false, true>(p, epi, fd, s) : launch_gnt<12, true, true>(p, epi, fd, s);
    return epi.n_obj == 21 ? launch_gnt<21, true>(p, epi, fd, s) : launch_gnt<12, true>(p, epi, fd, s);
  }
  const int num_m = (M + epi.tile_rows - 1) / epi.tile_rows;
  const int total_ct = ((num_m + p->cluster - 1) / p->cluster) * (epi.N / p->bn) * (epi.ksplit > 1 ? epi.ksplit : 1);
  if (total_ct == 0) return 0;
  int* flag_dev = nullptr;
  cudaHostGetDevicePointer((void**)&flag_dev, g_err_flag, 0);
  if (p->gn) return launch_one<256, true>(p, epi, total_ct, flag_dev, s);
  if (p->cluster == 2) return launch_one<256, false, true>(p, epi, total_ct, flag_dev, s);
  if (p->bn == 256) return launch_one<256, false>(p, epi, total_ct, flag_dev, s);
  return launch_one<128, false>(p, epi, total_ct, flag_dev, s);
}

int tc_error_flag() { return g_err_flag ? *g_err_flag : 0; }
// shared with the other tcgen05 kernels of the library (gemm_ln.cu)
bool tc_encode_2d(CUtensorMap* map, const void* base, uint64_t inner, uint64_t rows, uint64_t pitch_elems,
                  uint32_t box_rows, char* err, int err_len) {
  return encode_2d(map, base, inner, rows, pitch_elems, box_rows, err, err_len);
}
int* tc_error_flag_dev() {
  int* fd = nullptr;
  cudaHostGetDevicePointer((void**)&fd, g_err_flag, 0);
  return fd;
}
int tc_num_sms() { return g_num_sms; }

}  // namespace ds
