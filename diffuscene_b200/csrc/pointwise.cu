// Non-GEMM kernels of the denoiser and of the diffusion step (sm_100a).
//
// Activation matrices are token-major: row r = scene (r / n_obj), object (r % n_obj); columns are
// channels.  One warp owns one (scene, group) for GroupNorm, one token for LayerNorm and one
// (scene, head) for the attention cores, so every reduction is a register / shuffle reduction.
// Reference semantics: scene_synthesis/networks/denoise_net.py (Block :160-176, LayerNorm :93-102,
// LinearAttention :208-235, Attention :237-259, LinearAttentionCross :261-297) and
// scene_synthesis/networks/diffusion_ddpm.py (q_sample :276-286, p_sample :339-352, p_losses :520-652).
#include "kernels.cuh"
#include <utility>

namespace ds {

// Programmatic dependent launch for the pointwise kernels of the step program: launched with the PDL attribute, a
// kernel may be scheduled while the previous kernel in the stream (a GEMM that issued griddepcontrol.launch_dependents)
// drains; it touches no memory before `pdl_wait()`.  These kernels do NOT trigger their own dependents early (their
// dependents are 96-register, 216 KB GEMM CTAs that would crowd out the remaining waves).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
bool pdl_enabled(int64_t rows) { return rows <= 32768; }
// rows: tokens the launch works on (the PDL policy keys on it); the pointwise kernels pass their row count
template <typename... KArgs, typename... Args>
static void launch_pdl_rows(int64_t rows, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
  const bool pdl = pdl_enabled(rows);
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  if (pdl) {
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
  }
  (void)cudaLaunchKernelEx(&cfg, kern, KArgs(std::forward<Args>(args))...);   // errors surface at the caller's sync / cudaGetLastError
}
// every kernel launched through here uses at least one thread per 4 tokens ... the grid is a good proxy for the rows
template <typename... KArgs, typename... Args>
static void launch_pdl(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args&&... args) {
  launch_pdl_rows(int64_t(grid.x) * 8, kern, grid, block, smem, s, std::forward<Args>(args)...);
}


static inline int cdiv(int64_t a, int64_t b) { return int((a + b - 1) / b); }

// ------------------------------------------------------------------------------------------------
// input pack / output unpack
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void k_pack_input(const float* __restrict__ x, T* __restrict__ out, int ld_out, int M, int d) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)M * ld_out) return;
  int r = int(i / ld_out), c = int(i % ld_out);
  stf(out + i, c < d ? x[(int64_t)r * d + c] : 0.0f);
}
template <typename T>
void launch_pack_input(const float* x, T* out, int ld_out, int M, int d, cudaStream_t s) {
  int64_t n = (int64_t)M * ld_out;
  k_pack_input<T><<<cdiv(n, 256), 256, 0, s>>>(x, out, ld_out, M, d);
}

template <typename T>
__global__ void k_unpack_output(const T* __restrict__ in, int ld_in, float* __restrict__ out, int M, int d) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)M * d) return;
  int r = int(i / d), c = int(i % d);
  out[i] = ldf(in + (int64_t)r * ld_in + c);
}
template <typename T>
void launch_unpack_output(const T* in, int ld_in, float* out, int M, int d, cudaStream_t s) {
  int64_t n = (int64_t)M * d;
  k_unpack_output<T><<<cdiv(n, 256), 256, 0, s>>>(in, ld_in, out, M, d);
}

// ------------------------------------------------------------------------------------------------
// GroupNorm (+ affine) (+ FiLM) + SiLU (+ residual)      one warp per (scene, group)
// ------------------------------------------------------------------------------------------------
template <typename T, bool EXACT>
__global__ void __launch_bounds__(128) k_groupnorm(const T* __restrict__ in, int ld_in, T* __restrict__ out,
                                                   int ld_out, const float* __restrict__ gamma,
                                                   const float* __restrict__ beta, FilmRef film,
                                                   const T* __restrict__ res, int ld_res, int n_scenes, int n_obj,
                                                   int C, int groups) {
  const int lane = threadIdx.x & 31;
  const int w = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (w >= n_scenes * groups) return;
  const int scene = w / groups, grp = w % groups;
  const int cpg = C / groups;
  const int64_t row0 = (int64_t)scene * n_obj;
  const int c0 = grp * cpg;
  const float inv_cnt = 1.0f / float(n_obj * cpg);

  float s = 0.f;
  for (int r = 0; r < n_obj; ++r)
    for (int c = lane; c < cpg; c += 32) s += ldf(in + (row0 + r) * ld_in + c0 + c);
  const float mean = warp_sum(s) * inv_cnt;
  float q = 0.f;
  for (int r = 0; r < n_obj; ++r)
    for (int c = lane; c < cpg; c += 32) {
      float v = ldf(in + (row0 + r) * ld_in + c0 + c) - mean;
      q += v * v;
    }
  const float var = warp_sum(q) * inv_cnt;
  const float rstd = EXACT ? 1.0f / sqrtf(var + 1e-5f) : rsqrtf(var + 1e-5f);

  for (int r = 0; r < n_obj; ++r) {
    const float* frow = nullptr;
    if (film.mode == FILM_TIME) frow = film.base + (int64_t)film.t[scene] * film.row_stride;
    else if (film.mode == FILM_OBJECT) frow = film.base + (int64_t)r * film.row_stride;
    else if (film.mode == FILM_TOKEN) frow = film.base + (row0 + r) * film.row_stride;
    for (int c = lane; c < cpg; c += 32) {
      const int ch = c0 + c;
      float v = (ldf(in + (row0 + r) * ld_in + ch) - mean) * rstd * gamma[ch] + beta[ch];
      if (frow) v = v * (frow[ch] + 1.0f) + frow[C + ch];
      v = EXACT ? silu_exact(v) : silu(v);
      if (res) v += ldf(res + (row0 + r) * ld_res + ch);
      stf(out + (row0 + r) * ld_out + ch, v);
    }
  }
}
template <typename T>
void launch_groupnorm(const T* in, int ld_in, T* out, int ld_out, const float* gamma, const float* beta,
                      FilmRef film, const T* res, int ld_res, int n_scenes, int n_obj, int C, int groups,
                      cudaStream_t s) {
  int warps = n_scenes * groups;
  constexpr bool EX = sizeof(T) == 4;
  k_groupnorm<T, EX><<<cdiv(warps, 4), 128, 0, s>>>(in, ld_in, out, ld_out, gamma, beta, film, res, ld_res,
                                                    n_scenes, n_obj, C, groups);
}

// ------------------------------------------------------------------------------------------------
// channel LayerNorm (no bias) (+ residual)                one warp per token, C <= 1024
// ------------------------------------------------------------------------------------------------
template <typename T, bool EXACT>
__global__ void __launch_bounds__(128) k_layernorm(const T* __restrict__ in, int ld_in, T* __restrict__ out,
                                                   int ld_out, const float* __restrict__ g,
                                                   const T* __restrict__ res, int ld_res, int M, int C) {
  const int lane = threadIdx.x & 31;
  const int64_t row = blockIdx.x * 4 + (threadIdx.x >> 5);
  if (row >= M) return;
  float v[32];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    int c = i * 32 + lane;
    v[i] = c < C ? ldf(in + row * ld_in + c) : 0.f;
    s += v[i];
  }
  const float mean = warp_sum(s) / float(C);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    int c = i * 32 + lane;
    float dlt = c < C ? v[i] - mean : 0.f;
    q += dlt * dlt;
  }
  const float var = warp_sum(q) / float(C);
  const float rstd = EXACT ? 1.0f / sqrtf(var + 1e-5f) : rsqrtf(var + 1e-5f);
#pragma unroll
  for (int i = 0; i < 32; ++i) {
    int c = i * 32 + lane;
    if (c < C) {
      float y = (v[i] - mean) * rstd * g[c];
      if (res) y += ldf(res + row * ld_res + c);
      stf(out + row * ld_out + c, y);
    }
  }
}
// C == 512 fast path: each lane owns 16 contiguous channels (two 16-byte loads for bf16, four for fp32)
template <typename T> struct Vec16;
template <> struct Vec16<bf16> {
  static __device__ __forceinline__ void load(const bf16* row, int lane, float (&v)[16]) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      uint4 pk = *reinterpret_cast<const uint4*>(row + h * 256 + lane * 8);
      const __nv_bfloat162* h2 = reinterpret_cast<const __nv_bfloat162*>(&pk);
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        float2 f = __bfloat1622float2(h2[e]);
        v[h * 8 + e * 2] = f.x;
        v[h * 8 + e * 2 + 1] = f.y;
      }
    }
  }
  static __device__ __forceinline__ void store(bf16* row, int lane, const float (&v)[16]) {
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      uint4 pk;
      __nv_bfloat162* h2 = reinterpret_cast<__nv_bfloat162*>(&pk);
#pragma unroll
      for (int e = 0; e < 4; ++e) h2[e] = __floats2bfloat162_rn(v[h * 8 + e * 2], v[h * 8 + e * 2 + 1]);
      *reinterpret_cast<uint4*>(row + h * 256 + lane * 8) = pk;
    }
  }
};
template <> struct Vec16<float> {      // same channel ownership as the bf16 layout: 8*lane.. and 256 + 8*lane..
  static __device__ __forceinline__ void load(const float* row, int lane, float (&v)[16]) {
#pragma unroll
    for (int h = 0; h < 4; ++h) {
      float4 f = *reinterpret_cast<const float4*>(row + (h >> 1) * 256 + lane * 8 + (h & 1) * 4);
      v[h * 4] = f.x; v[h * 4 + 1] = f.y; v[h * 4 + 2] = f.z; v[h * 4 + 3] = f.w;
    }
  }
  static __device__ __forceinline__ void store(float* row, int lane, const float (&v)[16]) {
#pragma unroll
    for (int h = 0; h < 4; ++h)
      *reinterpret_cast<float4*>(row + (h >> 1) * 256 + lane * 8 + (h & 1) * 4) =
          make_float4(v[h * 4], v[h * 4 + 1], v[h * 4 + 2], v[h * 4 + 3]);
  }
};

template <typename T, bool EXACT>
__global__ void __launch_bounds__(256) k_layernorm512(const T* __restrict__ in, int ld_in, T* __restrict__ out,
                                                      int ld_out, const float* __restrict__ g,
                                                      const T* __restrict__ res, int ld_res, int M) {
  pdl_wait();
  const int lane = threadIdx.x & 31;
  const int64_t row = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (row >= M) return;
  // lane owns channels [8*lane, 8*lane+8) and [256 + 8*lane, ...): every warp load is 512 contiguous bytes (bf16)
  float v[16];
  Vec16<T>::load(in + row * ld_in, lane, v);
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) s += v[i];
  const float mean = warp_sum(s) * (1.0f / 512.0f);
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    float dlt = v[i] - mean;
    q = fmaf(dlt, dlt, q);
  }
  const float var = warp_sum(q) * (1.0f / 512.0f);
  const float rstd = EXACT ? 1.0f / sqrtf(var + 1e-5f) : rsqrtf(var + 1e-5f);
  float gg[16];
  Vec16<float>::load(g, lane, gg);
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = (v[i] - mean) * rstd * gg[i];
  if (res) {
    float r[16];
    Vec16<T>::load(res + row * ld_res, lane, r);
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] += r[i];
  }
  Vec16<T>::store(out + row * ld_out, lane, v);
}

template <typename T>
void launch_layernorm(const T* in, int ld_in, T* out, int ld_out, const float* g, const T* res, int ld_res, int M,
                      int C, cudaStream_t s) {
  constexpr bool EX = sizeof(T) == 4;
  const bool vec_ok = C == 512 && ld_in % 16 == 0 && ld_out % 16 == 0 && (!res || ld_res % 16 == 0);
  if (vec_ok) launch_pdl(k_layernorm512<T, EX>, dim3(cdiv(M, 8)), dim3(256), 0, s, in, ld_in, out, ld_out, g, res, ld_res, M);
  else k_layernorm<T, EX><<<cdiv(M, 4), 128, 0, s>>>(in, ld_in, out, ld_out, g, res, ld_res, M, C);
}

// ------------------------------------------------------------------------------------------------
// attention cores: 4 heads x 32 channels, one warp per (scene, head), lane = head channel
// dynamic smem: 4 warps x 3 x n_obj x 33 floats
// ------------------------------------------------------------------------------------------------
template <typename T, int NMAX, int NEXACT = 0>
__global__ void __launch_bounds__(128) k_linattn(const T* __restrict__ qkv, int ld, T* __restrict__ out, int ld_out,
                                                 int n_scenes, int n_rt) {
  const int n = NEXACT > 0 ? NEXACT : n_rt;      // compile-time scene size for the shipped configs (12, 21)
  extern __shared__ float sm[];
  const int lane = threadIdx.x & 31, h = threadIdx.x >> 5;
  const int scene = blockIdx.x;
  float* qs = sm + h * 2 * n * 32;
  float* ks = qs + n * 32;
  const int64_t row0 = (int64_t)scene * n;
  const float scale = 0.17677669529663687f;   // 32^-0.5
  // all rows of this (scene, head) are fetched up front: 3*n independent loads in flight per lane
  float qv[NMAX], kv[NMAX], vv[NMAX];
#pragma unroll
  for (int r = 0; r < NMAX; ++r) {
    if (r < n) {
      const T* p = qkv + (row0 + r) * ld + h * 32 + lane;
      qv[r] = ldf(p); kv[r] = ldf(p + 128); vv[r] = ldf(p + 256);
    } else {
      qv[r] = 0.f; kv[r] = -INFINITY; vv[r] = 0.f;
    }
  }
  // q: softmax over the 32 head channels of each token, then * scale (denoise_net.py:226-229)
#pragma unroll
  for (int r = 0; r < NMAX; ++r) {
    if (r < n) {
      float m = warp_max(qv[r]);
      float e = (sizeof(T) == 4) ? expf(qv[r] - m) : __expf(qv[r] - m);   // exact in the fp32 parity mode
      float ssum = warp_sum(e);
      qs[r * 32 + lane] = e / ssum * scale;
    }
  }
  // k: softmax over tokens for each channel (lane-private column)
  float kmax = -INFINITY;
#pragma unroll
  for (int r = 0; r < NMAX; ++r) kmax = fmaxf(kmax, kv[r]);
  float ksum = 0.f;
#pragma unroll
  for (int r = 0; r < NMAX; ++r) {
    kv[r] = r < n ? ((sizeof(T) == 4) ? expf(kv[r] - kmax) : __expf(kv[r] - kmax)) : 0.f;
    ksum += kv[r];
  }
  const float kinv = 1.0f / ksum;
#pragma unroll
  for (int r = 0; r < NMAX; ++r)
    if (r < n) ks[r * 32 + lane] = kv[r] * kinv;
  __syncwarp();
  // ctx[d][e] = sum_n k[d,n] v[e,n]; this lane keeps column e = lane (k rows read as broadcast float4)
  float ctx[32];
#pragma unroll
  for (int d = 0; d < 32; ++d) ctx[d] = 0.f;
#pragma unroll
  for (int r = 0; r < NMAX; ++r) {
    if (r < n) {
      const float v = vv[r];
      const float4* k4 = reinterpret_cast<const float4*>(ks + r * 32);
#pragma unroll
      for (int d4 = 0; d4 < 8; ++d4) {
        const float4 kk = k4[d4];
        ctx[4 * d4] = fmaf(kk.x, v, ctx[4 * d4]);
        ctx[4 * d4 + 1] = fmaf(kk.y, v, ctx[4 * d4 + 1]);
        ctx[4 * d4 + 2] = fmaf(kk.z, v, ctx[4 * d4 + 2]);
        ctx[4 * d4 + 3] = fmaf(kk.w, v, ctx[4 * d4 + 3]);
      }
    }
  }
  // out[e,n] = sum_d ctx[d][e] q[d,n]
#pragma unroll
  for (int r = 0; r < NMAX; ++r) {
    if (r < n) {
      const float4* q4 = reinterpret_cast<const float4*>(qs + r * 32);
      float o0 = 0.f, o1 = 0.f, o2 = 0.f, o3 = 0.f;
#pragma unroll
      for (int d4 = 0; d4 < 8; ++d4) {
        const float4 qq = q4[d4];
        o0 = fmaf(ctx[4 * d4], qq.x, o0);
        o1 = fmaf(ctx[4 * d4 + 1], qq.y, o1);
        o2 = fmaf(ctx[4 * d4 + 2], qq.z, o2);
        o3 = fmaf(ctx[4 * d4 + 3], qq.w, o3);
      }
      stf(out + (row0 + r) * ld_out + h * 32 + lane, (o0 + o1) + (o2 + o3));
    }
  }
}
// ---- tensor-core variant of the linear-attention core (bf16 mode) -------------------------------------------
// Same math as k_linattn, but the two tiny contractions of each (scene, head)
//     ctx^T[e][d] = sum_n v[n][e] k~[n][d]          (k~ = softmax of k over the scene's tokens)
//     out^T[e][n] = sum_d ctx^T[e][d] q~[n][d]      (q~ = softmax of q over the 32 head channels, * 32^-1/2)
// run on mma.sync.m16n8k16 (bf16 operands, fp32 accumulation): 16 HMMAs instead of ~770 FMAs per lane.  These
// are 32 x 32 x n problems (n <= 32 tokens), far below the 128-row minimum of tcgen05, hence warp-level MMA.
// The accumulator fragments of the first product are re-used directly as the A fragments of the second (the
// C layout of two adjacent n-tiles is the A layout of one k-tile).
__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  __nv_bfloat162 h2 = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<uint32_t*>(&h2);
}

template <int NT>     // tokens padded to NT (16 or 32)
__global__ void __launch_bounds__(128) k_linattn_mma(const bf16* __restrict__ qkv, int ld, bf16* __restrict__ out,
                                                     int ld_out, int n_scenes, int n) {
  constexpr int CS = NT + 8;          // channel-major row stride (bf16 elements): conflict-free fragment loads
  constexpr int QS = 40;              // token-major row stride of q~ (bf16 elements)
  constexpr int OS = 33;              // staging row stride of the output (fp32)
  constexpr int WARP_BYTES = 2 * 32 * CS * 2 + NT * QS * 2 + NT * OS * 4;
  extern __shared__ __align__(16) unsigned char smraw[];
  const int lane = threadIdx.x & 31, h = threadIdx.x >> 5;
  const int scene = blockIdx.x;
  unsigned char* wb = smraw + h * WARP_BYTES;
  bf16* vt = reinterpret_cast<bf16*>(wb);                     // [32 ch][CS]  v transposed
  bf16* kt = vt + 32 * CS;                                    // [32 ch][CS]  softmax(k) transposed
  bf16* qs = kt + 32 * CS;                                    // [NT tok][QS] softmax(q) * scale
  float* os = reinterpret_cast<float*>(qs + NT * QS);         // [NT tok][OS] output staging
  const int64_t row0 = (int64_t)scene * n;
  const float scale = 0.17677669529663687f;
  const int g = lane >> 2, t = lane & 3;

  float qv[NT], kv[NT], vv[NT];
#pragma unroll
  for (int r = 0; r < NT; ++r) {
    if (r < n) {
      const bf16* p = qkv + (row0 + r) * ld + h * 32 + lane;
      qv[r] = __bfloat162float(p[0]); kv[r] = __bfloat162float(p[128]); vv[r] = __bfloat162float(p[256]);
    } else {
      qv[r] = 0.f; kv[r] = -INFINITY; vv[r] = 0.f;
    }
  }
  // q~: softmax over the 32 channels (lanes) of each token
#pragma unroll
  for (int r = 0; r < NT; ++r) {
    float e = 0.f;
    if (r < n) {
      float m = warp_max(qv[r]);
      e = __expf(qv[r] - m);
      e = e / warp_sum(e) * scale;
    }
    qs[r * QS + lane] = __float2bfloat16_rn(e);
  }
  // k~: softmax over the tokens, per channel (lane-private); v: as is.  Both stored channel-major.
  float kmax = -INFINITY;
#pragma unroll
  for (int r = 0; r < NT; ++r) kmax = fmaxf(kmax, kv[r]);
  float ksum = 0.f;
#pragma unroll
  for (int r = 0; r < NT; ++r) {
    kv[r] = r < n ? __expf(kv[r] - kmax) : 0.f;
    ksum += kv[r];
  }
  const float kinv = 1.0f / ksum;
#pragma unroll
  for (int r = 0; r < NT; r += 2) {
    *reinterpret_cast<uint32_t*>(kt + lane * CS + r) = pack_bf16x2(kv[r] * kinv, kv[r + 1] * kinv);
    *reinterpret_cast<uint32_t*>(vt + lane * CS + r) = pack_bf16x2(vv[r], vv[r + 1]);
  }
  __syncwarp();

  // ---- ctx^T = V^T K~ : M = e (2 tiles), N = d (4 tiles), K = tokens (NT / 16 steps)
  float c[2][4][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) c[mt][nt][i] = 0.f;
#pragma unroll
  for (int ks = 0; ks < NT / 16; ++ks) {
    uint32_t a[2][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      const bf16* r0 = vt + (16 * mt + g) * CS + 16 * ks + 2 * t;
      const bf16* r1 = r0 + 8 * CS;
      a[mt][0] = *reinterpret_cast<const uint32_t*>(r0);
      a[mt][1] = *reinterpret_cast<const uint32_t*>(r1);
      a[mt][2] = *reinterpret_cast<const uint32_t*>(r0 + 8);
      a[mt][3] = *reinterpret_cast<const uint32_t*>(r1 + 8);
    }
#pragma unroll
    for (int nt = 0; nt < 4; ++nt) {
      const bf16* kr = kt + (8 * nt + g) * CS + 16 * ks + 2 * t;
      const uint32_t b0 = *reinterpret_cast<const uint32_t*>(kr);
      const uint32_t b1 = *reinterpret_cast<const uint32_t*>(kr + 8);
      mma_bf16_16816(c[0][nt], a[0], b0, b1);
      mma_bf16_16816(c[1][nt], a[1], b0, b1);
    }
  }
  // ---- out^T = ctx^T Q~^T : M = e (2 tiles), N = tokens (NT / 8 tiles), K = d (2 steps)
#pragma unroll
  for (int mt = 0; mt < 2; ++mt) {
    uint32_t a[2][4];
#pragma unroll
    for (int ks = 0; ks < 2; ++ks) {
      a[ks][0] = pack_bf16x2(c[mt][2 * ks][0], c[mt][2 * ks][1]);
      a[ks][1] = pack_bf16x2(c[mt][2 * ks][2], c[mt][2 * ks][3]);
      a[ks][2] = pack_bf16x2(c[mt][2 * ks + 1][0], c[mt][2 * ks + 1][1]);
      a[ks][3] = pack_bf16x2(c[mt][2 * ks + 1][2], c[mt][2 * ks + 1][3]);
    }
#pragma unroll
    for (int nt = 0; nt < NT / 8; ++nt) {
      float o[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int ks = 0; ks < 2; ++ks) {
        const bf16* qr = qs + (8 * nt + g) * QS + 16 * ks + 2 * t;
        mma_bf16_16816(o, a[ks], *reinterpret_cast<const uint32_t*>(qr), *reinterpret_cast<const uint32_t*>(qr + 8));
      }
      // o[0], o[1]: (e = 16mt + g, tokens 8nt + 2t, +1); o[2], o[3]: e + 8
      os[(8 * nt + 2 * t) * OS + 16 * mt + g] = o[0];
      os[(8 * nt + 2 * t + 1) * OS + 16 * mt + g] = o[1];
      os[(8 * nt + 2 * t) * OS + 16 * mt + g + 8] = o[2];
      os[(8 * nt + 2 * t + 1) * OS + 16 * mt + g + 8] = o[3];
    }
  }
  __syncwarp();
  for (int r = 0; r < n; ++r) out[(row0 + r) * ld_out + h * 32 + lane] = __float2bfloat16_rn(os[r * OS + lane]);
}
// ---- fragment-layout variant (the one the bf16 mode runs) ----------------------------------------------------
// Same two contractions, arranged so that almost nothing is reshuffled:
//   * q is loaded from global memory directly in the MMA fragment layout (thread (g, t) of the warp owns tokens
//     g, g + 8 and the channel pairs 2t + 8j): its channel softmax is 8 local values + a 4-lane butterfly, and the
//     result is the A operand of   out[n][e] = sum_d q~[n][d] ctx[d][e]   without touching shared memory;
//   * v is copied token-major (16-byte vectors) into shared memory and read back with ldmatrix.trans as the A
//     operand of   ctx^T[e][d] = sum_n v[n][e] k~[n][d];  k is soft-maxed over the tokens with one lane per channel,
//     stored token-major as bf16 and read back with ldmatrix.trans as the B operand;
//   * the fp32 accumulator fragments of ctx^T are exactly the B fragments of the second product;
//   * the output fragments (token g, channel pair 2t of each 8-channel block) are stored as packed bf16x2.
// ~400 instructions per (scene, head) warp instead of ~1400.
__device__ __forceinline__ void ldsm_x4_trans(uint32_t (&r)[4], uint32_t addr) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0, %1, %2, %3}, [%4];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
               : "r"(addr));
}
__device__ __forceinline__ float fast_exp2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float quad_max(float v) {
  v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 1));
  return fmaxf(v, __shfl_xor_sync(0xffffffffu, v, 2));
}
__device__ __forceinline__ float quad_sum(float v) {
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  return v + __shfl_xor_sync(0xffffffffu, v, 2);
}

template <int NT, int NE>     // tokens padded to NT (16 or 32); NE > 0: compile-time scene size
__global__ void __launch_bounds__(128) k_linattn_frag(const bf16* __restrict__ qkv, int ld, bf16* __restrict__ out,
                                                      int ld_out, int n_scenes, int n_rt) {
  constexpr int MT = NT / 16;         // 16-token tiles
  constexpr int RS = 40;              // shared-memory row stride (bf16): 80 B, conflict-free for ldmatrix
  pdl_wait();
  const int n = NE > 0 ? NE : n_rt;
  __shared__ __align__(16) bf16 sm_v[4][NT * RS];
  __shared__ __align__(16) bf16 sm_k[4][NT * RS];
  const int lane = threadIdx.x & 31, h = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int scene = blockIdx.x;
  const int64_t row0 = (int64_t)scene * n;
  bf16* vs = sm_v[h];
  bf16* ks = sm_k[h];
  const bf16* base = qkv + row0 * ld + h * 32;
  const float LOG2E = 1.4426950408889634f;

  // ---- v: token-major copy (rows >= n are zero)
#pragma unroll
  for (int idx = lane; idx < NT * 4; idx += 32) {
    const int r = idx >> 2, part = idx & 3;
    uint4 val = make_uint4(0u, 0u, 0u, 0u);
    if (r < n) val = __ldg(reinterpret_cast<const uint4*>(base + (int64_t)r * ld + 256 + part * 8));
    *reinterpret_cast<uint4*>(vs + r * RS + part * 8) = val;
  }
  // ---- k~: softmax over the tokens, one lane per channel
  {
    float kv[NT];
    float kmax = -INFINITY;
#pragma unroll
    for (int r = 0; r < NT; ++r) {
      kv[r] = -INFINITY;
      if (r < n) kv[r] = __bfloat162float(base[(int64_t)r * ld + 128 + lane]);
      kmax = fmaxf(kmax, kv[r]);
    }
    float ksum = 0.f;
    const float moff = -kmax * LOG2E;
#pragma unroll
    for (int r = 0; r < NT; ++r) {
      kv[r] = r < n ? fast_exp2(fmaf(kv[r], LOG2E, moff)) : 0.f;
      ksum += kv[r];
    }
    const float kinv = __fdividef(1.0f, ksum);
#pragma unroll
    for (int r = 0; r < NT; ++r) ks[r * RS + lane] = __float2bfloat16_rn(kv[r] * kinv);
  }
  // ---- q~: loaded in fragment layout; softmax over the 32 channels of a token = 8 local values + the quad
  uint32_t qa[MT][2][4];              // [token tile][k-step over d][a0..a3]
#pragma unroll
  for (int mq = 0; mq < MT; ++mq) {
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {  // tokens g (a0, a2) and g + 8 (a1, a3)
      const int tk = 16 * mq + 8 * hf + g;
      // every lane runs the quad shuffles (tokens >= n read token 0 and are zeroed afterwards)
      const bool ok = tk < n;
      const uint32_t* qp = reinterpret_cast<const uint32_t*>(base + (int64_t)(ok ? tk : 0) * ld + 2 * t);
      uint32_t raw[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) raw[j] = __ldg(qp + 4 * j);         // channels 8j + 2t, 8j + 2t + 1
      float v[8];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        v[2 * j] = __uint_as_float(raw[j] << 16);
        v[2 * j + 1] = __uint_as_float(raw[j] & 0xffff0000u);
      }
      float m = fmaxf(fmaxf(fmaxf(v[0], v[1]), fmaxf(v[2], v[3])), fmaxf(fmaxf(v[4], v[5]), fmaxf(v[6], v[7])));
      m = quad_max(m);
      const float moff = -m * LOG2E;
      float ssum = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        v[j] = fast_exp2(fmaf(v[j], LOG2E, moff));
        ssum += v[j];
      }
      ssum = quad_sum(ssum);
      const float sc = ok ? __fdividef(0.17677669529663687f, ssum) : 0.f;      // 32^-1/2 / sum
      uint32_t pk[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) pk[j] = pack_bf16x2(v[2 * j] * sc, v[2 * j + 1] * sc);
      // channel pair j lives in k-step j / 2, register a0/a1 (j even) or a2/a3 (j odd)
      qa[mq][0][hf] = pk[0];
      qa[mq][0][2 + hf] = pk[1];
      qa[mq][1][hf] = pk[2];
      qa[mq][1][2 + hf] = pk[3];
    }
  }
  __syncwarp();

  // ---- ctx^T[e][d] = sum_tok v[tok][e] k~[tok][d] : M = e (2 tiles), N = d (4 tiles), K = tokens (MT steps)
  float c[2][4][4];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt)
#pragma unroll
    for (int nt = 0; nt < 4; ++nt)
#pragma unroll
      for (int i = 0; i < 4; ++i) c[mt][nt][i] = 0.f;
  const uint32_t vs_a = (uint32_t)__cvta_generic_to_shared(vs), ks_a = (uint32_t)__cvta_generic_to_shared(ks);
  const int mi = lane >> 3, mr = lane & 7;          // ldmatrix: this lane addresses row mr of matrix mi
#pragma unroll
  for (int kt = 0; kt < MT; ++kt) {
    uint32_t a[2][4], b[2][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)    // matrices: (tok lo, e lo), (tok lo, e hi), (tok hi, e lo), (tok hi, e hi)
      ldsm_x4_trans(a[mt], vs_a + uint32_t(((16 * kt + 8 * (mi >> 1) + mr) * RS + 16 * mt + 8 * (mi & 1)) * 2));
#pragma unroll
    for (int np = 0; np < 2; ++np)    // matrices: (d tile 2np, tok lo), (2np, tok hi), (2np + 1, tok lo), (2np + 1, tok hi)
      ldsm_x4_trans(b[np], ks_a + uint32_t(((16 * kt + 8 * (mi & 1) + mr) * RS + 8 * (2 * np + (mi >> 1))) * 2));
#pragma unroll
    for (int mt = 0; mt < 2; ++mt)
#pragma unroll
      for (int nt = 0; nt < 4; ++nt) mma_bf16_16816(c[mt][nt], a[mt], b[nt >> 1][2 * (nt & 1)], b[nt >> 1][2 * (nt & 1) + 1]);
  }
  // ---- out[tok][e] = sum_d q~[tok][d] ctx[d][e] : M = tokens (MT tiles), N = e (4 tiles of 8), K = d (2 steps)
  uint32_t cb[4][2][2];               // [e tile][k-step][b0, b1]
#pragma unroll
  for (int eb = 0; eb < 4; ++eb)
#pragma unroll
    for (int ks2 = 0; ks2 < 2; ++ks2) {
      const int i0 = (eb & 1) * 2;
      cb[eb][ks2][0] = pack_bf16x2(c[eb >> 1][2 * ks2][i0], c[eb >> 1][2 * ks2][i0 + 1]);
      cb[eb][ks2][1] = pack_bf16x2(c[eb >> 1][2 * ks2 + 1][i0], c[eb >> 1][2 * ks2 + 1][i0 + 1]);
    }
#pragma unroll
  for (int mq = 0; mq < MT; ++mq) {
#pragma unroll
    for (int eb = 0; eb < 4; ++eb) {
      float o[4] = {0.f, 0.f, 0.f, 0.f};
      mma_bf16_16816(o, qa[mq][0], cb[eb][0][0], cb[eb][0][1]);
      mma_bf16_16816(o, qa[mq][1], cb[eb][1][0], cb[eb][1][1]);
      const int tk0 = 16 * mq + g, tk1 = tk0 + 8;
      bf16* op = out + (row0 + tk0) * ld_out + h * 32 + 8 * eb + 2 * t;
      if (tk0 < n) *reinterpret_cast<uint32_t*>(op) = pack_bf16x2(o[0], o[1]);
      if (tk1 < n) *reinterpret_cast<uint32_t*>(op + (int64_t)8 * ld_out) = pack_bf16x2(o[2], o[3]);
    }
  }
}

template <int NT> static size_t linattn_mma_smem() {
  return 4 * size_t(2 * 32 * (NT + 8) * 2 + NT * 40 * 2 + NT * 33 * 4);
}

template <typename T>
void launch_linattn(const T* qkv, int ld, T* out, int ld_out, int n_scenes, int n_obj, cudaStream_t s) {
  if constexpr (sizeof(T) == 2) {       // bf16 mode: warp-level tensor-core variants
    const bool vec_ok = (ld % 8 == 0) && (ld_out % 2 == 0) && ((uintptr_t)qkv % 16 == 0) && ((uintptr_t)out % 4 == 0);
    if (vec_ok && n_obj <= 32) {
      if (n_obj == 12) launch_pdl(k_linattn_frag<16, 12>, dim3(n_scenes), dim3(128), 0, s, qkv, ld, out, ld_out, n_scenes, n_obj);
      else if (n_obj == 21) launch_pdl(k_linattn_frag<32, 21>, dim3(n_scenes), dim3(128), 0, s, qkv, ld, out, ld_out, n_scenes, n_obj);
      else if (n_obj <= 16) launch_pdl(k_linattn_frag<16, 0>, dim3(n_scenes), dim3(128), 0, s, qkv, ld, out, ld_out, n_scenes, n_obj);
      else launch_pdl(k_linattn_frag<32, 0>, dim3(n_scenes), dim3(128), 0, s, qkv, ld, out, ld_out, n_scenes, n_obj);
      return;
    }
    if (n_obj <= 16) {
      k_linattn_mma<16><<<n_scenes, 128, linattn_mma_smem<16>(), s>>>(qkv, ld, out, ld_out, n_scenes, n_obj);
      return;
    }
    if (n_obj <= 32) {
      k_linattn_mma<32><<<n_scenes, 128, linattn_mma_smem<32>(), s>>>(qkv, ld, out, ld_out, n_scenes, n_obj);
      return;
    }
  }
  size_t smem = size_t(4) * 2 * n_obj * 32 * sizeof(float);
  if (n_obj == 12) k_linattn<T, 12, 12><<<n_scenes, 128, smem, s>>>(qkv, ld, out, ld_out, n_scenes, n_obj);
  else if (n_obj == 21) k_linattn<T, 21, 21><<<n_scenes, 128, smem, s>>>(qkv, ld, out, ld_out, n_scenes, n_obj);
  else if (n_obj <= 16) k_linattn<T, 16><<<n_scenes, 128, smem, s>>>(qkv, ld, out, ld_out, n_scenes, n_obj);
  else if (n_obj <= 32) k_linattn<T, 32><<<n_scenes, 128, smem, s>>>(qkv, ld, out, ld_out, n_scenes, n_obj);
  else k_linattn<T, 64><<<n_scenes, 128, smem, s>>>(qkv, ld, out, ld_out, n_scenes, n_obj);
}

template <typename T>
__global__ void __launch_bounds__(128) k_softattn(const T* __restrict__ qkv, int ld, T* __restrict__ out, int ld_out,
                                                  int n_scenes, int n) {
  extern __shared__ float sm[];
  const int lane = threadIdx.x & 31, h = threadIdx.x >> 5;
  const int scene = blockIdx.x;
  float* qs = sm + h * 3 * n * 33;
  float* ks = qs + n * 33;
  float* vs = ks + n * 33;
  const int64_t row0 = (int64_t)scene * n;
  const float scale = 0.17677669529663687f;
  for (int r = 0; r < n; ++r) {
    const T* p = qkv + (row0 + r) * ld + h * 32 + lane;
    qs[r * 33 + lane] = ldf(p) * scale;
    ks[r * 33 + lane] = ldf(p + 128);
    vs[r * 33 + lane] = ldf(p + 256);
  }
  __syncwarp();
  for (int i = 0; i < n; ++i) {
    // this lane scores keys j = lane and lane + 32 (n <= 64)
    float s0 = -INFINITY, s1 = -INFINITY;
    if (lane < n) {
      float a = 0.f;
#pragma unroll
      for (int d = 0; d < 32; ++d) a += qs[i * 33 + d] * ks[lane * 33 + d];
      s0 = a;
    }
    if (lane + 32 < n) {
      float a = 0.f;
#pragma unroll
      for (int d = 0; d < 32; ++d) a += qs[i * 33 + d] * ks[(lane + 32) * 33 + d];
      s1 = a;
    }
    float m = warp_max(fmaxf(s0, s1));
    float e0 = lane < n ? expf(s0 - m) : 0.f;
    float e1 = lane + 32 < n ? expf(s1 - m) : 0.f;
    float inv = 1.0f / warp_sum(e0 + e1);
    e0 *= inv;
    e1 *= inv;
    float o = 0.f;
    for (int j = 0; j < n; ++j) {
      float p = j < 32 ? __shfl_sync(0xffffffffu, e0, j) : __shfl_sync(0xffffffffu, e1, j - 32);
      o += p * vs[j * 33 + lane];
    }
    stf(out + (row0 + i) * ld_out + h * 32 + lane, o);
  }
}
// ---- tensor-core softmax attention (bf16 mode): S = q k^T on mma.sync with q and k loaded from global memory
// directly as A / B fragments, row softmax on the accumulator fragments (keys of a query live in one lane quad),
// O = P v with the probability fragments re-used as the A operand and v read through ldmatrix.trans.
template <int NT, int NE>
__global__ void __launch_bounds__(128) k_softattn_frag(const bf16* __restrict__ qkv, int ld, bf16* __restrict__ out,
                                                       int ld_out, int n_scenes, int n_rt) {
  constexpr int MT = NT / 16;
  constexpr int RS = 40;
  pdl_wait();
  const int n = NE > 0 ? NE : n_rt;
  __shared__ __align__(16) bf16 sm_v[4][NT * RS];
  const int lane = threadIdx.x & 31, h = threadIdx.x >> 5;
  const int g = lane >> 2, t = lane & 3;
  const int64_t row0 = (int64_t)blockIdx.x * n;
  bf16* vs = sm_v[h];
  const bf16* base = qkv + row0 * ld + h * 32;
#pragma unroll
  for (int idx = lane; idx < NT * 4; idx += 32) {
    const int r = idx >> 2, part = idx & 3;
    uint4 val = make_uint4(0u, 0u, 0u, 0u);
    if (r < n) val = __ldg(reinterpret_cast<const uint4*>(base + (int64_t)r * ld + 256 + part * 8));
    *reinterpret_cast<uint4*>(vs + r * RS + part * 8) = val;
  }
  // q (A operand: rows = query tokens) and k (B operand: columns = key tokens), both K = d in pairs 8j + 2t
  uint32_t qa[MT][2][4], kb[2 * MT][2][2];
#pragma unroll
  for (int tt = 0; tt < 2 * MT; ++tt) {           // token 8 tt + g
    const int tk = 8 * tt + g;
    uint32_t rq[4] = {0u, 0u, 0u, 0u}, rk[4] = {0u, 0u, 0u, 0u};
    if (tk < n) {
      const uint32_t* p = reinterpret_cast<const uint32_t*>(base + (int64_t)tk * ld + 2 * t);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        rq[j] = __ldg(p + 4 * j);
        rk[j] = __ldg(p + 64 + 4 * j);              // k block: + 128 channels
      }
    }
    qa[tt >> 1][0][tt & 1] = rq[0];
    qa[tt >> 1][0][2 + (tt & 1)] = rq[1];
    qa[tt >> 1][1][tt & 1] = rq[2];
    qa[tt >> 1][1][2 + (tt & 1)] = rq[3];
    kb[tt][0][0] = rk[0];
    kb[tt][0][1] = rk[1];
    kb[tt][1][0] = rk[2];
    kb[tt][1][1] = rk[3];
  }
  __syncwarp();
  const uint32_t vs_a = (uint32_t)__cvta_generic_to_shared(vs);
  const int mi = lane >> 3, mr = lane & 7;
  const float SCL = 0.17677669529663687f * 1.4426950408889634f;       // 32^-1/2 * log2(e)
#pragma unroll
  for (int mq = 0; mq < MT; ++mq) {
    float sc[2 * MT][4];
#pragma unroll
    for (int nt = 0; nt < 2 * MT; ++nt) {
      sc[nt][0] = sc[nt][1] = sc[nt][2] = sc[nt][3] = 0.f;
      mma_bf16_16816(sc[nt], qa[mq][0], kb[nt][0][0], kb[nt][0][1]);
      mma_bf16_16816(sc[nt], qa[mq][1], kb[nt][1][0], kb[nt][1][1]);
    }
    // rows g (values 0, 1) and g + 8 (values 2, 3); keys 8 nt + 2 t + {0, 1}
    float m0 = -INFINITY, m1 = -INFINITY;
#pragma unroll
    for (int nt = 0; nt < 2 * MT; ++nt)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        const bool ok = 8 * nt + 2 * t + e < n;
        sc[nt][e] = ok ? sc[nt][e] * SCL : -INFINITY;
        sc[nt][2 + e] = ok ? sc[nt][2 + e] * SCL : -INFINITY;
        m0 = fmaxf(m0, sc[nt][e]);
        m1 = fmaxf(m1, sc[nt][2 + e]);
      }
    m0 = quad_max(m0);
    m1 = quad_max(m1);
    float s0 = 0.f, s1 = 0.f;
#pragma unroll
    for (int nt = 0; nt < 2 * MT; ++nt)
#pragma unroll
      for (int e = 0; e < 2; ++e) {
        sc[nt][e] = fast_exp2(sc[nt][e] - m0);
        sc[nt][2 + e] = fast_exp2(sc[nt][2 + e] - m1);
        s0 += sc[nt][e];
        s1 += sc[nt][2 + e];
      }
    const float i0 = __fdividef(1.0f, quad_sum(s0)), i1 = __fdividef(1.0f, quad_sum(s1));
    uint32_t pa[MT][4];
#pragma unroll
    for (int kt = 0; kt < MT; ++kt) {
      pa[kt][0] = pack_bf16x2(sc[2 * kt][0] * i0, sc[2 * kt][1] * i0);
      pa[kt][1] = pack_bf16x2(sc[2 * kt][2] * i1, sc[2 * kt][3] * i1);
      pa[kt][2] = pack_bf16x2(sc[2 * kt + 1][0] * i0, sc[2 * kt + 1][1] * i0);
      pa[kt][3] = pack_bf16x2(sc[2 * kt + 1][2] * i1, sc[2 * kt + 1][3] * i1);
    }
    float o[4][4];
#pragma unroll
    for (int eb = 0; eb < 4; ++eb) o[eb][0] = o[eb][1] = o[eb][2] = o[eb][3] = 0.f;
#pragma unroll
    for (int kt = 0; kt < MT; ++kt) {
#pragma unroll
      for (int ep = 0; ep < 2; ++ep) {            // matrices: (e tile 2ep, tok lo), (2ep, tok hi), (2ep + 1, lo), (2ep + 1, hi)
        uint32_t b[4];
        ldsm_x4_trans(b, vs_a + uint32_t(((16 * kt + 8 * (mi & 1) + mr) * RS + 8 * (2 * ep + (mi >> 1))) * 2));
        mma_bf16_16816(o[2 * ep], pa[kt], b[0], b[1]);
        mma_bf16_16816(o[2 * ep + 1], pa[kt], b[2], b[3]);
      }
    }
    const int tk0 = 16 * mq + g, tk1 = tk0 + 8;
#pragma unroll
    for (int eb = 0; eb < 4; ++eb) {
      bf16* op = out + (row0 + tk0) * ld_out + h * 32 + 8 * eb + 2 * t;
      if (tk0 < n) *reinterpret_cast<uint32_t*>(op) = pack_bf16x2(o[eb][0], o[eb][1]);
      if (tk1 < n) *reinterpret_cast<uint32_t*>(op + (int64_t)8 * ld_out) = pack_bf16x2(o[eb][2], o[eb][3]);
    }
  }
}

template <typename T>
void launch_softattn(const T* qkv, int ld, T* out, int ld_out, int n_scenes, int n_obj, cudaStream_t s) {
  if constexpr (sizeof(T) == 2) {
    const bool vec_ok = (ld % 8 == 0) && (ld_out % 2 == 0) && ((uintptr_t)qkv % 16 == 0) && ((uintptr_t)out % 4 == 0);
    if (vec_ok && n_obj <= 32) {
      if (n_obj == 12) launch_pdl(k_softattn_frag<16, 12>, dim3(n_scenes), dim3(128), 0, s, qkv, ld, out, ld_out, n_scenes, n_obj);
      else if (n_obj == 21) launch_pdl(k_softattn_frag<32, 21>, dim3(n_scenes), dim3(128), 0, s, qkv, ld, out, ld_out, n_scenes, n_obj);
      else if (n_obj <= 16) launch_pdl(k_softattn_frag<16, 0>, dim3(n_scenes), dim3(128), 0, s, qkv, ld, out, ld_out, n_scenes, n_obj);
      else launch_pdl(k_softattn_frag<32, 0>, dim3(n_scenes), dim3(128), 0, s, qkv, ld, out, ld_out, n_scenes, n_obj);
      return;
    }
  }
  size_t smem = size_t(4) * 3 * n_obj * 33 * sizeof(float);
  k_softattn<T><<<n_scenes, 128, smem, s>>>(qkv, ld, out, ld_out, n_scenes, n_obj);
}

// cross linear attention -- text side: ctx[scene][h][d][e] (fp32) from the scene's L rows of k | v (storage type T).
// Once per sampling call (ds_set_context_cross) and once per training step.  One CTA per scene, one warp per head;
// the tokens are streamed in chunks (common.cuh), so every L the API accepts (<= 512) launches.
template <typename T>
__global__ void __launch_bounds__(128) k_xattn_prepare(const T* __restrict__ kv, int ld_kv, float* __restrict__ ctx, int L) {
  __shared__ float sm[4][2][XATTN_CHUNK][33];
  const int lane = threadIdx.x & 31, h = threadIdx.x >> 5;
  const int scene = blockIdx.x;
  const T* kvs = kv + (int64_t)scene * L * ld_kv;
  float kmax, kinv;
  xattn_k_stats(kvs, ld_kv, L, h, lane, kmax, kinv);
  float acc[32];      // lane = e: acc[d] = ctx[d][e]
  xattn_context<T, false>(kvs, ld_kv, L, h, lane, kmax, kinv, sm[h][0], sm[h][1], acc);
  float* o = ctx + ((int64_t)scene * 4 + h) * 1024;
#pragma unroll
  for (int d = 0; d < 32; ++d) o[d * 32 + lane] = acc[d];
}
template <typename T>
void launch_xattn_prepare(const T* kv, int ld_kv, float* ctx, int n_scenes, int L, cudaStream_t s) {
  if (n_scenes > 0) k_xattn_prepare<T><<<n_scenes, 128, 0, s>>>(kv, ld_kv, ctx, L);
}

template <typename T>
__global__ void __launch_bounds__(128) k_xattn_apply(const T* __restrict__ q, int ldq, const float* __restrict__ ctx,
                                                     T* __restrict__ out, int ld_out, int n_scenes, int n) {
  const int lane = threadIdx.x & 31, h = threadIdx.x >> 5;
  const int scene = blockIdx.x;
  const float* cx = ctx + ((int64_t)scene * 4 + h) * 1024;
  float c[32];
#pragma unroll
  for (int d = 0; d < 32; ++d) c[d] = cx[d * 32 + lane];
  const int64_t row0 = (int64_t)scene * n;
  const float scale = 0.17677669529663687f;
  for (int r = 0; r < n; ++r) {
    float qv = ldf(q + (row0 + r) * ldq + h * 32 + lane);
    float m = warp_max(qv);
    float e = expf(qv - m);
    float sm_ = warp_sum(e);
    float qn = e / sm_ * scale;
    float o = 0.f;
#pragma unroll
    for (int d = 0; d < 32; ++d) o += c[d] * __shfl_sync(0xffffffffu, qn, d);
    stf(out + (row0 + r) * ld_out + h * 32 + lane, o);
  }
}
template <typename T>
void launch_xattn_apply(const T* q, int ldq, const float* ctx, T* out, int ld_out, int n_scenes, int n_obj,
                        cudaStream_t s) {
  k_xattn_apply<T><<<n_scenes, 128, 0, s>>>(q, ldq, ctx, out, ld_out, n_scenes, n_obj);
}

// ------------------------------------------------------------------------------------------------
// time embedding helpers
// ------------------------------------------------------------------------------------------------
// out[t][k] = sin(t * f_k), out[t][half + k] = cos(t * f_k); f_k supplied by the host (denoise_net.py:132-139)
__global__ void k_sinusoid(float* __restrict__ out, const float* __restrict__ freq, int T, int dim) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int half = dim / 2;
  if (i >= T * half) return;
  int t = i / half, k = i % half;
  float a = float(t) * freq[k];
  out[(int64_t)t * dim + k] = sinf(a);
  out[(int64_t)t * dim + half + k] = cosf(a);
}
// frequencies f_k = exp(-k ln(1e4) / (half - 1)), computed on the host in fp32 like the reference's torch.exp on
// the CPU tensor (denoise_net.py:134-136); the caller owns the device copy (one per handle / device)
void sinusoid_freqs_host(int dim, float* hf) {
  const int half = dim / 2;
  const float neg_emb = -float(9.210340371976184 / double(half - 1));   // -(ln 1e4)/(half-1) as fp32
  for (int k = 0; k < half; ++k) hf[k] = expf(float(k) * neg_emb);
}
void launch_sinusoid(float* out, const float* freq_dev, int T, int dim, cudaStream_t s) {
  const int half = dim / 2;
  k_sinusoid<<<cdiv((int64_t)T * half, 256), 256, 0, s>>>(out, freq_dev, T, dim);
}
// per-sample variant (training: one timestep per scene): out[b][:] = sinusoid(t[b])
__global__ void k_sinusoid_t(float* __restrict__ out, const float* __restrict__ freq, const int* __restrict__ t, int B,
                             int dim) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  int half = dim / 2;
  if (i >= B * half) return;
  int b = i / half, k = i % half;
  float a = float(t[b]) * freq[k];
  out[(int64_t)b * dim + k] = sinf(a);
  out[(int64_t)b * dim + half + k] = cosf(a);
}
void launch_sinusoid_t(float* out, const float* freq_dev, const int* t_dev, int B, int dim, cudaStream_t s) {
  const int half = dim / 2;
  k_sinusoid_t<<<cdiv((int64_t)B * half, 256), 256, 0, s>>>(out, freq_dev, t_dev, B, dim);
}

__global__ void k_silu_f32(const float* __restrict__ in, float* __restrict__ out, int64_t n) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < n) out[i] = silu_exact(in[i]);
}
void launch_silu_f32(const float* in, float* out, int64_t n, cudaStream_t s) {
  k_silu_f32<<<cdiv(n, 256), 256, 0, s>>>(in, out, n);
}

__global__ void k_t_convert(const int64_t* __restrict__ t, int* __restrict__ out, int B) {
  int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < B) out[i] = int(t[i]);
}
void launch_t_convert(const int64_t* t, int* out, int B, cudaStream_t s) {
  k_t_convert<<<cdiv(B, 256), 256, 0, s>>>(t, out, B);
}

// ------------------------------------------------------------------------------------------------
// sampling-step kernels
// ------------------------------------------------------------------------------------------------
// N(0,1) for element quad `qd` of global scene `gs`; independent of how scenes are sharded over GPUs
__device__ __forceinline__ float4 randn4(uint64_t seed, uint64_t gs, uint32_t qd, uint32_t step, uint32_t stream_id) {
  uint4 ctr = make_uint4(qd, uint32_t(gs), uint32_t(gs >> 32), step | (stream_id << 24));
  uint4 r = philox4x32_10(ctr, make_uint2(uint32_t(seed), uint32_t(seed >> 32)));
  float2 a = box_muller(r.x, r.y), b = box_muller(r.z, r.w);
  return make_float4(a.x, a.y, b.x, b.y);
}

__global__ void k_begin_step(const StepCoef* __restrict__ coef, const StepState* __restrict__ st,
                             int* __restrict__ t_dev, float* __restrict__ x, const float* __restrict__ partial,
                             const float* __restrict__ partial_noise, int B, int n_obj, int d, int P) {
  const int step = st->step;
  const uint64_t seed = st->seed, scene_offset = st->scene_offset;
  const StepCoef c = coef[step];
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < B) t_dev[i] = c.t;
  if (P > 0) {
    const int per_part = P * d, quads = (per_part + 3) / 4;
    if (i < (int64_t)B * quads) {
      int b = int(i / quads), qd = int(i % quads);
      float z[4];
      if (partial_noise) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          int e = qd * 4 + k;
          z[k] = e < per_part ? partial_noise[((int64_t)step * B + b) * per_part + e] : 0.f;
        }
      } else {
        float4 r = randn4(seed, scene_offset + b, qd, step, 1u);
        z[0] = r.x; z[1] = r.y; z[2] = r.z; z[3] = r.w;
      }
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        int e = qd * 4 + k;
        if (e < per_part)
          x[(int64_t)b * n_obj * d + e] =
              __fadd_rn(__fmul_rn(c.q_a, partial[(int64_t)b * per_part + e]), __fmul_rn(c.q_b, z[k]));
      }
    }
  }
}
void launch_begin_step(const StepCoef* coef, const StepState* st, int* t_dev, float* x, const float* partial,
                       const float* partial_noise, int B, int n_obj, int d, int P, cudaStream_t s) {
  int64_t n = B;
  if (P > 0) {
    int64_t m = (int64_t)B * ((P * d + 3) / 4);
    if (m > n) n = m;
  }
  k_begin_step<<<cdiv(n, 256), 256, 0, s>>>(coef, st, t_dev, x, partial, partial_noise, B, n_obj, d, P);
}

// x0 = a_x*x + a_o*out ; clamp ; x' = c_0*x0 + c_x*x + c_z*z   (rounding order of diffusion_ddpm.py:236-240,
// 294-297, 348-350: every product and sum rounded separately, no FMA contraction)
template <typename T>
__global__ void k_step_update(const StepCoef* __restrict__ coef, StepState* st, float* __restrict__ x,
                              const T* __restrict__ model_out, int ld_out, const float* __restrict__ noise, int B,
                              int n_obj, int d, int clip) {
  const int step = st->step;
  const uint64_t seed = st->seed, scene_offset = st->scene_offset;
  const StepCoef c = coef[step];
  const int per_scene = n_obj * d, quads = (per_scene + 3) / 4;
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i < (int64_t)B * quads) {
    int b = int(i / quads), qd = int(i % quads);
    float z[4] = {0.f, 0.f, 0.f, 0.f};
    if (c.c_z != 0.f) {
      if (noise) {
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          int e = qd * 4 + k;
          if (e < per_scene) z[k] = noise[((int64_t)step * B + b) * per_scene + e];
        }
      } else {
        float4 r = randn4(seed, scene_offset + b, qd, step, 0u);
        z[0] = r.x; z[1] = r.y; z[2] = r.z; z[3] = r.w;
      }
    }
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      int e = qd * 4 + k;
      if (e < per_scene) {
        int o = e / d, ch = e % d;
        int64_t xi = (int64_t)b * per_scene + e;
        float xv = x[xi];
        float ov = ldf(model_out + ((int64_t)b * n_obj + o) * ld_out + ch);
        float x0 = __fadd_rn(__fmul_rn(c.a_x, xv), __fmul_rn(c.a_o, ov));
        if (clip) x0 = fminf(fmaxf(x0, -1.0f), 1.0f);
        float mean = __fadd_rn(__fmul_rn(c.c_0, x0), __fmul_rn(c.c_x, xv));
        x[xi] = __fadd_rn(mean, __fmul_rn(c.c_z, z[k]));
      }
    }
  }
  // the last block to finish advances the loop counter (every block has read st->step by then)
  __syncthreads();
  if (threadIdx.x == 0) {
    __threadfence();
    unsigned int done = atomicAdd(&st->done, 1u);
    if (done == gridDim.x - 1) {
      st->done = 0;
      st->step = step + 1;
      __threadfence();
    }
  }
}
template <typename T>
void launch_step_update(const StepCoef* coef, StepState* st, float* x, const T* model_out, int ld_out,
                        const float* noise, int B, int n_obj, int d, int clip, cudaStream_t s) {
  int64_t n = (int64_t)B * ((n_obj * d + 3) / 4);
  k_step_update<T><<<cdiv(n, 256), 256, 0, s>>>(coef, st, x, model_out, ld_out, noise, B, n_obj, d, clip);
}

__global__ void k_randn(float* __restrict__ out, int B, int per_scene, uint64_t seed, uint64_t scene_offset,
                        uint32_t stream_id) {
  const int quads = (per_scene + 3) / 4;
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * quads) return;
  int b = int(i / quads), qd = int(i % quads);
  float4 r = randn4(seed, scene_offset + b, qd, 0xFFFFFFu, stream_id);
  float z[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    int e = qd * 4 + k;
    if (e < per_scene) out[(int64_t)b * per_scene + e] = z[k];
  }
}
void launch_randn(float* out, int B, int per_scene, uint64_t seed, uint64_t scene_offset, uint32_t stream_id,
                  cudaStream_t s) {
  int64_t n = (int64_t)B * ((per_scene + 3) / 4);
  k_randn<<<cdiv(n, 256), 256, 0, s>>>(out, B, per_scene, seed, scene_offset, stream_id);
}

template <typename T>
__global__ void k_p_sample(const float* __restrict__ x, const T* __restrict__ model_out, int ld_out,
                           const int* __restrict__ t, const float* __restrict__ noise, float* __restrict__ out,
                           const float* __restrict__ a_x, const float* __restrict__ a_o,
                           const float* __restrict__ c1, const float* __restrict__ c2,
                           const float* __restrict__ sigma, int B, int n_obj, int d, int clip) {
  const int per_scene = n_obj * d;
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * per_scene) return;
  int b = int(i / per_scene), e = int(i % per_scene);
  int o = e / d, ch = e % d;
  int tt = t[b];
  float xv = x[i];
  float ov = ldf(model_out + ((int64_t)b * n_obj + o) * ld_out + ch);
  float x0 = __fadd_rn(__fmul_rn(a_x[tt], xv), __fmul_rn(a_o[tt], ov));
  if (clip) x0 = fminf(fmaxf(x0, -1.0f), 1.0f);
  float mean = __fadd_rn(__fmul_rn(c1[tt], x0), __fmul_rn(c2[tt], xv));
  out[i] = __fadd_rn(mean, __fmul_rn(sigma[tt], noise[i]));
}
template <typename T>
void launch_p_sample(const float* x, const T* model_out, int ld_out, const int* t, const float* noise, float* out,
                     const float* a_x, const float* a_o, const float* c1, const float* c2, const float* sigma, int B,
                     int n_obj, int d, int clip, cudaStream_t s) {
  int64_t n = (int64_t)B * n_obj * d;
  k_p_sample<T><<<cdiv(n, 256), 256, 0, s>>>(x, model_out, ld_out, t, noise, out, a_x, a_o, c1, c2, sigma, B, n_obj,
                                             d, clip);
}

__global__ void k_q_sample(const float* __restrict__ x0, const int64_t* __restrict__ t,
                           const float* __restrict__ noise, float* __restrict__ out,
                           const float* __restrict__ sqrt_ac, const float* __restrict__ sqrt_1mac, int B,
                           int per_scene) {
  int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * per_scene) return;
  int tt = int(t[i / per_scene]);
  out[i] = __fadd_rn(__fmul_rn(sqrt_ac[tt], x0[i]), __fmul_rn(sqrt_1mac[tt], noise[i]));
}
void launch_q_sample(const float* x0, const int64_t* t, const float* noise, float* out, const float* sqrt_ac,
                     const float* sqrt_1mac, int B, int per_scene, cudaStream_t s) {
  int64_t n = (int64_t)B * per_scene;
  k_q_sample<<<cdiv(n, 256), 256, 0, s>>>(x0, t, noise, out, sqrt_ac, sqrt_1mac, B, per_scene);
}

// ------------------------------------------------------------------------------------------------
// p_losses value: one CTA (128 threads) per scene
// parts[b] = {bbox, trans, size, angle, class, object, objfeat, liou, bbox_iou}
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(128) k_p_losses(const float* __restrict__ x0, const float* __restrict__ noise,
                                                  const float* __restrict__ x_t, const T* __restrict__ model_out,
                                                  int ld_out, const int64_t* __restrict__ t,
                                                  const float* __restrict__ sqrt_ac,
                                                  const float* __restrict__ sqrt_1mac,
                                                  const float* __restrict__ sqrt_recip_ac,
                                                  const float* __restrict__ sqrt_recipm1_ac,
                                                  const float* __restrict__ loss_weight,
                                                  const float* __restrict__ alphas_cumprod, LossArgs a,
                                                  float* __restrict__ losses, float* __restrict__ parts) {
  __shared__ float acc[8];          // trans, size, angle, class, object, objfeat, full, (unused)
  __shared__ float box[64][6];      // clamped, descaled corners
  __shared__ float valid[64];
  __shared__ float iou_acc[3];      // sum(iou*mask), sum(mask), unused
  const int b = blockIdx.x, tid = threadIdx.x;
  const int tt = int(t[b]);
  const int n = a.n_obj, d = a.d;
  if (tid < 8) acc[tid] = 0.f;
  if (tid < 3) iou_acc[tid] = 0.f;
  __syncthreads();
  const float sa = sqrt_ac[tt], sb = sqrt_1mac[tt];
  const int bb = a.trans + a.size + a.angle;
  const int c_end = bb + a.cls;
  const int obj_lo = a.objn > 0 ? c_end : c_end - 1, obj_hi = a.objn > 0 ? c_end + a.objn : c_end;
  float l[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int e = tid; e < n * d; e += 128) {
    int o = e / d, ch = e % d;
    int64_t gi = (int64_t)b * n * d + e;
    float x0v = x0[gi], nz = noise[gi];
    float target;
    if (a.mean_type == 0) target = nz;
    else if (a.mean_type == 1) target = x0v;
    else target = __fadd_rn(__fmul_rn(sa, nz), -__fmul_rn(sb, x0v));
    float ov = ldf(model_out + ((int64_t)b * n + o) * ld_out + ch);
    float df = target - ov;
    float se = df * df;
    l[6] += se;
    if (a.arrange) {
      if (ch < a.trans) l[0] += se; else l[2] += se;
    } else {
      if (ch < a.trans) l[0] += se;
      else if (ch < a.trans + a.size) l[1] += se;
      else if (ch < bb) l[2] += se;
      else if (ch < c_end) l[3] += se;
      if (ch >= obj_lo && ch < obj_hi) l[4] += se;
      if (ch >= c_end + a.objn) l[5] += se;
    }
  }
#pragma unroll
  for (int k = 0; k < 7; ++k) {
    float v = warp_sum(l[k]);
    if ((tid & 31) == 0) atomicAdd(&acc[k], v);
  }
  // IoU regulariser (diffusion_ddpm.py:600-635, loss.py:7-102)
  if (a.loss_iou && !a.arrange) {
    for (int o = tid; o < n; o += 128) {
      float rec[7];
      int chs[7] = {0, 1, 2, a.trans, a.trans + 1, a.trans + 2, a.objn > 0 ? c_end : c_end - 1};
      for (int k = 0; k < 7; ++k) {
        int64_t gi = ((int64_t)b * n + o) * d + chs[k];
        float xt = x_t[gi];
        float ov = ldf(model_out + ((int64_t)b * n + o) * ld_out + chs[k]);
        float r;
        if (a.mean_type == 0) r = __fadd_rn(__fmul_rn(sqrt_recip_ac[tt], xt), -__fmul_rn(sqrt_recipm1_ac[tt], ov));
        else if (a.mean_type == 1) r = ov;
        else r = __fadd_rn(__fmul_rn(sa, xt), -__fmul_rn(sb, ov));
        rec[k] = fminf(fmaxf(r, -1.0f), 1.0f);
      }
      valid[o] = a.objn > 0 ? (rec[6] >= 0.f ? 1.f : 0.f) : (rec[6] <= 0.f ? 1.f : 0.f);
      for (int k = 0; k < 3; ++k) {
        float tr = (rec[k] + 1.0f) / 2.0f * (a.bounds[3 + k] - a.bounds[k]) + a.bounds[k];
        float sz = (rec[3 + k] + 1.0f) / 2.0f * (a.bounds[9 + k] - a.bounds[6 + k]) + a.bounds[6 + k];
        box[o][k] = tr - sz;
        box[o][3 + k] = tr + sz;
      }
    }
    __syncthreads();
    float si = 0.f, sm_ = 0.f;
    for (int p = tid; p < n * n; p += 128) {
      int i = p / n, j = p % n;
      float vi = (box[i][3] - box[i][0]) * (box[i][4] - box[i][1]) * (box[i][5] - box[i][2]);
      float vj = (box[j][3] - box[j][0]) * (box[j][4] - box[j][1]) * (box[j][5] - box[j][2]);
      float w0 = fmaxf(fminf(box[i][3], box[j][3]) - fmaxf(box[i][0], box[j][0]), 0.f);
      float w1 = fmaxf(fminf(box[i][4], box[j][4]) - fmaxf(box[i][1], box[j][1]), 0.f);
      float w2 = fmaxf(fminf(box[i][5], box[j][5]) - fmaxf(box[i][2], box[j][2]), 0.f);
      float inter = w0 * w1 * w2;
      float uni = fmaxf(vi + vj - inter, 1e-6f);
      float m = valid[i] * valid[j];
      si += inter / uni * m;
      sm_ += m;
    }
    si = warp_sum(si);
    sm_ = warp_sum(sm_);
    if ((tid & 31) == 0) {
      atomicAdd(&iou_acc[0], si);
      atomicAdd(&iou_acc[1], sm_);
    }
  }
  __syncthreads();
  if (tid == 0) {
    float* p = parts + (int64_t)b * 9;
    const float fn = float(n);
    float loss;
    if (a.arrange) {
      float ltr = acc[0] / (fn * a.trans), lan = acc[2] / (fn * a.angle);
      loss = a.loss_separate ? ltr + lan : acc[6] / (fn * d);
      for (int k = 0; k < 9; ++k) p[k] = 0.f;
      p[1] = ltr;
      p[3] = lan;
      losses[b] = loss * loss_weight[tt];
      return;
    }
    float ltr = acc[0] / (fn * a.trans), lsz = acc[1] / (fn * a.size), lan = acc[2] / (fn * a.angle);
    float lbb = (acc[0] + acc[1] + acc[2]) / (fn * bb), lcl = acc[3] / (fn * a.cls);
    float lob = acc[4] / (fn * (a.objn > 0 ? a.objn : 1));
    float lof = a.feat > 0 ? acc[5] / (fn * a.feat) : 0.f;
    if (a.loss_separate) {
      loss = lbb + lcl;
      if (a.objn > 0) loss += lob;
      if (a.feat > 0) loss += lof;
    } else {
      loss = acc[6] / (fn * d);
    }
    loss *= loss_weight[tt];
    float liou = 0.f, iou_avg = 0.f;
    if (a.loss_iou) {
      float den = iou_acc[1] + 1e-6f;
      iou_avg = iou_acc[0] / den;
      liou = alphas_cumprod[tt] * 0.1f * iou_acc[0] / den;
      loss += liou;
    }
    p[0] = lbb; p[1] = ltr; p[2] = lsz; p[3] = lan; p[4] = lcl; p[5] = lob; p[6] = lof; p[7] = liou; p[8] = iou_avg;
    losses[b] = loss;
  }
}
template <typename T>
void launch_p_losses(const float* x0, const float* noise, const float* x_t, const T* model_out, int ld_out,
                     const int64_t* t, const float* sqrt_ac, const float* sqrt_1mac, const float* sqrt_recip_ac,
                     const float* sqrt_recipm1_ac, const float* loss_weight, const float* alphas_cumprod, LossArgs a,
                     float* losses, float* parts, int B, cudaStream_t s) {
  k_p_losses<T><<<B, 128, 0, s>>>(x0, noise, x_t, model_out, ld_out, t, sqrt_ac, sqrt_1mac, sqrt_recip_ac,
                                  sqrt_recipm1_ac, loss_weight, alphas_cumprod, a, losses, parts);
}

__global__ void k_loss_dict_mean(const float* __restrict__ parts, float* __restrict__ dict9, int B) {
  int k = blockIdx.x;      // 9 blocks
  float s = 0.f;
  for (int b = threadIdx.x; b < B; b += blockDim.x) s += parts[(int64_t)b * 9 + k];
  __shared__ float red[8];
  s = warp_sum(s);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tot = 0.f;
    for (int w = 0; w < int(blockDim.x >> 5); ++w) tot += red[w];
    dict9[k] = tot / float(B);
  }
}
void launch_loss_dict_mean(const float* parts, float* dict9, int B, cudaStream_t s) {
  k_loss_dict_mean<<<9, 256, 0, s>>>(parts, dict9, B);
}

// raise the dynamic shared-memory limit of the attention cores once, outside any stream capture
void init_pointwise_attrs() {
  const int lim = 200 * 1024;
  cudaFuncSetAttribute(k_linattn<float, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim);
  cudaFuncSetAttribute(k_linattn<bf16, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim);
  cudaFuncSetAttribute(k_softattn<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim);
  cudaFuncSetAttribute(k_softattn<bf16>, cudaFuncAttributeMaxDynamicSharedMemorySize, lim);
}

// ---- explicit instantiations ----
#define INST(T)                                                                                                   \
  template void launch_pack_input<T>(const float*, T*, int, int, int, cudaStream_t);                              \
  template void launch_unpack_output<T>(const T*, int, float*, int, int, cudaStream_t);                           \
  template void launch_groupnorm<T>(const T*, int, T*, int, const float*, const float*, FilmRef, const T*, int,   \
                                    int, int, int, int, cudaStream_t);                                            \
  template void launch_layernorm<T>(const T*, int, T*, int, const float*, const T*, int, int, int, cudaStream_t); \
  template void launch_linattn<T>(const T*, int, T*, int, int, int, cudaStream_t);                                \
  template void launch_softattn<T>(const T*, int, T*, int, int, int, cudaStream_t);                               \
  template void launch_xattn_apply<T>(const T*, int, const float*, T*, int, int, int, cudaStream_t);              \
  template void launch_xattn_prepare<T>(const T*, int, float*, int, int, cudaStream_t);                           \
  template void launch_step_update<T>(const StepCoef*, StepState*, float*, const T*, int, const float*, int, int, \
                                      int, int, cudaStream_t);                                                    \
  template void launch_p_sample<T>(const float*, const T*, int, const int*, const float*, float*, const float*,   \
                                   const float*, const float*, const float*, const float*, int, int, int, int,    \
                                   cudaStream_t);                                                                 \
  template void launch_p_losses<T>(const float*, const float*, const float*, const T*, int, const int64_t*,       \
                                   const float*, const float*, const float*, const float*, const float*,          \
                                   const float*, LossArgs, float*, float*, int, cudaStream_t);
INST(float)
INST(bf16)


// ------------------------------------------------------------------------------------------------
// object retrieval: nearest catalogue model per generated object (SURVEY 8f row 3)
// ------------------------------------------------------------------------------------------------
// Reference: ThreedFutureDataset.get_closest_furniture_to_objfeats_and_size / _to_objfeats / _to_box
// (scene_synthesis/datasets/threed_future_dataset.py:28-77): among the catalogue entries of the query's class,
// the entry minimising (size mse, feature mse) lexicographically (np.lexsort((mses_feat, mses_size)): size is the
// primary key), ties -> first entry in catalogue order.  The catalogue is stored grouped by class (stable), so a
// class is a contiguous range.  One warp per query; squared distances are accumulated in EXACTLY numpy's order for
// float32 `np.sum(d ** 2, axis=-1)` (8 running partials over strided elements, then the fixed 3-level tree; plain
// left-to-right below 8 elements), products and sums rounded separately -- so the keys, not only the winners, are
// bit-identical to the host computation and ties resolve identically.
namespace {
__device__ __forceinline__ float np_sum_sq_diff(const float* __restrict__ a, const float* __restrict__ b, int n) {
  if (n < 8) {
    float s = 0.f;      // numpy: res = 0.; res += a[i]
    for (int i = 0; i < n; ++i) { const float d = __fsub_rn(a[i], b[i]); s = __fadd_rn(s, __fmul_rn(d, d)); }
    return s;
  }
  float r[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { const float d = __fsub_rn(a[j], b[j]); r[j] = __fmul_rn(d, d); }
  int i = 8;
  for (; i + 8 <= n; i += 8) {
#pragma unroll
    for (int j = 0; j < 8; ++j) { const float d = __fsub_rn(a[i + j], b[i + j]); r[j] = __fadd_rn(r[j], __fmul_rn(d, d)); }
  }
  float res = __fadd_rn(__fadd_rn(__fadd_rn(r[0], r[1]), __fadd_rn(r[2], r[3])),
                        __fadd_rn(__fadd_rn(r[4], r[5]), __fadd_rn(r[6], r[7])));
  for (; i < n; ++i) { const float d = __fsub_rn(a[i], b[i]); res = __fadd_rn(res, __fmul_rn(d, d)); }
  return res;
}
struct RKey { float k0, k1; int idx; };
__device__ __forceinline__ bool rkey_less(const RKey& a, const RKey& b) {
  if (a.k0 != b.k0) return a.k0 < b.k0;
  if (a.k1 != b.k1) return a.k1 < b.k1;
  return a.idx < b.idx;
}
}  // namespace

// mode 0: (size, feature) lexicographic; 1: feature only; 2: size only
__global__ void k_retrieve(const int* __restrict__ class_start, int n_classes, const float* __restrict__ cat_feat,
                           const float* __restrict__ cat_size, int feat_dim, int size_dim,
                           const int64_t* __restrict__ q_label, const float* __restrict__ q_feat,
                           const float* __restrict__ q_size, int Q, int mode, int64_t* __restrict__ out) {
  const int q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (q >= Q) return;
  const int64_t lab = q_label[q];
  RKey best;
  best.k0 = INFINITY; best.k1 = INFINITY; best.idx = 0x7fffffff;
  if (lab >= 0 && lab < n_classes) {
    const int beg = class_start[lab], end = class_start[lab + 1];
    const float* qf = q_feat ? q_feat + (int64_t)q * feat_dim : nullptr;
    const float* qs = q_size ? q_size + (int64_t)q * size_dim : nullptr;
    for (int e = beg + lane; e < end; e += 32) {
      RKey k;
      k.idx = e;
      const float mf = mode != 2 ? np_sum_sq_diff(cat_feat + (int64_t)e * feat_dim, qf, feat_dim) : 0.f;
      const float ms = mode != 1 ? np_sum_sq_diff(cat_size + (int64_t)e * size_dim, qs, size_dim) : 0.f;
      k.k0 = mode == 1 ? mf : ms;
      k.k1 = mode == 0 ? mf : 0.f;
      if (rkey_less(k, best)) best = k;
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    RKey other;
    other.k0 = __shfl_xor_sync(0xffffffffu, best.k0, o);
    other.k1 = __shfl_xor_sync(0xffffffffu, best.k1, o);
    other.idx = __shfl_xor_sync(0xffffffffu, best.idx, o);
    if (rkey_less(other, best)) best = other;
  }
  if (lane == 0) out[q] = best.idx == 0x7fffffff ? -1 : (int64_t)best.idx;
}
void launch_retrieve(const int* class_start, int n_classes, const float* cat_feat, const float* cat_size, int feat_dim,
                     int size_dim, const int64_t* q_label, const float* q_feat, const float* q_size, int Q, int mode,
                     int64_t* out, cudaStream_t s) {
  const int wpb = 8;
  k_retrieve<<<cdiv(Q, wpb), wpb * 32, 0, s>>>(class_start, n_classes, cat_feat, cat_size, feat_dim, size_dim, q_label,
                                                q_feat, q_size, Q, mode, out);
}

}  // namespace ds
