// Backward kernels of the native training path (reference: the autograd graph behind
// GaussianDiffusion.p_losses, scene_synthesis/networks/diffusion_ddpm.py:520-652, through Unet1D.forward,
// denoise_net.py:507-593).  Every op of the training step program (plan.cpp, train mode: one op per reference
// layer, all intermediates kept) has its hand-written adjoint here:
//   GEMM            k_gemm_nn (dX = dY W), k_gemm_tn (dW = dY^T X, split over tokens, fp32 atomics), k_colsum (db)
//   GELU / SiLU     k_act / k_act_bwd
//   Block           k_gn_bwd: GroupNorm(8) + affine + FiLM + SiLU (+ residual passthrough) in one pass per (scene, group)
//   LayerNorm       k_ln_bwd
//   LinearAttention k_linattn_bwd, Attention k_softattn_bwd (one warp per (scene, head), everything in shared memory)
//   LinearAttentionCross k_xattn_bwd (one CTA per scene, one warp per head; text tokens streamed in chunks)
//   loss            k_p_losses_bwd: d(loss)/d(model output) for the MSE terms and the IoU regulariser
//   weights         k_ws_unpack: packed-matrix gradients -> named tensors through the weight-standardisation adjoint
//   optimizer       k_adam, k_sumsq (global gradient norm for clip_grad_norm_)
// Storage type T is float (parity mode) or bf16; all arithmetic and every gradient w.r.t. a parameter is fp32.
#include <stdlib.h>

#include "../../include/diffuscene_b200.h"
#include "kernels.cuh"

namespace ds {

static inline int64_t cdiv64(int64_t a, int64_t b) { return (a + b - 1) / b; }

// ------------------------------------------------------------------------------------------------
// GEMMs
// ------------------------------------------------------------------------------------------------
// D[M, N] (= | +=) A[M, K] * B[K, N]; A row-major (k contiguous), B row-major (n contiguous)
template <typename TA, typename TB, typename TD>
__global__ void __launch_bounds__(256) k_gemm_nn(const TA* __restrict__ A, int lda, const TB* __restrict__ B, int ldb,
                                                 TD* __restrict__ D, int ldd, int M, int N, int K, int accumulate) {
  __shared__ __align__(16) float As[16][64 + 4];
  __shared__ __align__(16) float Bs[16][64 + 4];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  const int arow = tid >> 2, ak = (tid & 3) * 4;       // A: 64 rows x 16 k
  const int bk = tid >> 4, bn = (tid & 15) * 4;        // B: 16 k x 64 n
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int kb = 0; kb < K; kb += 16) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int m = m0 + arow, kk = kb + ak + i;
      As[ak + i][arow] = (m < M && kk < K) ? ldf(A + (int64_t)m * lda + kk) : 0.f;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int kk = kb + bk, n = n0 + bn + i;
      Bs[bk][bn + i] = (kk < K && n < N) ? ldf(B + (int64_t)kk * ldb + n) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const float4 av = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float a[4] = {av.x, av.y, av.z, av.w}, b[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= N) continue;
      TD* p = D + (int64_t)m * ldd + n;
      stf(p, accumulate ? ldf(p) + acc[i][j] : acc[i][j]);
    }
  }
}
template <typename TA, typename TB, typename TD>
void launch_gemm_nn(const TA* A, int lda, const TB* B, int ldb, TD* D, int ldd, int M, int N, int K, int accumulate,
                    cudaStream_t s) {
  if (M <= 0 || N <= 0 || K <= 0) return;
  dim3 grid((N + 63) / 64, (M + 63) / 64);
  k_gemm_nn<TA, TB, TD><<<grid, 256, 0, s>>>(A, lda, B, ldb, D, ldd, M, N, K, accumulate);
}

// D[Ka, Kb] += A[M, Ka]^T * B[M, Kb]  (fp32 D, atomics: the token dimension is split over blockIdx.z)
template <typename TA, typename TB>
__global__ void __launch_bounds__(256) k_gemm_tn(const TA* __restrict__ A, int lda, const TB* __restrict__ B, int ldb,
                                                 float* __restrict__ D, int ldd, int M, int Ka, int Kb, int m_chunk) {
  __shared__ __align__(16) float As[16][64 + 4];
  __shared__ __align__(16) float Bs[16][64 + 4];
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int a0 = blockIdx.y * 64, b0 = blockIdx.x * 64;
  const int mb = blockIdx.z * m_chunk, me = min(M, mb + m_chunk);
  const int lm = tid >> 4, lc = (tid & 15) * 4;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (int m = mb; m < me; m += 16) {
    const int mm = m + lm;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      As[lm][lc + i] = (mm < me && a0 + lc + i < Ka) ? ldf(A + (int64_t)mm * lda + a0 + lc + i) : 0.f;
      Bs[lm][lc + i] = (mm < me && b0 + lc + i < Kb) ? ldf(B + (int64_t)mm * ldb + b0 + lc + i) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int k = 0; k < 16; ++k) {
      const float4 av = *reinterpret_cast<const float4*>(&As[k][ty * 4]);
      const float4 bv = *reinterpret_cast<const float4*>(&Bs[k][tx * 4]);
      const float a[4] = {av.x, av.y, av.z, av.w}, b[4] = {bv.x, bv.y, bv.z, bv.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int a = a0 + ty * 4 + i;
    if (a >= Ka) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int b = b0 + tx * 4 + j;
      if (b < Kb) atomicAdd(D + (int64_t)a * ldd + b, acc[i][j]);
    }
  }
}
template <typename TA, typename TB>
void launch_gemm_tn(const TA* A, int lda, const TB* B, int ldb, float* D, int ldd, int M, int Ka, int Kb, cudaStream_t s) {
  if (M <= 0 || Ka <= 0 || Kb <= 0) return;
  const int tiles = ((Ka + 63) / 64) * ((Kb + 63) / 64);
  int splits = (4 * 148 + tiles - 1) / tiles;                   // ~4 blocks per SM
  int m_chunk = ((M + splits - 1) / splits + 15) / 16 * 16;
  if (m_chunk < 64) m_chunk = 64;
  splits = (M + m_chunk - 1) / m_chunk;
  dim3 grid((Kb + 63) / 64, (Ka + 63) / 64, splits);
  k_gemm_tn<TA, TB><<<grid, 256, 0, s>>>(A, lda, B, ldb, D, ldd, M, Ka, Kb, m_chunk);
}

// out[n] += sum_m A[m, n]
template <typename T>
__global__ void k_colsum(const T* __restrict__ A, int lda, float* __restrict__ out, int M, int N, int m_chunk) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const int mb = blockIdx.y * m_chunk, me = min(M, mb + m_chunk);
  float s = 0.f;
  for (int m = mb; m < me; ++m) s += ldf(A + (int64_t)m * lda + n);
  atomicAdd(out + n, s);
}
template <typename T>
void launch_colsum(const T* A, int lda, float* out, int M, int N, cudaStream_t s) {
  if (M <= 0 || N <= 0) return;
  const int m_chunk = 256;
  dim3 grid((N + 127) / 128, (M + m_chunk - 1) / m_chunk);
  k_colsum<T><<<grid, 128, 0, s>>>(A, lda, out, M, N, m_chunk);
}

// dst (= | +=) src over an [M, N] block
template <typename T>
__global__ void k_add_block(const T* __restrict__ src, int lds, T* __restrict__ dst, int ldd, int M, int N, int accumulate) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)M * N) return;
  const int m = int(i / N), n = int(i % N);
  const float v = ldf(src + (int64_t)m * lds + n);
  T* p = dst + (int64_t)m * ldd + n;
  stf(p, accumulate ? ldf(p) + v : v);
}
template <typename T>
void launch_add_block(const T* src, int lds, T* dst, int ldd, int M, int N, int accumulate, cudaStream_t s) {
  const int64_t n = (int64_t)M * N;
  if (n > 0) k_add_block<T><<<cdiv64(n, 256), 256, 0, s>>>(src, lds, dst, ldd, M, N, accumulate);
}

// ------------------------------------------------------------------------------------------------
// activations (exact forms in both precisions: training follows torch's erf-GELU / SiLU)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float act_fwd(float x, int act) { return act == ACT_GELU ? gelu_erf(x) : (act == ACT_SILU ? silu_exact(x) : x); }
__device__ __forceinline__ float act_grad(float x, int act) {
  if (act == ACT_GELU) {
    const float cdf = 0.5f * (1.0f + erff(x * 0.70710678118654752440f));
    return cdf + x * 0.39894228040143267794f * expf(-0.5f * x * x);
  }
  if (act == ACT_SILU) {
    const float sg = 1.0f / (1.0f + expf(-x));
    return sg * (1.0f + x * (1.0f - sg));
  }
  return 1.0f;
}
template <typename T>
__global__ void k_act(const T* __restrict__ z, int ldz, T* __restrict__ out, int ldo, int M, int N, int act) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)M * N) return;
  const int m = int(i / N), n = int(i % N);
  stf(out + (int64_t)m * ldo + n, act_fwd(ldf(z + (int64_t)m * ldz + n), act));
}
template <typename T>
void launch_act(const T* z, int ldz, T* out, int ldo, int M, int N, int act, cudaStream_t s) {
  const int64_t n = (int64_t)M * N;
  if (n > 0) k_act<T><<<cdiv64(n, 256), 256, 0, s>>>(z, ldz, out, ldo, M, N, act);
}
// dz = dy * act'(z)
template <typename T>
__global__ void k_act_bwd(const T* __restrict__ z, int ldz, const T* __restrict__ dy, int ldy, T* __restrict__ dz, int lddz,
                          int M, int N, int act) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)M * N) return;
  const int m = int(i / N), n = int(i % N);
  stf(dz + (int64_t)m * lddz + n, ldf(dy + (int64_t)m * ldy + n) * act_grad(ldf(z + (int64_t)m * ldz + n), act));
}
template <typename T>
void launch_act_bwd(const T* z, int ldz, const T* dy, int ldy, T* dz, int lddz, int M, int N, int act, cudaStream_t s) {
  const int64_t n = (int64_t)M * N;
  if (n > 0) k_act_bwd<T><<<cdiv64(n, 256), 256, 0, s>>>(z, ldz, dy, ldy, dz, lddz, M, N, act);
}

// ---- register-resident variants for the shipped shapes (64 channels per group, N = 12 / 21 objects) -----------------
// A warp owns one (scene, group) and a lane owns the channel pair (2 lane, 2 lane + 1) of the group for ALL tokens of
// the scene: the group is read from HBM exactly once into registers (4-byte bf16x2 / 8-byte float2 loads, 128 / 256 B
// per warp instruction), statistics, adjoint sums and outputs are computed from registers.  The generic kernels above
// make three passes over global memory; these are bound by one read and one write of the activation.
template <typename T> struct Pair;
template <> struct Pair<float> {
  static __device__ __forceinline__ float2 ld(const float* p) { return *reinterpret_cast<const float2*>(p); }
  static __device__ __forceinline__ void st(float* p, float2 v) { *reinterpret_cast<float2*>(p) = v; }
};
template <> struct Pair<bf16> {
  static __device__ __forceinline__ float2 ld(const bf16* p) { return __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(p)); }
  static __device__ __forceinline__ void st(bf16* p, float2 v) { *reinterpret_cast<__nv_bfloat162*>(p) = __floats2bfloat162_rn(v.x, v.y); }
};
__device__ __forceinline__ const float* film_row(const FilmRef& film, int scene, int r, int64_t row) {
  if (film.mode == FILM_TIME) return film.base + (int64_t)film.t[scene] * film.row_stride;
  if (film.mode == FILM_OBJECT) return film.base + (int64_t)r * film.row_stride;
  if (film.mode == FILM_TOKEN) return film.base + row * film.row_stride;
  return nullptr;
}

template <typename T, int NOBJ>
__global__ void __launch_bounds__(256) k_gn_fwd_reg(const T* __restrict__ in, int ld_in, T* __restrict__ out, int ld_out,
                                                    const float* __restrict__ gamma, const float* __restrict__ beta,
                                                    FilmRef film, const T* __restrict__ res, int ld_res, int n_scenes, int C) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n_scenes * 8) return;
  const int scene = warp >> 3, grp = warp & 7, ch = grp * 64 + 2 * lane;
  const int64_t row0 = (int64_t)scene * NOBJ;
  float2 v[NOBJ];
  float s = 0.f;
#pragma unroll
  for (int r = 0; r < NOBJ; ++r) {
    v[r] = Pair<T>::ld(in + (row0 + r) * ld_in + ch);
    s += v[r].x + v[r].y;
  }
  const float inv = 1.0f / float(NOBJ * 64);
  const float mean = warp_sum(s) * inv;
  float q = 0.f;
#pragma unroll
  for (int r = 0; r < NOBJ; ++r) {
    const float a = v[r].x - mean, b = v[r].y - mean;
    q = fmaf(a, a, q);
    q = fmaf(b, b, q);
  }
  const float rstd = 1.0f / sqrtf(warp_sum(q) * inv + 1e-5f);
  const float2 ga = *reinterpret_cast<const float2*>(gamma + ch), be = *reinterpret_cast<const float2*>(beta + ch);
#pragma unroll
  for (int r = 0; r < NOBJ; ++r) {
    const int64_t row = row0 + r;
    float2 y = make_float2(fmaf((v[r].x - mean) * rstd, ga.x, be.x), fmaf((v[r].y - mean) * rstd, ga.y, be.y));
    if (const float* fr = film_row(film, scene, r, row)) {
      const float2 sc = *reinterpret_cast<const float2*>(fr + ch), sh = *reinterpret_cast<const float2*>(fr + C + ch);
      y = make_float2(fmaf(y.x, sc.x + 1.0f, sh.x), fmaf(y.y, sc.y + 1.0f, sh.y));
    }
    y = make_float2(silu_exact(y.x), silu_exact(y.y));
    if (res) {
      const float2 rv = Pair<T>::ld(res + row * ld_res + ch);
      y.x += rv.x;
      y.y += rv.y;
    }
    Pair<T>::st(out + row * ld_out + ch, y);
  }
}

template <typename T, int NOBJ>
__global__ void __launch_bounds__(256) k_gn_bwd_reg(const T* __restrict__ c, int ldc, const T* __restrict__ dy, int ldy,
                                                    T* __restrict__ dc, int lddc, T* __restrict__ dres, int ldr,
                                                    int res_accumulate, const float* __restrict__ gamma,
                                                    const float* __restrict__ beta, FilmRef film, float* __restrict__ dgamma,
                                                    float* __restrict__ dbeta, float* __restrict__ dfilm,
                                                    int64_t dfilm_row_stride, int n_scenes, int C) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n_scenes * 8) return;
  const int scene = warp >> 3, grp = warp & 7, ch = grp * 64 + 2 * lane;
  const int64_t row0 = (int64_t)scene * NOBJ;
  float2 xh[NOBJ], gy[NOBJ];
  float s = 0.f;
#pragma unroll
  for (int r = 0; r < NOBJ; ++r) {
    xh[r] = Pair<T>::ld(c + (row0 + r) * ldc + ch);
    gy[r] = Pair<T>::ld(dy + (row0 + r) * ldy + ch);
    s += xh[r].x + xh[r].y;
  }
  const float inv = 1.0f / float(NOBJ * 64);
  const float mean = warp_sum(s) * inv;
  float q = 0.f;
#pragma unroll
  for (int r = 0; r < NOBJ; ++r) {
    xh[r].x -= mean;
    xh[r].y -= mean;
    q = fmaf(xh[r].x, xh[r].x, q);
    q = fmaf(xh[r].y, xh[r].y, q);
  }
  const float rstd = 1.0f / sqrtf(warp_sum(q) * inv + 1e-5f);
  const float2 ga = *reinterpret_cast<const float2*>(gamma + ch), be = *reinterpret_cast<const float2*>(beta + ch);
  float2 dga = make_float2(0.f, 0.f), dbe = dga, dsc = dga, dsh = dga;
  float g1 = 0.f, g2 = 0.f;
  // gy[r] is turned into dxhat in place; the residual passthrough leaves first
#pragma unroll
  for (int r = 0; r < NOBJ; ++r) {
    const int64_t row = row0 + r;
    if (dres) {
      T* p = dres + row * ldr + ch;
      float2 o = gy[r];
      if (res_accumulate) {
        const float2 old = Pair<T>::ld(p);
        o.x += old.x;
        o.y += old.y;
      }
      Pair<T>::st(p, o);
    }
    xh[r].x *= rstd;
    xh[r].y *= rstd;
    const float2 u = make_float2(fmaf(xh[r].x, ga.x, be.x), fmaf(xh[r].y, ga.y, be.y));
    float2 sc = make_float2(1.0f, 1.0f), sh = make_float2(0.f, 0.f);
    if (const float* fr = film_row(film, scene, r, row)) {
      const float2 a = *reinterpret_cast<const float2*>(fr + ch);
      sc = make_float2(a.x + 1.0f, a.y + 1.0f);
      sh = *reinterpret_cast<const float2*>(fr + C + ch);
    }
    const float2 dw = make_float2(gy[r].x * act_grad(fmaf(u.x, sc.x, sh.x), ACT_SILU), gy[r].y * act_grad(fmaf(u.y, sc.y, sh.y), ACT_SILU));
    if (film.mode == FILM_TIME) {
      dsc.x = fmaf(dw.x, u.x, dsc.x); dsc.y = fmaf(dw.y, u.y, dsc.y);
      dsh.x += dw.x; dsh.y += dw.y;
    } else if (film.mode == FILM_OBJECT) {
      atomicAdd(dfilm + (int64_t)r * dfilm_row_stride + ch, dw.x * u.x);
      atomicAdd(dfilm + (int64_t)r * dfilm_row_stride + ch + 1, dw.y * u.y);
      atomicAdd(dfilm + (int64_t)r * dfilm_row_stride + C + ch, dw.x);
      atomicAdd(dfilm + (int64_t)r * dfilm_row_stride + C + ch + 1, dw.y);
    } else if (film.mode == FILM_TOKEN) {
      *reinterpret_cast<float2*>(dfilm + row * dfilm_row_stride + ch) = make_float2(dw.x * u.x, dw.y * u.y);
      *reinterpret_cast<float2*>(dfilm + row * dfilm_row_stride + C + ch) = dw;
    }
    const float2 du = make_float2(dw.x * sc.x, dw.y * sc.y);
    dga.x = fmaf(du.x, xh[r].x, dga.x); dga.y = fmaf(du.y, xh[r].y, dga.y);
    dbe.x += du.x; dbe.y += du.y;
    gy[r] = make_float2(du.x * ga.x, du.y * ga.y);      // dxhat
    g1 += gy[r].x + gy[r].y;
    g2 = fmaf(gy[r].x, xh[r].x, g2);
    g2 = fmaf(gy[r].y, xh[r].y, g2);
  }
  atomicAdd(dgamma + ch, dga.x); atomicAdd(dgamma + ch + 1, dga.y);
  atomicAdd(dbeta + ch, dbe.x); atomicAdd(dbeta + ch + 1, dbe.y);
  if (film.mode == FILM_TIME) {
    *reinterpret_cast<float2*>(dfilm + (int64_t)scene * dfilm_row_stride + ch) = dsc;
    *reinterpret_cast<float2*>(dfilm + (int64_t)scene * dfilm_row_stride + C + ch) = dsh;
  }
  g1 = warp_sum(g1) * inv;
  g2 = warp_sum(g2) * inv;
#pragma unroll
  for (int r = 0; r < NOBJ; ++r)
    Pair<T>::st(dc + (row0 + r) * lddc + ch, make_float2(rstd * (gy[r].x - g1 - xh[r].x * g2), rstd * (gy[r].y - g1 - xh[r].y * g2)));
}
template <typename T>
bool launch_gn_fwd_reg(const T* in, int ld_in, T* out, int ld_out, const float* gamma, const float* beta, FilmRef film,
                       const T* res, int ld_res, int n_scenes, int n_obj, int C, int groups, cudaStream_t s) {
  if (groups != 8 || C != 512 || (n_obj != 12 && n_obj != 21) || n_scenes <= 0) return false;
  const int64_t warps = (int64_t)n_scenes * 8;
  if (n_obj == 12) k_gn_fwd_reg<T, 12><<<cdiv64(warps, 8), 256, 0, s>>>(in, ld_in, out, ld_out, gamma, beta, film, res, ld_res, n_scenes, C);
  else k_gn_fwd_reg<T, 21><<<cdiv64(warps, 8), 256, 0, s>>>(in, ld_in, out, ld_out, gamma, beta, film, res, ld_res, n_scenes, C);
  return true;
}

// ------------------------------------------------------------------------------------------------
// Block backward: y = SiLU( (GN(c) * gamma + beta) * (scale + 1) + shift ) (+ res)        (denoise_net.py:160-176)
// one warp per (scene, group of C / 8 channels): lane <-> channels lane, lane + 32 of the group, loop over the tokens
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void k_gn_bwd(const T* __restrict__ c, int ldc, const T* __restrict__ dy, int ldy, T* __restrict__ dc, int lddc,
                         T* __restrict__ dres, int ldr, int res_accumulate, const float* __restrict__ gamma,
                         const float* __restrict__ beta, FilmRef film, float* __restrict__ dgamma,
                         float* __restrict__ dbeta, float* __restrict__ dfilm, int64_t dfilm_row_stride, int n_scenes,
                         int n_obj, int C, int groups) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (warp >= n_scenes * groups) return;
  const int scene = warp / groups, grp = warp % groups, cg = C / groups;      // cg = 64
  const int64_t row0 = (int64_t)scene * n_obj;
  const float inv = 1.0f / float(cg * n_obj);
  // pass 1: statistics
  float s = 0.f, ss = 0.f;
  for (int r = 0; r < n_obj; ++r)
    for (int ch = lane; ch < cg; ch += 32) {
      const float v = ldf(c + (row0 + r) * ldc + grp * cg + ch);
      s += v;
      ss = fmaf(v, v, ss);
    }
  s = warp_sum(s);
  ss = warp_sum(ss);
  const float mean = s * inv;
  const float rstd = rsqrtf(fmaxf(ss * inv - mean * mean, 0.f) + 1e-5f);
  // pass 2: dw, per-channel sums, group sums of dxhat and dxhat * xhat
  float g1 = 0.f, g2 = 0.f;
  for (int ch = lane; ch < cg; ch += 32) {
    const int n = grp * cg + ch;
    const float ga = gamma[n], be = beta[n];
    float dga = 0.f, dbe = 0.f, dsc_s = 0.f, dsh_s = 0.f;       // per-channel accumulators over the scene's tokens
    for (int r = 0; r < n_obj; ++r) {
      const int64_t row = row0 + r;
      const float xh = (ldf(c + row * ldc + n) - mean) * rstd;
      const float u = fmaf(xh, ga, be);
      float sc = 1.0f, sh = 0.f;
      const float* fr = nullptr;
      if (film.mode == FILM_TIME) fr = film.base + (int64_t)film.t[scene] * film.row_stride;
      else if (film.mode == FILM_OBJECT) fr = film.base + (int64_t)r * film.row_stride;
      else if (film.mode == FILM_TOKEN) fr = film.base + row * film.row_stride;
      if (fr) { sc = fr[n] + 1.0f; sh = fr[C + n]; }
      const float w = fmaf(u, sc, sh);
      const float gy = ldf(dy + row * ldy + n);
      const float dw = gy * act_grad(w, ACT_SILU);
      const float du = dw * sc;
      dga = fmaf(du, xh, dga);
      dbe += du;
      const float dxh = du * ga;
      g1 += dxh;
      g2 = fmaf(dxh, xh, g2);
      if (film.mode == FILM_TIME) { dsc_s = fmaf(dw, u, dsc_s); dsh_s += dw; }
      else if (film.mode == FILM_OBJECT) {
        atomicAdd(dfilm + (int64_t)r * dfilm_row_stride + n, dw * u);
        atomicAdd(dfilm + (int64_t)r * dfilm_row_stride + C + n, dw);
      } else if (film.mode == FILM_TOKEN) {
        dfilm[row * dfilm_row_stride + n] = dw * u;
        dfilm[row * dfilm_row_stride + C + n] = dw;
      }
    }
    atomicAdd(dgamma + n, dga);
    atomicAdd(dbeta + n, dbe);
    if (film.mode == FILM_TIME) {      // one row per scene: plain stores (this warp owns (scene, these channels))
      dfilm[(int64_t)scene * dfilm_row_stride + n] = dsc_s;
      dfilm[(int64_t)scene * dfilm_row_stride + C + n] = dsh_s;
    }
  }
  g1 = warp_sum(g1) * inv;
  g2 = warp_sum(g2) * inv;
  // pass 3: dc = rstd * (dxhat - mean(dxhat) - xhat * mean(dxhat * xhat)); residual passthrough
  for (int r = 0; r < n_obj; ++r)
    for (int ch = lane; ch < cg; ch += 32) {
      const int n = grp * cg + ch;
      const int64_t row = row0 + r;
      const float xh = (ldf(c + row * ldc + n) - mean) * rstd;
      const float u = fmaf(xh, gamma[n], beta[n]);
      float sc = 1.0f, sh = 0.f;
      const float* fr = nullptr;
      if (film.mode == FILM_TIME) fr = film.base + (int64_t)film.t[scene] * film.row_stride;
      else if (film.mode == FILM_OBJECT) fr = film.base + (int64_t)r * film.row_stride;
      else if (film.mode == FILM_TOKEN) fr = film.base + row * film.row_stride;
      if (fr) { sc = fr[n] + 1.0f; sh = fr[C + n]; }
      const float w = fmaf(u, sc, sh);
      const float gy = ldf(dy + row * ldy + n);
      const float dxh = gy * act_grad(w, ACT_SILU) * sc * gamma[n];
      stf(dc + row * lddc + n, rstd * (dxh - g1 - xh * g2));
      if (dres) {
        T* p = dres + row * ldr + n;
        stf(p, res_accumulate ? ldf(p) + gy : gy);
      }
    }
}
template <typename T>
void launch_gn_bwd(const T* c, int ldc, const T* dy, int ldy, T* dc, int lddc, T* dres, int ldr, int res_accumulate,
                   const float* gamma, const float* beta, FilmRef film, float* dgamma, float* dbeta, float* dfilm,
                   int64_t dfilm_row_stride, int n_scenes, int n_obj, int C, int groups, cudaStream_t s) {
  const int64_t warps = (int64_t)n_scenes * groups;
  if (warps <= 0) return;
  if (groups == 8 && C == 512 && n_obj == 12)
    k_gn_bwd_reg<T, 12><<<cdiv64(warps, 8), 256, 0, s>>>(c, ldc, dy, ldy, dc, lddc, dres, ldr, res_accumulate, gamma, beta, film,
                                                         dgamma, dbeta, dfilm, dfilm_row_stride, n_scenes, C);
  else if (groups == 8 && C == 512 && n_obj == 21)
    k_gn_bwd_reg<T, 21><<<cdiv64(warps, 8), 256, 0, s>>>(c, ldc, dy, ldy, dc, lddc, dres, ldr, res_accumulate, gamma, beta, film,
                                                         dgamma, dbeta, dfilm, dfilm_row_stride, n_scenes, C);
  else
    k_gn_bwd<T><<<cdiv64(warps, 8), 256, 0, s>>>(c, ldc, dy, ldy, dc, lddc, dres, ldr, res_accumulate, gamma, beta, film,
                                                 dgamma, dbeta, dfilm, dfilm_row_stride, n_scenes, n_obj, C, groups);
}

// ------------------------------------------------------------------------------------------------
// LayerNorm backward: y = (x - mean) * rstd * g (+ res)   (denoise_net.py:93-102); warp per token row
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(256) k_ln_bwd(const T* __restrict__ x, int ldx, const T* __restrict__ dy, int ldy,
                                                T* __restrict__ dx, int lddx, int dx_accumulate, T* __restrict__ dres,
                                                int ldr, int res_accumulate, const float* __restrict__ g,
                                                float* __restrict__ dg, int M, int C, int rows_per_block) {
  __shared__ float dg_s[1024];                       // C <= 1024
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int n = threadIdx.x; n < C; n += blockDim.x) dg_s[n] = 0.f;
  __syncthreads();
  const float inv = 1.0f / float(C);
  const int64_t r0 = (int64_t)blockIdx.x * rows_per_block;
  for (int64_t row = r0 + warp; row < r0 + rows_per_block && row < M; row += 8) {
    float s = 0.f, ss = 0.f;
    for (int n = lane; n < C; n += 32) {
      const float v = ldf(x + row * ldx + n);
      s += v;
      ss = fmaf(v, v, ss);
    }
    s = warp_sum(s);
    ss = warp_sum(ss);
    const float mean = s * inv, rstd = rsqrtf(fmaxf(ss * inv - mean * mean, 0.f) + 1e-5f);
    float g1 = 0.f, g2 = 0.f;
    for (int n = lane; n < C; n += 32) {
      const float xh = (ldf(x + row * ldx + n) - mean) * rstd;
      const float gy = ldf(dy + row * ldy + n);
      const float dxh = gy * g[n];
      g1 += dxh;
      g2 = fmaf(dxh, xh, g2);
      atomicAdd(&dg_s[n], gy * xh);                  // shared-memory atomics: 8 warps per address at most
    }
    g1 = warp_sum(g1) * inv;
    g2 = warp_sum(g2) * inv;
    for (int n = lane; n < C; n += 32) {
      const float xh = (ldf(x + row * ldx + n) - mean) * rstd;
      const float gy = ldf(dy + row * ldy + n);
      const float v = rstd * (gy * g[n] - g1 - xh * g2);
      T* p = dx + row * lddx + n;
      stf(p, dx_accumulate ? ldf(p) + v : v);
      if (dres) {
        T* q = dres + row * ldr + n;
        stf(q, res_accumulate ? ldf(q) + gy : gy);
      }
    }
  }
  __syncthreads();
  for (int n = threadIdx.x; n < C; n += blockDim.x) atomicAdd(dg + n, dg_s[n]);
}
template <typename T>
void launch_ln_bwd(const T* x, int ldx, const T* dy, int ldy, T* dx, int lddx, int dx_accumulate, T* dres, int ldr,
                   int res_accumulate, const float* g, float* dg, int M, int C, cudaStream_t s) {
  const int rpb = 64;
  if (M > 0) k_ln_bwd<T><<<cdiv64((int64_t)M, rpb), 256, 0, s>>>(x, ldx, dy, ldy, dx, lddx, dx_accumulate, dres, ldr,
                                                                    res_accumulate, g, dg, M, C, rpb);
}

// ------------------------------------------------------------------------------------------------
// attention cores: one warp per (scene, head); 4 heads x 32 channels; N <= 32 tokens
// qkv row layout: [q (4 x 32) | k (4 x 32) | v (4 x 32)]
// ------------------------------------------------------------------------------------------------
constexpr int ATT_MAXN = 32;
// LinearAttention (denoise_net.py:208-235): q = softmax over the 32 head channels * 32^-1/2, k = softmax over tokens,
// ctx[d][e] = sum_n k[d][n] v[e][n], out[e][n] = sum_d ctx[d][e] q[d][n]
template <typename T>
__global__ void __launch_bounds__(32) k_linattn_bwd(const T* __restrict__ qkv, int ld, const T* __restrict__ dout, int ldo,
                                                     T* __restrict__ dqkv, int lddq, int n_scenes, int N) {
  __shared__ float sm[1][5][ATT_MAXN][33];       // q~ (softmaxed, unscaled), k (softmaxed), v, dout, scratch
  const int w = 0, lane = threadIdx.x & 31;
  const int task = blockIdx.x;
  if (task >= n_scenes * 4) return;
  const int scene = task >> 2, h = task & 3;
  const int64_t row0 = (int64_t)scene * N;
  float (*Q)[33] = sm[w][0];
  float (*Kk)[33] = sm[w][1];
  float (*V)[33] = sm[w][2];
  float (*DO)[33] = sm[w][3];
  float (*X)[33] = sm[w][4];
  const float scale = 0.17677669529663687f;      // 32^-1/2
  // load; lane = head channel
  for (int n = 0; n < N; ++n) {
    const T* r = qkv + (row0 + n) * ld;
    Q[n][lane] = ldf(r + h * 32 + lane);
    Kk[n][lane] = ldf(r + 128 + h * 32 + lane);
    V[n][lane] = ldf(r + 256 + h * 32 + lane);
    DO[n][lane] = ldf(dout + (row0 + n) * ldo + h * 32 + lane);
  }
  __syncwarp();
  // q softmax over channels (per token: across lanes)
  for (int n = 0; n < N; ++n) {
    const float v = Q[n][lane];
    const float mx = warp_max(v);
    const float e = expf(v - mx);
    Q[n][lane] = e / warp_sum(e);
  }
  // k softmax over tokens (per channel: in-lane)
  {
    float mx = -INFINITY;
    for (int n = 0; n < N; ++n) mx = fmaxf(mx, Kk[n][lane]);
    float sum = 0.f;
    for (int n = 0; n < N; ++n) { const float e = expf(Kk[n][lane] - mx); Kk[n][lane] = e; sum += e; }
    const float is = 1.0f / sum;
    for (int n = 0; n < N; ++n) Kk[n][lane] *= is;
  }
  __syncwarp();
  // lane = d: ctx[d][e] and dctx[d][e] for all e, kept in registers
  float ctx[32], dctx[32];
#pragma unroll
  for (int e = 0; e < 32; ++e) { ctx[e] = 0.f; dctx[e] = 0.f; }
  for (int n = 0; n < N; ++n) {
    const float kd = Kk[n][lane], qd = Q[n][lane] * scale;
#pragma unroll
    for (int e = 0; e < 32; ++e) {
      ctx[e] = fmaf(kd, V[n][e], ctx[e]);
      dctx[e] = fmaf(DO[n][e], qd, dctx[e]);
    }
  }
  // dq[d][n] = sum_e ctx[d][e] dout[e][n]  (scaled q);  dk[d][n] = sum_e dctx[d][e] v[e][n]
  float dkk[ATT_MAXN];
  for (int n = 0; n < N; ++n) {
    float dq = 0.f, dk = 0.f;
#pragma unroll
    for (int e = 0; e < 32; ++e) {
      dq = fmaf(ctx[e], DO[n][e], dq);
      dk = fmaf(dctx[e], V[n][e], dk);
    }
    X[n][lane] = dq * scale;            // gradient w.r.t. the softmaxed (unscaled) q
    dkk[n] = dk;
  }
  // dv[e][n] = sum_d dctx[d][e] k[d][n]: lane = e needs column e of dctx -> transpose through shared memory
  __syncwarp();
  // q softmax backward (across lanes per token)
  for (int n = 0; n < N; ++n) {
    const float qs = Q[n][lane], g = X[n][lane];
    const float dot = warp_sum(g * qs);
    stf(dqkv + (row0 + n) * lddq + h * 32 + lane, qs * (g - dot));
  }
  // k softmax backward (in-lane over tokens)
  {
    float dot = 0.f;
    for (int n = 0; n < N; ++n) dot = fmaf(dkk[n], Kk[n][lane], dot);
    for (int n = 0; n < N; ++n) stf(dqkv + (row0 + n) * lddq + 128 + h * 32 + lane, Kk[n][lane] * (dkk[n] - dot));
  }
  __syncwarp();
  // dctx -> X[d][e] (reuse scratch rows 0..31 as [d][e]); N <= 32 rows are allocated, d needs 32 rows
  for (int e = 0; e < 32; ++e) X[lane][e] = dctx[e];
  __syncwarp();
  for (int n = 0; n < N; ++n) {
    float dv = 0.f;
#pragma unroll 8
    for (int d = 0; d < 32; ++d) dv = fmaf(X[d][lane], Kk[n][d], dv);
    stf(dqkv + (row0 + n) * lddq + 256 + h * 32 + lane, dv);
  }
}
template <typename T>
void launch_linattn_bwd(const T* qkv, int ld, const T* dout, int ldo, T* dqkv, int lddq, int n_scenes, int N, cudaStream_t s) {
  if (n_scenes > 0) k_linattn_bwd<T><<<n_scenes * 4, 32, 0, s>>>(qkv, ld, dout, ldo, dqkv, lddq, n_scenes, N);
}

// LinearAttentionCross core (denoise_net.py:261-297): q^ = softmax over the 32 head channels * 32^-1/2 (per object),
// k^ = softmax over the L text tokens, ctx[d][e] = sum_l k^[l][d] v[l][e], out[n][e] = sum_d ctx[d][e] q^[n][d].
// One CTA per scene, one warp per head.  q^, k^ and ctx are recomputed from q and the layer's k | v; the text tokens
// are streamed in chunks of XATTN_CHUNK, so shared memory is fixed for every L.  Writes dq (overwrites, or adds when
// dq_accumulate) and d(k | v) of the layer: dctx[d][e] = sum_n q^[n][d] dout[n][e], dv[l][e] = sum_d k^[l][d] dctx[d][e],
// dk^[l][d] = sum_e dctx[d][e] v[l][e], dk = k^ (dk^ - sum_l dk^ k^).
template <typename T>
__global__ void __launch_bounds__(128) k_xattn_bwd(const T* __restrict__ q, int ldq, const T* __restrict__ dout, int ldo,
                                                   const T* __restrict__ kv, int ld_kv, T* __restrict__ dq, int lddq,
                                                   int dq_accumulate, T* __restrict__ dkv, int ld_dkv, int n_obj, int L) {
  __shared__ float sm[4][2][XATTN_CHUNK][33];
  const int lane = threadIdx.x & 31, h = threadIdx.x >> 5;
  const int scene = blockIdx.x;
  float (*A)[33] = sm[h][0];
  float (*Bv)[33] = sm[h][1];
  const T* kvs = kv + (int64_t)scene * L * ld_kv;
  T* dkvs = dkv + (int64_t)scene * L * ld_dkv;
  const float scale = 0.17677669529663687f;      // 32^-1/2
  float kmax, kinv;
  xattn_k_stats(kvs, ld_kv, L, h, lane, kmax, kinv);
  float ctx[32];      // lane = d: ctx[e] = ctx[d][e]
  xattn_context<T, true>(kvs, ld_kv, L, h, lane, kmax, kinv, A, Bv, ctx);
  // object side (n_obj <= 32 rows): A = softmax(q) unscaled, Bv = dout; lane = channel
  const int64_t row0 = (int64_t)scene * n_obj;
  for (int n = 0; n < n_obj; ++n) {
    const float v = ldf(q + (row0 + n) * ldq + h * 32 + lane);
    const float e = expf(v - warp_max(v));
    A[n][lane] = e / warp_sum(e);
    Bv[n][lane] = ldf(dout + (row0 + n) * ldo + h * 32 + lane);
  }
  __syncwarp();
  float dctx[32];      // lane = d
#pragma unroll
  for (int e = 0; e < 32; ++e) dctx[e] = 0.f;
  for (int n = 0; n < n_obj; ++n) {
    const float qs = A[n][lane];
    float g = 0.f;
#pragma unroll
    for (int e = 0; e < 32; ++e) {
      const float de = Bv[n][e];
      dctx[e] = fmaf(qs * scale, de, dctx[e]);
      g = fmaf(ctx[e], de, g);
    }
    g *= scale;      // gradient w.r.t. the softmaxed (unscaled) q
    const float r = qs * (g - warp_sum(g * qs));
    T* p = dq + (row0 + n) * lddq + h * 32 + lane;
    stf(p, dq_accumulate ? ldf(p) + r : r);
  }
  __syncwarp();
  // lane = e needs column e of dctx for dv: transpose through the first tile
#pragma unroll
  for (int e = 0; e < 32; ++e) A[lane][e] = dctx[e];
  __syncwarp();
  float dctxT[32];      // lane = e: dctxT[d] = dctx[d][e]
#pragma unroll
  for (int d = 0; d < 32; ++d) dctxT[d] = A[d][lane];
  __syncwarp();
  // pass 1 over the tokens: dv, and S[d] = sum_l dk^[l][d] k^[l][d]; pass 2: dk
  float S = 0.f;
  for (int pass = 0; pass < 2; ++pass) {
    for (int l0 = 0; l0 < L; l0 += XATTN_CHUNK) {
      const int nl = min(XATTN_CHUNK, L - l0);
      for (int l = 0; l < nl; ++l) {
        const T* p = kvs + (int64_t)(l0 + l) * ld_kv + h * 32 + lane;
        A[l][lane] = expf(ldf(p) - kmax) * kinv;
        Bv[l][lane] = ldf(p + 128);
      }
      __syncwarp();
      for (int l = 0; l < nl; ++l) {
        const float kd = A[l][lane];
        float dkh = 0.f;
#pragma unroll
        for (int e = 0; e < 32; ++e) dkh = fmaf(dctx[e], Bv[l][e], dkh);
        T* o = dkvs + (int64_t)(l0 + l) * ld_dkv + h * 32 + lane;
        if (pass == 0) {
          S = fmaf(dkh, kd, S);
          float dv = 0.f;
#pragma unroll
          for (int d = 0; d < 32; ++d) dv = fmaf(A[l][d], dctxT[d], dv);
          stf(o + 128, dv);
        } else {
          stf(o, kd * (dkh - S));
        }
      }
      __syncwarp();
    }
  }
}
template <typename T>
void launch_xattn_bwd(const T* q, int ldq, const T* dout, int ldo, const T* kv, int ld_kv, T* dq, int lddq, int dq_accumulate,
                      T* dkv, int ld_dkv, int n_scenes, int n_obj, int L, cudaStream_t s) {
  if (n_scenes > 0) k_xattn_bwd<T><<<n_scenes, 128, 0, s>>>(q, ldq, dout, ldo, kv, ld_kv, dq, lddq, dq_accumulate, dkv, ld_dkv, n_obj, L);
}

// Attention (denoise_net.py:237-259): sim[i][j] = scale * sum_d q[d][i] k[d][j], attn = softmax_j, out[i][d] = sum_j attn[i][j] v[j][d]
template <typename T>
__global__ void __launch_bounds__(32) k_softattn_bwd(const T* __restrict__ qkv, int ld, const T* __restrict__ dout, int ldo,
                                                      T* __restrict__ dqkv, int lddq, int n_scenes, int N) {
  __shared__ float sm[1][6][ATT_MAXN][33];       // q, k, v, dout, attn, dsim
  const int w = 0, lane = threadIdx.x & 31;
  const int task = blockIdx.x;
  if (task >= n_scenes * 4) return;
  const int scene = task >> 2, h = task & 3;
  const int64_t row0 = (int64_t)scene * N;
  float (*Q)[33] = sm[w][0];
  float (*Kk)[33] = sm[w][1];
  float (*V)[33] = sm[w][2];
  float (*DO)[33] = sm[w][3];
  float (*P)[33] = sm[w][4];
  float (*DS)[33] = sm[w][5];
  const float scale = 0.17677669529663687f;
  for (int n = 0; n < N; ++n) {
    const T* r = qkv + (row0 + n) * ld;
    Q[n][lane] = ldf(r + h * 32 + lane);
    Kk[n][lane] = ldf(r + 128 + h * 32 + lane);
    V[n][lane] = ldf(r + 256 + h * 32 + lane);
    DO[n][lane] = ldf(dout + (row0 + n) * ldo + h * 32 + lane);
  }
  __syncwarp();
  // lane = key j (j < N): attn[i][j] for every query i; dattn[i][j] = sum_d dout[i][d] v[j][d]
  for (int i = 0; i < N; ++i) {
    float sim = -INFINITY, da = 0.f;
    if (lane < N) {
      sim = 0.f;
#pragma unroll 8
      for (int d = 0; d < 32; ++d) {
        sim = fmaf(Q[i][d] * scale, Kk[lane][d], sim);
        da = fmaf(DO[i][d], V[lane][d], da);
      }
    }
    const float mx = warp_max(sim);
    const float e = lane < N ? expf(sim - mx) : 0.f;
    const float p = e / warp_sum(e);
    const float dot = warp_sum(p * da);
    P[i][lane] = p;
    DS[i][lane] = p * (da - dot) * scale;        // d(loss)/d(q_i . k_j)
  }
  __syncwarp();
  // lane = channel d
  for (int n = 0; n < N; ++n) {
    float dq = 0.f, dk = 0.f, dv = 0.f;
    for (int j = 0; j < N; ++j) {
      dq = fmaf(DS[n][j], Kk[j][lane], dq);      // dq_n = sum_j dsim[n][j] k_j
      dk = fmaf(DS[j][n], Q[j][lane], dk);       // dk_n = sum_i dsim[i][n] q_i
      dv = fmaf(P[j][n], DO[j][lane], dv);       // dv_n = sum_i attn[i][n] dout_i
    }
    stf(dqkv + (row0 + n) * lddq + h * 32 + lane, dq);
    stf(dqkv + (row0 + n) * lddq + 128 + h * 32 + lane, dk);
    stf(dqkv + (row0 + n) * lddq + 256 + h * 32 + lane, dv);
  }
}
template <typename T>
void launch_softattn_bwd(const T* qkv, int ld, const T* dout, int ldo, T* dqkv, int lddq, int n_scenes, int N, cudaStream_t s) {
  if (n_scenes > 0) k_softattn_bwd<T><<<n_scenes * 4, 32, 0, s>>>(qkv, ld, dout, ldo, dqkv, lddq, n_scenes, N);
}

// ------------------------------------------------------------------------------------------------
// d(mean-over-batch loss) / d(model output): MSE terms + IoU regulariser (diffusion_ddpm.py:548-635, loss.py:7-102)
// one CTA (128 threads) per scene; writes dout [B*N, ld] in the activation dtype (padding columns zeroed)
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(128) k_p_losses_bwd(const float* __restrict__ x0, const float* __restrict__ noise,
                                                      const float* __restrict__ x_t, const T* __restrict__ out, int ld,
                                                      const int64_t* __restrict__ t, const float* __restrict__ sqrt_ac,
                                                      const float* __restrict__ sqrt_1mac,
                                                      const float* __restrict__ sqrt_recip_ac,
                                                      const float* __restrict__ sqrt_recipm1_ac,
                                                      const float* __restrict__ loss_weight,
                                                      const float* __restrict__ alphas_cumprod, LossArgs a,
                                                      T* __restrict__ dout, int ldd, int dpad, int B, float grad_scale) {
  const int b = blockIdx.x;
  if (b >= B) return;
  const int N = a.n_obj, d = a.d, tid = threadIdx.x;
  const int tb = int(t[b]);
  const float sa = sqrt_ac[tb], s1 = sqrt_1mac[tb], lw = loss_weight[tb];
  const int bb = a.trans + a.size + a.angle;
  __shared__ float xr[64][6];          // clamped reconstruction: trans(3), size(3)   (N <= 64)
  __shared__ float pass[64][6];        // 1 where the clamp passes the gradient
  __shared__ float valid[64];
  __shared__ float dcorn[64][6];       // d(loss) / d(lo[3], hi[3]) of every box
  __shared__ float s_nvalid;
  const float per_scene = grad_scale / float(B);      // loss = mean over the batch
  // ---- MSE part: slice means over (N, slice width), weights as in the reference's branches
  for (int i = tid; i < N * dpad; i += blockDim.x) {
    const int o = i / dpad, ch = i % dpad;
    float g = 0.f;
    if (ch < d) {
      const int64_t xi = ((int64_t)b * N + o) * d + ch;
      float target;
      if (a.mean_type == DS_MEAN_EPS) target = noise[xi];
      else if (a.mean_type == DS_MEAN_X0) target = x0[xi];
      else target = sa * noise[xi] - s1 * x0[xi];
      const float diff = ldf(out + ((int64_t)b * N + o) * ld + ch) - target;
      float wsl;      // 1 / (elements of the mean this channel belongs to), 0 if its term is not in the loss
      if (!a.loss_separate) wsl = 1.0f / float(N * d);
      else if (a.arrange) wsl = 1.0f / float(N * (ch < a.trans ? a.trans : d - a.trans));
      else if (ch < bb) wsl = 1.0f / float(N * bb);
      else if (ch < bb + a.cls) wsl = 1.0f / float(N * a.cls);
      else if (ch < bb + a.cls + a.objn) wsl = 1.0f / float(N * a.objn);
      else wsl = 1.0f / float(N * a.feat);
      g = 2.0f * diff * wsl * lw * per_scene;
    }
    stf(dout + ((int64_t)b * N + o) * ldd + ch, g);
  }
  if (!a.loss_iou) return;
  __syncthreads();
  // ---- IoU regulariser on the clamped x0 estimate
  float ax, ao;
  if (a.mean_type == DS_MEAN_V) { ax = sa; ao = -s1; }
  else if (a.mean_type == DS_MEAN_EPS) { ax = sqrt_recip_ac[tb]; ao = -sqrt_recipm1_ac[tb]; }
  else { ax = 0.f; ao = 1.f; }
  for (int i = tid; i < N * 6; i += blockDim.x) {
    const int o = i / 6, k = i % 6;
    const int ch = k < 3 ? k : a.trans + (k - 3);
    const int64_t xi = ((int64_t)b * N + o) * d + ch;
    const float raw = ax * x_t[xi] + ao * ldf(out + ((int64_t)b * N + o) * ld + ch);
    xr[o][k] = fminf(fmaxf(raw, -1.0f), 1.0f);
    pass[o][k] = (raw >= -1.0f && raw <= 1.0f) ? 1.0f : 0.f;
  }
  for (int o = tid; o < N; o += blockDim.x) {
    const int vch = a.objn > 0 ? bb + a.cls : bb + a.cls - 1;
    const int64_t xi = ((int64_t)b * N + o) * d + vch;
    const float raw = ax * x_t[xi] + ao * ldf(out + ((int64_t)b * N + o) * ld + vch);
    const float cl = fminf(fmaxf(raw, -1.0f), 1.0f);
    valid[o] = a.objn > 0 ? (cl >= 0.f ? 1.f : 0.f) : (cl <= 0.f ? 1.f : 0.f);
    for (int k = 0; k < 6; ++k) dcorn[o][k] = 0.f;
  }
  __syncthreads();
  if (tid == 0) {
    float nv = 0.f;
    for (int o = 0; o < N; ++o) nv += valid[o];
    s_nvalid = nv;
  }
  __syncthreads();
  const float denom = s_nvalid * s_nvalid + 1e-6f;
  const float wpair = alphas_cumprod[tb] * 0.1f / denom * per_scene;      // d(loss) / d(IoU_ij) for valid pairs
  auto corner = [&](int o, int k, bool hi) {      // world-space box corner k of object o
    const float tr = (xr[o][k] + 1.0f) * 0.5f * (a.bounds[3 + k] - a.bounds[k]) + a.bounds[k];
    const float sz = (xr[o][3 + k] + 1.0f) * 0.5f * (a.bounds[9 + k] - a.bounds[6 + k]) + a.bounds[6 + k];
    return hi ? tr + sz : tr - sz;
  };
  for (int pidx = tid; pidx < N * N; pidx += blockDim.x) {
    const int i = pidx / N, j = pidx % N;
    if (valid[i] == 0.f || valid[j] == 0.f) continue;
    float lo_i[3], hi_i[3], lo_j[3], hi_j[3], wh[3], raww[3];
    float area_i = 1.f, area_j = 1.f, ov = 1.f;
    for (int k = 0; k < 3; ++k) {
      lo_i[k] = corner(i, k, false); hi_i[k] = corner(i, k, true);
      lo_j[k] = corner(j, k, false); hi_j[k] = corner(j, k, true);
      area_i *= hi_i[k] - lo_i[k];
      area_j *= hi_j[k] - lo_j[k];
      raww[k] = fminf(hi_i[k], hi_j[k]) - fmaxf(lo_i[k], lo_j[k]);
      wh[k] = fmaxf(raww[k], 0.f);
      ov *= wh[k];
    }
    const float un_raw = area_i + area_j - ov;
    const float un = fmaxf(un_raw, 1e-6f);
    // IoU = ov / un ; d/d(ov) = 1/un + (un passes ? ov / un^2 : 0) ; d/d(area) = -(passes) ov / un^2
    const float passes = un_raw > 1e-6f ? 1.f : (un_raw == 1e-6f ? 0.5f : 0.f);
    const float d_ov = wpair * (1.0f / un + passes * ov / (un * un));
    const float d_area = -wpair * passes * ov / (un * un);
    for (int k = 0; k < 3; ++k) {
      // areas
      float prod_i = 1.f, prod_j = 1.f;
      for (int m = 0; m < 3; ++m) if (m != k) { prod_i *= hi_i[m] - lo_i[m]; prod_j *= hi_j[m] - lo_j[m]; }
      atomicAdd(&dcorn[i][3 + k], d_area * prod_i);
      atomicAdd(&dcorn[i][k], -d_area * prod_i);
      atomicAdd(&dcorn[j][3 + k], d_area * prod_j);
      atomicAdd(&dcorn[j][k], -d_area * prod_j);
      // overlap: clamp(min = 0) passes the gradient where rb - lt >= 0 (torch: min <= x)
      if (raww[k] >= 0.f) {
        float other = 1.f;
        for (int m = 0; m < 3; ++m) if (m != k) other *= wh[m];
        const float gwh = d_ov * other;
        // rb = min(hi_i, hi_j): ties split evenly (torch.minimum); lt = max(lo_i, lo_j) likewise
        const float wi_hi = hi_i[k] < hi_j[k] ? 1.f : (hi_i[k] == hi_j[k] ? 0.5f : 0.f);
        const float wi_lo = lo_i[k] > lo_j[k] ? 1.f : (lo_i[k] == lo_j[k] ? 0.5f : 0.f);
        atomicAdd(&dcorn[i][3 + k], gwh * wi_hi);
        atomicAdd(&dcorn[j][3 + k], gwh * (1.f - wi_hi));
        atomicAdd(&dcorn[i][k], -gwh * wi_lo);
        atomicAdd(&dcorn[j][k], -gwh * (1.f - wi_lo));
      }
    }
  }
  __syncthreads();
  // corners -> (trans, size) -> clamp -> model output
  for (int i = tid; i < N * 6; i += blockDim.x) {
    const int o = i / 6, k = i % 6;
    float g;
    if (k < 3) g = (dcorn[o][k] + dcorn[o][3 + k]) * 0.5f * (a.bounds[3 + k] - a.bounds[k]);                 // d/d trans
    else g = (dcorn[o][k] - dcorn[o][k - 3]) * 0.5f * (a.bounds[9 + (k - 3)] - a.bounds[6 + (k - 3)]);       // d/d size: hi - lo
    g *= pass[o][k] * ao;
    const int ch = k < 3 ? k : a.trans + (k - 3);
    T* p = dout + ((int64_t)b * N + o) * ldd + ch;
    stf(p, ldf(p) + g);
  }
}
template <typename T>
void launch_p_losses_bwd(const float* x0, const float* noise, const float* x_t, const T* out, int ld, const int64_t* t,
                         const float* sqrt_ac, const float* sqrt_1mac, const float* sqrt_recip_ac,
                         const float* sqrt_recipm1_ac, const float* loss_weight, const float* alphas_cumprod, LossArgs a,
                         T* dout, int ldd, int dpad, int B, float grad_scale, cudaStream_t s) {
  if (B > 0)
    k_p_losses_bwd<T><<<B, 128, 0, s>>>(x0, noise, x_t, out, ld, t, sqrt_ac, sqrt_1mac, sqrt_recip_ac, sqrt_recipm1_ac,
                                        loss_weight, alphas_cumprod, a, dout, ldd, dpad, B, grad_scale);
}

// ------------------------------------------------------------------------------------------------
// weights: flat fp32 parameter buffer <-> packed matrices
// ------------------------------------------------------------------------------------------------
// one warp per row of a piece: dst[row_off + r][col_off + c] = (ws ? standardised : plain) src[r][c]
template <typename T>
__global__ void k_pack_piece(const float* __restrict__ src, int rows, int cols, T* __restrict__ dst, int ldd, int ws,
                             T* __restrict__ dstT, int ldt) {
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float* sr = src + (int64_t)r * cols;
  float fm = 0.f, rs = 1.f;
  if (ws) {      // fp32 like the reference (denoise_net.py:86-89): biased variance, eps 1e-5; sums in double
    double m = 0;
    for (int c = lane; c < cols; c += 32) m += sr[c];
    for (int o = 16; o > 0; o >>= 1) m += __shfl_xor_sync(0xffffffffu, m, o);
    m /= cols;
    double v = 0;
    for (int c = lane; c < cols; c += 32) v += (sr[c] - m) * (sr[c] - m);
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    v /= cols;
    fm = float(m);
    rs = 1.0f / sqrtf(float(v) + 1e-5f);
  }
  for (int c = lane; c < cols; c += 32) {
    const float v = ws ? (sr[c] - fm) * rs : sr[c];
    stf(dst + (int64_t)r * ldd + c, v);
    if (dstT) stf(dstT + (int64_t)c * ldt + r, v);      // transposed copy [K, N]: the K-major operand of dX = dY W
  }
}
template <typename T>
void launch_pack_piece(const float* src, int rows, int cols, T* dst, int ldd, int ws, T* dstT, int ldt, cudaStream_t s) {
  if (rows > 0) k_pack_piece<T><<<cdiv64(rows, 8), 256, 0, s>>>(src, rows, cols, dst, ldd, ws, dstT, ldt);
}
// out[c][m] = in[m][c] for m < M, 0 for M <= m < Mcap  (token-major activations -> the K-major operands of dW = dY^T X)
// colsum (optional): colsum[c] += sum_m in[m][c] -- the bias gradient, for free while the tile is in shared memory
template <typename T>
__global__ void k_transpose_pad(const T* __restrict__ in, int ld, T* __restrict__ out, int ldo, int M, int Mcap, int C,
                                float* __restrict__ colsum) {
  __shared__ float tile[32][33];
  __shared__ float part[8][33];
  const int m0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  float cs = 0.f;
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int m = m0 + i, c = c0 + threadIdx.x;
    const float v = (m < M && c < C) ? ldf(in + (int64_t)m * ld + c) : 0.f;
    tile[i][threadIdx.x] = v;
    cs += v;
  }
  if (colsum) part[threadIdx.y][threadIdx.x] = cs;
  __syncthreads();
  if (colsum && threadIdx.y == 0 && c0 + threadIdx.x < C && m0 < M) {
    float tsum = 0.f;
#pragma unroll
    for (int y = 0; y < 8; ++y) tsum += part[y][threadIdx.x];
    atomicAdd(colsum + c0 + threadIdx.x, tsum);
  }
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int c = c0 + i, m = m0 + threadIdx.x;
    if (c < C && m < Mcap) stf(out + (int64_t)c * ldo + m, tile[threadIdx.x][i]);
  }
}
template <typename T>
void launch_transpose_pad(const T* in, int ld, T* out, int ldo, int M, int Mcap, int C, float* colsum, cudaStream_t s) {
  dim3 grid((Mcap + 31) / 32, (C + 31) / 32), block(32, 8);
  k_transpose_pad<T><<<grid, block, 0, s>>>(in, ld, out, ldo, M, Mcap, C, colsum);
}
// gradient of a piece: dsrc[r][c] = (ws adjoint of) dpacked[row_off + r][col_off + c]
__global__ void k_unpack_piece_grad(const float* __restrict__ dpacked, int ldp, const float* __restrict__ w, int rows,
                                    int cols, float* __restrict__ dw, int ws) {
  const int r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  if (r >= rows) return;
  const float* g = dpacked + (int64_t)r * ldp;
  float* o = dw + (int64_t)r * cols;
  if (!ws) {
    for (int c = lane; c < cols; c += 32) o[c] = g[c];
    return;
  }
  const float* wr = w + (int64_t)r * cols;
  double m = 0;
  for (int c = lane; c < cols; c += 32) m += wr[c];
  for (int of = 16; of > 0; of >>= 1) m += __shfl_xor_sync(0xffffffffu, m, of);
  m /= cols;
  double v = 0;
  for (int c = lane; c < cols; c += 32) v += (wr[c] - m) * (wr[c] - m);
  for (int of = 16; of > 0; of >>= 1) v += __shfl_xor_sync(0xffffffffu, v, of);
  v /= cols;
  const float fm = float(m), rs = 1.0f / sqrtf(float(v) + 1e-5f);
  float g1 = 0.f, g2 = 0.f;
  for (int c = lane; c < cols; c += 32) {
    const float wh = (wr[c] - fm) * rs;
    g1 += g[c];
    g2 = fmaf(g[c], wh, g2);
  }
  g1 = warp_sum(g1) / float(cols);
  g2 = warp_sum(g2) / float(cols);
  for (int c = lane; c < cols; c += 32) {
    const float wh = (wr[c] - fm) * rs;
    o[c] = rs * (g[c] - g1 - wh * g2);
  }
}
void launch_unpack_piece_grad(const float* dpacked, int ldp, const float* w, int rows, int cols, float* dw, int ws,
                              cudaStream_t s) {
  if (rows > 0) k_unpack_piece_grad<<<cdiv64(rows, 8), 256, 0, s>>>(dpacked, ldp, w, rows, cols, dw, ws);
}

// ------------------------------------------------------------------------------------------------
// optimizer: global gradient norm + Adam (torch.optim.Adam semantics, weight decay 0; clip_grad_norm_ folded in)
// ------------------------------------------------------------------------------------------------
__global__ void k_sumsq(const float* __restrict__ g, int64_t n, float* __restrict__ out) {
  float s = 0.f;
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) s = fmaf(g[i], g[i], s);
  s = warp_sum(s);
  __shared__ float sh[8];
  if ((threadIdx.x & 31) == 0) sh[threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float tsum = 0.f;
    for (int i = 0; i < (blockDim.x >> 5); ++i) tsum += sh[i];
    atomicAdd(out, tsum);
  }
}
void launch_sumsq(const float* g, int64_t n, float* out, cudaStream_t s) {
  if (n > 0) k_sumsq<<<592, 256, 0, s>>>(g, n, out);
}
// sumsq_in: optional device scalar = squared L2 norm of ALL gradients (this buffer's and the caller's other
// parameters'); the clip coefficient max_norm / (norm + 1e-6), capped at 1, multiplies the gradient in registers
__global__ void k_adam(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                       int64_t n, float lr, float b1, float b2, float eps, float bc1, float bc2_sqrt,
                       const float* __restrict__ sumsq_in, float max_norm) {
  float clip = 1.0f;
  if (sumsq_in && max_norm > 0.f) clip = fminf(1.0f, max_norm / (sqrtf(*sumsq_in) + 1e-6f));
  for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) {
    const float gi = g[i] * clip;
    const float mi = b1 * m[i] + (1.0f - b1) * gi;
    const float vi = b2 * v[i] + (1.0f - b2) * gi * gi;
    m[i] = mi;
    v[i] = vi;
    // torch: denom = sqrt(v) / sqrt(bias_correction2) + eps ; p -= (lr / bias_correction1) * m / denom
    p[i] -= (lr / bc1) * mi / (sqrtf(vi) / bc2_sqrt + eps);
  }
}
void launch_adam(float* p, const float* g, float* m, float* v, int64_t n, float lr, float b1, float b2, float eps,
                 int step, const float* sumsq_in, float max_norm, cudaStream_t s) {
  if (n <= 0) return;
  const float bc1 = 1.0f - powf(b1, float(step)), bc2 = 1.0f - powf(b2, float(step));
  k_adam<<<1184, 256, 0, s>>>(p, g, m, v, n, lr, b1, b2, eps, bc1, sqrtf(bc2), sumsq_in, max_norm);
}

// ---- explicit instantiations ----
#define INSTB(T)                                                                                                      \
  template void launch_colsum<T>(const T*, int, float*, int, int, cudaStream_t);                                      \
  template void launch_add_block<T>(const T*, int, T*, int, int, int, int, cudaStream_t);                             \
  template void launch_act<T>(const T*, int, T*, int, int, int, int, cudaStream_t);                                   \
  template void launch_act_bwd<T>(const T*, int, const T*, int, T*, int, int, int, int, cudaStream_t);                \
  template void launch_gn_bwd<T>(const T*, int, const T*, int, T*, int, T*, int, int, const float*, const float*,     \
                                 FilmRef, float*, float*, float*, int64_t, int, int, int, int, cudaStream_t);         \
  template bool launch_gn_fwd_reg<T>(const T*, int, T*, int, const float*, const float*, FilmRef, const T*, int, int, int,   \
                                     int, int, cudaStream_t);                                                         \
  template void launch_ln_bwd<T>(const T*, int, const T*, int, T*, int, int, T*, int, int, const float*, float*, int, \
                                 int, cudaStream_t);                                                                  \
  template void launch_linattn_bwd<T>(const T*, int, const T*, int, T*, int, int, int, cudaStream_t);                 \
  template void launch_softattn_bwd<T>(const T*, int, const T*, int, T*, int, int, int, cudaStream_t);                \
  template void launch_xattn_bwd<T>(const T*, int, const T*, int, const T*, int, T*, int, int, T*, int, int, int, int, \
                                    cudaStream_t);                                                                    \
  template void launch_p_losses_bwd<T>(const float*, const float*, const float*, const T*, int, const int64_t*,       \
                                       const float*, const float*, const float*, const float*, const float*,          \
                                       const float*, LossArgs, T*, int, int, int, float, cudaStream_t);               \
  template void launch_pack_piece<T>(const float*, int, int, T*, int, int, T*, int, cudaStream_t);                    \
  template void launch_transpose_pad<T>(const T*, int, T*, int, int, int, int, float*, cudaStream_t);                 \
  template void launch_gemm_nn<T, T, T>(const T*, int, const T*, int, T*, int, int, int, int, int, cudaStream_t);     \
  template void launch_gemm_tn<T, T>(const T*, int, const T*, int, float*, int, int, int, int, cudaStream_t);
INSTB(float)
INSTB(bf16)
template void launch_gemm_nn<float, float, bf16>(const float*, int, const float*, int, bf16*, int, int, int, int, int, cudaStream_t);

}  // namespace ds
