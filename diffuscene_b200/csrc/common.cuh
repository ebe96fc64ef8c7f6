// Shared device helpers for the diffuscene_b200 kernels (sm_100a only).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace ds {

typedef __nv_bfloat16 bf16;

// ---- storage-type traits: activations are float (parity mode) or bf16 (throughput mode) ----
template <typename T> struct ST;
template <> struct ST<float> {
  static __device__ __forceinline__ float ld(const float* p) { return *p; }
  static __device__ __forceinline__ void st(float* p, float v) { *p = v; }
};
template <> struct ST<bf16> {
  static __device__ __forceinline__ float ld(const bf16* p) { return __bfloat162float(*p); }
  static __device__ __forceinline__ void st(bf16* p, float v) { *p = __float2bfloat16_rn(v); }
};

template <typename T> __device__ __forceinline__ float ldf(const T* p) { return ST<T>::ld(p); }
template <typename T> __device__ __forceinline__ void stf(T* p, float v) { ST<T>::st(p, v); }

// ---- activations (exact forms: parity mode must match torch's erf-GELU / SiLU) ----
enum Act { ACT_NONE = 0, ACT_GELU = 1, ACT_SILU = 2 };

__device__ __forceinline__ float gelu_erf(float x) { return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f)); }
__device__ __forceinline__ float silu(float x) { return x / (1.0f + __expf(-x)); }
__device__ __forceinline__ float silu_exact(float x) { return x / (1.0f + expf(-x)); }
template <bool EXACT> __device__ __forceinline__ float apply_act(float x, int act) {
  if (act == ACT_GELU) return gelu_erf(x);
  if (act == ACT_SILU) return EXACT ? silu_exact(x) : silu(x);
  return x;
}

// ---- warp reductions ----
__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

// ---- cross linear attention, text side (LinearAttentionCross, denoise_net.py:261-297) ----
// kv rows of one scene: [L][ld], k of head h at columns h*32 .. h*32+31, v at 128 + h*32 ..; one warp per head.
// The L text tokens are streamed through two [XATTN_CHUNK][33] shared tiles per warp, so shared memory does not grow
// with L (k_xattn_prepare, k_xattn_bwd).
constexpr int XATTN_CHUNK = 32;
// softmax over L of k channel d = lane: max and 1 / sum(exp(k - max)), summed in token order
template <typename T>
__device__ __forceinline__ void xattn_k_stats(const T* kv, int ld, int L, int h, int lane, float& kmax, float& kinv) {
  float m = -INFINITY;
  for (int l = 0; l < L; ++l) m = fmaxf(m, ldf(kv + (int64_t)l * ld + h * 32 + lane));
  float s = 0.f;
  for (int l = 0; l < L; ++l) s += expf(ldf(kv + (int64_t)l * ld + h * 32 + lane) - m);
  kmax = m;
  kinv = 1.0f / s;
}
// ctx[d][e] = sum_l softmax_L(k)[l][d] v[l][e].  LANE_D: lane = d, acc[e] = ctx[d][e]; otherwise lane = e, acc[d]
template <typename T, bool LANE_D>
__device__ __forceinline__ void xattn_context(const T* kv, int ld, int L, int h, int lane, float kmax, float kinv,
                                              float (*Ks)[33], float (*Vs)[33], float* acc) {
#pragma unroll
  for (int i = 0; i < 32; ++i) acc[i] = 0.f;
  for (int l0 = 0; l0 < L; l0 += XATTN_CHUNK) {
    const int n = min(XATTN_CHUNK, L - l0);
    for (int l = 0; l < n; ++l) {
      const T* p = kv + (int64_t)(l0 + l) * ld + h * 32 + lane;
      Ks[l][lane] = expf(ldf(p) - kmax) * kinv;
      Vs[l][lane] = ldf(p + 128);
    }
    __syncwarp();
    for (int l = 0; l < n; ++l) {
      const float mine = LANE_D ? Ks[l][lane] : Vs[l][lane];
#pragma unroll
      for (int i = 0; i < 32; ++i) acc[i] = fmaf(LANE_D ? Vs[l][i] : Ks[l][i], mine, acc[i]);
    }
    __syncwarp();
  }
}

// ---- Philox4x32-10 counter-based RNG (Salmon et al. 2011), one call -> 4 x u32 ----
__device__ __forceinline__ uint4 philox4x32_10(uint4 ctr, uint2 key) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint32_t hi0 = __umulhi(M0, ctr.x), lo0 = M0 * ctr.x;
    uint32_t hi1 = __umulhi(M1, ctr.z), lo1 = M1 * ctr.z;
    ctr = make_uint4(hi1 ^ ctr.y ^ key.x, lo1, hi0 ^ ctr.w ^ key.y, lo0);
    key.x += W0;
    key.y += W1;
  }
  return ctr;
}
// two N(0,1) draws from two u32 (Box-Muller)
__device__ __forceinline__ float2 box_muller(uint32_t a, uint32_t b) {
  float u1 = (float(a) + 0.5f) * 2.3283064365386963e-10f;   // (0,1)
  float u2 = (float(b) + 0.5f) * 2.3283064365386963e-10f;
  float r = sqrtf(-2.0f * logf(u1));
  float s, c;
  sincospif(2.0f * u2, &s, &c);
  return make_float2(r * c, r * s);
}

}  // namespace ds
