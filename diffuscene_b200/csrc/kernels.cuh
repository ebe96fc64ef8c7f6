// Host-side launchers of every kernel in the library (definitions in pointwise.cu, gemm_simt.cu,
// gemm_tc.cu).  All pointers are device pointers; `ld*` are row pitches in elements.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "common.cuh"

namespace ds {

// FiLM (scale, shift) source for the GroupNorm op.  Row `r` of the activation matrix belongs to scene
// r / n_obj and object r % n_obj.  The table row holds [scale(C) | shift(C)] (chunk(2, dim=1),
// reference denoise_net.py:200).
enum FilmMode { FILM_NONE = 0, FILM_TIME = 1, FILM_OBJECT = 2, FILM_TOKEN = 3 };
struct FilmRef {
  const float* base;      // already offset to this block's [2C] slice
  int mode;
  int64_t row_stride;     // floats between consecutive table rows
  const int* t;           // FILM_TIME: per-scene timestep index (device)
};

template <typename T>
void launch_pack_input(const float* x, T* out, int ld_out, int M, int d, cudaStream_t s);
template <typename T>
void launch_unpack_output(const T* in, int ld_in, float* out, int M, int d, cudaStream_t s);
template <typename T>
void launch_groupnorm(const T* in, int ld_in, T* out, int ld_out, const float* gamma, const float* beta,
                      FilmRef film, const T* res, int ld_res, int n_scenes, int n_obj, int C, int groups,
                      cudaStream_t s);
template <typename T>
void launch_layernorm(const T* in, int ld_in, T* out, int ld_out, const float* g, const T* res, int ld_res,
                      int M, int C, cudaStream_t s);
template <typename T>
void launch_linattn(const T* qkv, int ld, T* out, int ld_out, int n_scenes, int n_obj, cudaStream_t s);
template <typename T>
void launch_softattn(const T* qkv, int ld, T* out, int ld_out, int n_scenes, int n_obj, cudaStream_t s);
// cross linear attention: ctx [n_scenes][4][32(d)][32(e)] fp32 precomputed from the text
template <typename T>
void launch_xattn_apply(const T* q, int ldq, const float* ctx, T* out, int ld_out, int n_scenes, int n_obj,
                        cudaStream_t s);
// kv: [n_scenes * L, ld_kv] rows of k | v (128 columns each) in storage type T; any 1 <= L <= 512
template <typename T>
void launch_xattn_prepare(const T* kv, int ld_kv, float* ctx, int n_scenes, int L, cudaStream_t s);

void sinusoid_freqs_host(int dim, float* hf /*[dim / 2]*/);
void launch_sinusoid(float* out, const float* freq_dev, int T, int dim, cudaStream_t s);
void launch_sinusoid_t(float* out, const float* freq_dev, const int* t_dev, int B, int dim, cudaStream_t s);
void launch_silu_f32(const float* in, float* out, int64_t n, cudaStream_t s);
void launch_t_convert(const int64_t* t, int* out, int B, cudaStream_t s);

// ---- sampling-step kernels --------------------------------------------------------------------
// Per-step coefficients, one row per loop iteration (device table).
struct StepCoef {
  float a_x, a_o;         // x0 = a_x * x_t + a_o * model_out
  float c_0, c_x, c_z;    // x_next = c_0 * x0 + c_x * x_t + c_z * noise
  float q_a, q_b;         // completion re-noising: x[:P] = q_a * partial + q_b * noise2
  int   t;                // timestep fed to the denoiser
};
struct StepState {        // device-resident loop state (advanced by the kernels themselves), one per handle
  int step;               // loop iteration index (0 .. n_steps-1)
  unsigned int done;      // blocks of the running step_update kernel that have finished (last one advances `step`)
  // Philox key / global index of scene 0 of this call: read from HERE by the step kernels (not passed as kernel
  // parameters), so that a captured step graph is reusable across calls with different seeds / shards
  unsigned long long seed;
  unsigned long long scene_offset;
};
// start of a step: t_dev[b] = coef[step].t ; optional completion re-noise of the first P objects
void launch_begin_step(const StepCoef* coef, const StepState* st, int* t_dev, float* x, const float* partial,
                       const float* partial_noise, int B, int n_obj, int d, int P, cudaStream_t s);
// end of a step: x <- update(x, model_out, noise) ; advances st->step
template <typename T>
void launch_step_update(const StepCoef* coef, StepState* st, float* x, const T* model_out, int ld_out,
                        const float* noise, int B, int n_obj, int d, int clip, cudaStream_t s);
void launch_randn(float* out, int B, int per_scene, uint64_t seed, uint64_t scene_offset, uint32_t stream_id,
                  cudaStream_t s);
// single explicit reverse step with per-sample t (p_sample)
template <typename T>
void launch_p_sample(const float* x, const T* model_out, int ld_out, const int* t, const float* noise, float* out,
                     const float* a_x, const float* a_o, const float* c1, const float* c2, const float* sigma,
                     int B, int n_obj, int d, int clip, cudaStream_t s);
void launch_q_sample(const float* x0, const int64_t* t, const float* noise, float* out, const float* sqrt_ac,
                     const float* sqrt_1mac, int B, int per_scene, cudaStream_t s);

// p_losses value (reference diffusion_ddpm.py:520-652): one CTA per scene
struct LossArgs {
  int n_obj, d, trans, size, angle, cls, objn, feat;
  int mean_type, loss_separate, loss_iou, arrange;
  float bounds[12];     // trans_min[3], trans_max[3], size_min[3], size_max[3]
};
template <typename T>
void launch_p_losses(const float* x0, const float* noise, const float* x_t, const T* model_out, int ld_out,
                     const int64_t* t, const float* sqrt_ac, const float* sqrt_1mac, const float* sqrt_recip_ac,
                     const float* sqrt_recipm1_ac, const float* loss_weight, const float* alphas_cumprod,
                     LossArgs a, float* losses, float* parts /*[B][9]*/, int B, cudaStream_t s);
void launch_loss_dict_mean(const float* parts, float* dict9, int B, cudaStream_t s);

// nearest catalogue model per query object (threed_future_dataset.py:28-77); see k_retrieve
void launch_retrieve(const int* class_start, int n_classes, const float* cat_feat, const float* cat_size, int feat_dim,
                     int size_dim, const int64_t* q_label, const float* q_feat, const float* q_size, int Q, int mode,
                     int64_t* out, cudaStream_t s);

// ---- GEMMs: D[M,N] = act([A0 | A1][M, K0+K1] * W[N, K0+K1]^T + bias) (+ residual) -----------------
struct GemmArgs {
  const void* a0; int lda0; int k0;
  const void* a1; int lda1; int k1;      // a1 == nullptr when there is no second operand
  const void* w;  int ldw;               // [N, K] row-major, same element type as A
  const float* bias;                     // [N] or nullptr
  void* d; int ldd;
  const void* res; int ldres;            // optional residual added after the activation
  int M, N, act;
  // fused GroupNorm(8 groups) + affine + FiLM + SiLU epilogue (tcgen05 backend only)
  int gn;
  int n_obj;
  int film_C;
  const float* gamma;
  const float* beta;
  FilmRef film;
  // tcgen05 backend: never use the CTA-pair instantiation for this GEMM.  Set by the training step: its GEMMs measured
  // 4.5 % slower per iteration as pairs (26.8 k vs 28.0 k scenes/s, profiles/round2_final_bench_train_*), unlike the
  // sampling path's large plain GEMMs
  int no_pair;
};
template <typename T> void launch_gemm_simt(const GemmArgs& g, bool exact, cudaStream_t s);
// fp32 A/W in, fp32 out (time / context FiLM tables; always fp32)
void launch_gemm_f32(const GemmArgs& g, cudaStream_t s);

// tcgen05 path: operands described by TMA tensor maps built by the engine (gemm_tc.cu)
struct TcGemmPlan;   // opaque, owns tensor maps
TcGemmPlan* tc_plan_create(const GemmArgs& g, int rows_capacity, char* err, int err_len);
void tc_plan_destroy(TcGemmPlan* p);
void tc_plan_set_film(TcGemmPlan* p, const FilmRef& f);
void tc_plan_set_trace(TcGemmPlan* p, unsigned long long* trace);
// Programmatic-dependent-launch policy shared by every launcher of the library (pointwise.cu): on when `rows` (tokens
// of the launch) <= 32768.  Measured on B200 (profiles/round2_probe_pdl.txt, round2_probe_epi.txt), bedroom N = 12:
// 1 / 128 / 512 / 1024 / 2048 scenes per GPU gain 8 / 7.5 / 8 / 6 / 3 % (the ~5 us kernel prologue is a large share of
// each launch), 4096 scenes lose 1.4 % (the chip runs at its power cap there and the early-resident CTAs cost clock).
bool pdl_enabled(int64_t rows);
void tc_plan_set_atomic_out(TcGemmPlan* p, float* d32, int ldd, int ksplit);      // split-K, fp32 atomics (dW GEMMs)
int tc_plan_tiles(const TcGemmPlan* p, int M);
void tc_plan_set_residual(TcGemmPlan* p, const void* res);      // nullptr: plain store; == output: accumulate in place
void tc_plan_set_uniform_t(TcGemmPlan* p, int uniform);   // all scenes share one timestep (sampling loop)   // [grid][8] cycle counters   // FiLM tables may be (re)allocated after planning
int launch_gemm_tc(const TcGemmPlan* p, int M, cudaStream_t s);   // returns 0 or cudaError
bool tc_runtime_available(char* err, int err_len);
// GemmArgs.gn == 2 selects the channels-on-lanes GroupNorm GEMM: weight rows must be stored permuted inside every
// block of 32 output channels (stored row 32 b + l holds channel 32 b + 8 (l % 4) + l / 4)
bool tc_gnt_supported(int n_obj, int N);
// GemmArgs.gn == 3: the same kernel as a plain GEMM (bias, activation, residual); same weight row order
bool tc_gnt_plain_supported(int n_obj, int N);
// fused GEMM + channel LayerNorm (+ residual) for K <= 128, N = 512 (gemm_ln.cu): GemmArgs.gamma = LayerNorm gain
struct LnGemmPlan;
bool ln_gemm_supported(int N, int K);
LnGemmPlan* ln_plan_create(const GemmArgs& g, int rows_capacity, char* err, int err_len);
void ln_plan_destroy(LnGemmPlan* p);
int launch_gemm_ln(const LnGemmPlan* p, int M, cudaStream_t s);
// fused channel LayerNorm + to_qkv + linear-attention core (gemm_attn.cu)
struct AttnQkvPlan;
bool attn_qkv_supported(int n_obj, int C);
AttnQkvPlan* attn_qkv_plan_create(const void* x, int ldx, const void* w, int ldw, const float* cs, void* o, int ldo,
                                  int n_obj, int K, int rows_capacity, char* err, int err_len);
void attn_qkv_plan_destroy(AttnQkvPlan* p);
int launch_ln_qkv_attn(const AttnQkvPlan* p, int M, cudaStream_t s);
inline int tc_gnt_row(int stored_row) { const int l = stored_row & 31; return (stored_row & ~31) + 8 * (l & 3) + (l >> 2); }

}  // namespace ds
