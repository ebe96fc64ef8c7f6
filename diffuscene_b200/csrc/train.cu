// Native training step: forward with every intermediate kept, the p_losses value, and the hand-written backward pass
// down to gradients of every named parameter (reference: what `loss.backward()` does behind
// DiffusionSceneLayout_DDPM.get_loss / train_on_batch, scene_synthesis/networks/diffusion_scene_layout_ddpm.py:131-226,
// 456-473, through GaussianDiffusion.p_losses, diffusion_ddpm.py:520-652, and Unet1D.forward, denoise_net.py:507-593).
//
// Parameters and gradients travel as ONE flat fp32 device buffer each, laid out in ds_expected_weight() order, so that
// the optimizer (ds_adam_step) and the data-parallel all-reduce work on contiguous memory and nothing is repacked on
// the host.  The training step program is the plan of plan.cpp in train mode (one op per reference layer); its
// adjoint is executed op by op in reverse (kernels: backward.cu).  The time-embedding MLP and the 19 + 9 FiLM
// projections run per sample here (fp32), not from the hoisted tables of the sampling path: their weights are trained.
// Likewise the text side of the cross-attention layers (to_kv projection, softmax over the tokens, k^T v context) is
// computed every step from the flat parameters and differentiated down to d(to_kv.weight) and d(context_cross).
#include "engine_internal.h"

namespace ds {
// backward.cu
template <typename TA, typename TB, typename TD>
void launch_gemm_nn(const TA* A, int lda, const TB* B, int ldb, TD* D, int ldd, int M, int N, int K, int accumulate, cudaStream_t s);
template <typename TA, typename TB>
void launch_gemm_tn(const TA* A, int lda, const TB* B, int ldb, float* D, int ldd, int M, int Ka, int Kb, cudaStream_t s);
template <typename T> void launch_colsum(const T* A, int lda, float* out, int M, int N, cudaStream_t s);
template <typename T> void launch_add_block(const T* src, int lds, T* dst, int ldd, int M, int N, int accumulate, cudaStream_t s);
template <typename T> void launch_act(const T* z, int ldz, T* out, int ldo, int M, int N, int act, cudaStream_t s);
template <typename T> void launch_act_bwd(const T* z, int ldz, const T* dy, int ldy, T* dz, int lddz, int M, int N, int act, cudaStream_t s);
template <typename T>
void launch_gn_bwd(const T* c, int ldc, const T* dy, int ldy, T* dc, int lddc, T* dres, int ldr, int res_accumulate,
                   const float* gamma, const float* beta, FilmRef film, float* dgamma, float* dbeta, float* dfilm,
                   int64_t dfilm_row_stride, int n_scenes, int n_obj, int C, int groups, cudaStream_t s);
template <typename T>
bool launch_gn_fwd_reg(const T* in, int ld_in, T* out, int ld_out, const float* gamma, const float* beta, FilmRef film,
                       const T* res, int ld_res, int n_scenes, int n_obj, int C, int groups, cudaStream_t s);
template <typename T>
void launch_ln_bwd(const T* x, int ldx, const T* dy, int ldy, T* dx, int lddx, int dx_accumulate, T* dres, int ldr,
                   int res_accumulate, const float* g, float* dg, int M, int C, cudaStream_t s);
template <typename T> void launch_linattn_bwd(const T* qkv, int ld, const T* dout, int ldo, T* dqkv, int lddq, int n_scenes, int N, cudaStream_t s);
template <typename T> void launch_softattn_bwd(const T* qkv, int ld, const T* dout, int ldo, T* dqkv, int lddq, int n_scenes, int N, cudaStream_t s);
template <typename T>
void launch_xattn_bwd(const T* q, int ldq, const T* dout, int ldo, const T* kv, int ld_kv, T* dq, int lddq, int dq_accumulate,
                      T* dkv, int ld_dkv, int n_scenes, int n_obj, int L, cudaStream_t s);
template <typename T>
void launch_p_losses_bwd(const float* x0, const float* noise, const float* x_t, const T* out, int ld, const int64_t* t,
                         const float* sqrt_ac, const float* sqrt_1mac, const float* sqrt_recip_ac,
                         const float* sqrt_recipm1_ac, const float* loss_weight, const float* alphas_cumprod, LossArgs a,
                         T* dout, int ldd, int dpad, int B, float grad_scale, cudaStream_t s);
template <typename T> void launch_pack_piece(const float* src, int rows, int cols, T* dst, int ldd, int ws, T* dstT, int ldt, cudaStream_t s);
template <typename T> void launch_transpose_pad(const T* in, int ld, T* out, int ldo, int M, int Mcap, int C, float* colsum, cudaStream_t s);
void launch_unpack_piece_grad(const float* dpacked, int ldp, const float* w, int rows, int cols, float* dw, int ws, cudaStream_t s);
void launch_sumsq(const float* g, int64_t n, float* out, cudaStream_t s);
void launch_adam(float* p, const float* g, float* m, float* v, int64_t n, float lr, float b1, float b2, float eps, int step,
                 const float* sumsq_in, float max_norm, cudaStream_t s);
}  // namespace ds

namespace {
__global__ void k_vec_add(float* __restrict__ dst, const float* __restrict__ src, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] += src[i];
}
__global__ void k_iota(int* __restrict__ out, int n) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) out[i] = i;
}
// fp32 [B, cols] (row pitch ld) -> bf16 copy (row pitch ldo) for rows < B
__global__ void k_f32_to_bf16(const float* __restrict__ in, int ld, ds::bf16* __restrict__ out, int ldo, int B, int cols) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * cols) return;
  const int b = int(i / cols), c = int(i % cols);
  out[(int64_t)b * ldo + c] = __float2bfloat16_rn(in[(int64_t)b * ld + c]);
}
__global__ void k_bf16_to_f32(const ds::bf16* __restrict__ in, int ld, float* __restrict__ out, int ldo, int B, int cols) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= (int64_t)B * cols) return;
  const int b = int(i / cols), c = int(i % cols);
  out[(int64_t)b * ldo + c] = __bfloat162float(in[(int64_t)b * ld + c]);
}
// d(FiLM) of one time block: fp32 [B, cols] -> bf16 copy (for dX), bf16 transpose [cols, Bp] zero-padded (for dW), and
// the column sums (bias gradient), one pass
__global__ void k_dfilm_prepare(const float* __restrict__ in, int ld, ds::bf16* __restrict__ out, int ldo,
                                ds::bf16* __restrict__ outT, int Bp, int B, int cols, float* __restrict__ colsum) {
  __shared__ float tile[32][33];
  __shared__ float part[8][33];
  const int m0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  float cs = 0.f;
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int m = m0 + i, c = c0 + threadIdx.x;
    const float v = (m < B && c < cols) ? in[(int64_t)m * ld + c] : 0.f;
    tile[i][threadIdx.x] = v;
    cs += v;
    if (m < B && c < cols) out[(int64_t)m * ldo + c] = __float2bfloat16_rn(v);
  }
  part[threadIdx.y][threadIdx.x] = cs;
  __syncthreads();
  if (threadIdx.y == 0 && c0 + threadIdx.x < cols && m0 < B) {
    float tsum = 0.f;
#pragma unroll
    for (int y = 0; y < 8; ++y) tsum += part[y][threadIdx.x];
    atomicAdd(colsum + c0 + threadIdx.x, tsum);
  }
  for (int i = threadIdx.y; i < 32; i += 8) {
    const int c = c0 + i, m = m0 + threadIdx.x;
    if (c < cols && m < Bp) outT[(int64_t)c * Bp + m] = __float2bfloat16_rn(tile[threadIdx.x][i]);
  }
}
// dst = src * act'(z) elementwise (fp32 conditioning path)
__global__ void k_mul_actgrad(const float* __restrict__ g, const float* __restrict__ z, float* __restrict__ out, int64_t n, int act) {
  const int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float x = z[i];
  float d;
  if (act == ACT_GELU) {
    const float cdf = 0.5f * (1.0f + erff(x * 0.70710678118654752440f));
    d = cdf + x * 0.39894228040143267794f * expf(-0.5f * x * x);
  } else {
    const float sg = 1.0f / (1.0f + expf(-x));
    d = sg * (1.0f + x * (1.0f - sg));
  }
  out[i] = g[i] * d;
}
}  // namespace

struct TrainState {
  Plan plan;
  bool bf16 = false;
  size_t esz = 4;
  int cap_scenes = 0, rows_cap = 0;
  std::vector<void*> bufs, gbufs;
  char* warena = nullptr;
  std::vector<size_t> w_off;        // bytes
  float* dwarena = nullptr;
  std::vector<size_t> dw_off;       // floats
  size_t dw_total = 0;
  float *varena = nullptr, *dvarena = nullptr;
  std::vector<size_t> v_off;
  size_t v_total = 0;
  std::map<std::string, int64_t> flat_off;
  int64_t flat_n = 0;
  int pack_buf = -1;
  // per-sample conditioning path (fp32)
  float *emb = nullptr, *z1 = nullptr, *h1 = nullptr, *temb = nullptr, *st = nullptr, *film = nullptr, *dfilm = nullptr,
        *dst = nullptr, *dtemb = nullptr, *dh1 = nullptr;
  float *ctx_act = nullptr, *ctx_film = nullptr, *dctx_film = nullptr, *dctx_act = nullptr;
  int ctx_rows_cap = 0;
  int* t_idx = nullptr;
  int* t_int = nullptr;
  float* x_t = nullptr;
  float* loss_parts = nullptr;
  // bf16 mode: tensor-core plans.  Forward GEMMs and dX = dY W (W^T copies `wtarena`, K-major) run the row-major
  // tcgen05 kernel; dW = dY^T X runs it in split-K mode on transposed copies of dY and X (`trA`, `trB`: [C, rows_cap])
  bool use_tc = false;
  char* wtarena = nullptr;
  std::vector<TcGemmPlan*> tc_fwd;
  std::vector<TcGemmPlan*> tc_dx[2], tc_dw[2];
  ds::bf16 *trA = nullptr, *trB = nullptr;
  // time-FiLM projections on the tensor cores (bf16 mode): [B, 4C] x 19 x [2C, 4C]
  int Bp = 0;
  ds::bf16 *st_bf = nullptr, *film_bf = nullptr, *dfilm_bf = nullptr, *dst_bf = nullptr, *wall_bf = nullptr,
           *wallT_bf = nullptr, *trF = nullptr, *stT = nullptr;
  float* ball = nullptr;
  std::vector<TcGemmPlan*> tc_film;      // forward, one per <= 4096-column chunk
  std::vector<int> tc_film_n0;
  TcGemmPlan* tc_dst = nullptr;
  std::vector<TcGemmPlan*> tc_dwf;       // dW of every time block (split-K, fp32 atomics straight into the flat gradients)
  // gradient buckets for the overlapped data-parallel all-reduce: bucket k = flat range [bounds[k], bounds[k + 1]);
  // its event is recorded as soon as every parameter gradient inside it is final (the backward pass finalises the
  // flat buffer from its END towards its start: parameters are laid out in forward order)
  std::vector<int64_t> bucket_bounds;
  std::vector<cudaEvent_t> bucket_events;
  // text condition (ds_train_set_context_cross; the pointers are borrowed).  The to_kv projections of all cross-attention
  // layers run as ONE GEMM: kv [B*L, NKV] = context_cross [B*L, TD] x kvw^T, kvw = the layers' to_kv weights stacked
  // [NKV = layers * 256, TD] in storage dtype.  bf16 with the tcgen05 backend (`text_tc`): the forward, d(to_kv.weight)
  // (split-K on the transposed copies trKV = dkv_l^T, crossT) and d(context_cross) = dkv x kvw (kvwT: K-major copy)
  // run on the tensor cores
  const float* cross = nullptr;
  float* dcross = nullptr;
  int cross_batch = 0, cross_L = 0;
  bool text_tc = false;
  int x_rows_cap = 0, x_rows_pad = 0, x_scenes_cap = 0;
  void *kvw = nullptr, *kv = nullptr, *dkv = nullptr;
  float* xctx = nullptr;                 // [layers][B][4][32][32] text context of every layer
  ds::bf16 *kvwT = nullptr, *cross_bf = nullptr, *crossT = nullptr, *trKV = nullptr, *dcross_bf = nullptr;
  TcGemmPlan *tc_kv = nullptr, *tc_kvdw = nullptr, *tc_dcross = nullptr;
  cudaEvent_t ev[7] = {nullptr};      // phase boundaries of the last step (ds_train_phase_ms)
  bool ev_valid = false;
};

void train_state_destroy(TrainState* t) {
  if (!t) return;
  for (void* p : t->bufs) cudaFree(p);
  for (void* p : t->gbufs) cudaFree(p);
  cudaFree(t->warena); cudaFree(t->dwarena); cudaFree(t->varena); cudaFree(t->dvarena);
  for (float* p : {t->emb, t->z1, t->h1, t->temb, t->st, t->film, t->dfilm, t->dst, t->dtemb, t->dh1, t->ctx_act,
                   t->ctx_film, t->dctx_film, t->dctx_act, t->x_t, t->loss_parts})
    cudaFree(p);
  cudaFree(t->t_idx); cudaFree(t->t_int);
  for (auto e : t->ev) if (e) cudaEventDestroy(e);
  for (auto* p : t->tc_fwd) if (p) tc_plan_destroy(p);
  for (int k = 0; k < 2; ++k) {
    for (auto* p : t->tc_dx[k]) if (p) tc_plan_destroy(p);
    for (auto* p : t->tc_dw[k]) if (p) tc_plan_destroy(p);
  }
  cudaFree(t->wtarena); cudaFree(t->trA); cudaFree(t->trB);
  for (auto* p : t->tc_film) if (p) tc_plan_destroy(p);
  for (auto* p : t->tc_dwf) if (p) tc_plan_destroy(p);
  if (t->tc_dst) tc_plan_destroy(t->tc_dst);
  for (ds::bf16* p : {t->st_bf, t->film_bf, t->dfilm_bf, t->dst_bf, t->wall_bf, t->wallT_bf, t->trF, t->stT}) cudaFree(p);
  cudaFree(t->ball);
  for (void* p : {t->kvw, t->kv, t->dkv, (void*)t->xctx, (void*)t->kvwT, (void*)t->cross_bf, (void*)t->crossT, (void*)t->trKV,
                  (void*)t->dcross_bf})
    cudaFree(p);
  for (auto* p : {t->tc_kv, t->tc_kvdw, t->tc_dcross}) if (p) tc_plan_destroy(p);
  delete t;
}

static int train_round_up(int a, int b) { return (a + b - 1) / b * b; }

static int train_init(ds_handle* h) {
  if (h->train) return 0;
  TrainState* t = new TrainState();
  ds_config cfg = h->cfg;
  cfg.train = 1;
  cfg.fuse_level = 0;
  if (!build_plan(cfg, true, &t->plan)) {
    int rc = fail(DS_ERR_INVALID, "%s", t->plan.error.c_str());
    delete t;
    return rc;
  }
  const Plan& P = t->plan;
  t->bf16 = h->bf16_mode;
  t->esz = t->bf16 ? 2 : 4;
  for (const Op& o : P.ops)
    if (o.kind == OP_PACK) t->pack_buf = o.out;
  // flat layout = the handle's expected order (identical name set: train mode changes ops, not parameters)
  int64_t off = 0;
  for (const std::string& n : h->plan.expected_order) {
    t->flat_off[n] = off;
    off += h->plan.expected[n];
  }
  t->flat_n = off;
  for (const std::string& n : P.expected_order)
    if (!t->flat_off.count(n)) {
      int rc = fail(DS_ERR_STATE, "train plan expects parameter '%s' unknown to the handle", n.c_str());
      delete t;
      return rc;
    }
  size_t total = 0, dtot = 0;
  t->w_off.resize(P.wmats.size());
  t->dw_off.resize(P.wmats.size());
  for (size_t i = 0; i < P.wmats.size(); ++i) {
    t->w_off[i] = total;
    t->dw_off[i] = dtot;
    total += ((size_t)P.wmats[i].N * P.wmats[i].K * t->esz + 255) / 256 * 256;
    dtot += (size_t)P.wmats[i].N * P.wmats[i].K;
  }
  t->dw_total = dtot;
  CK(cudaMalloc(&t->warena, total));
  CK(cudaMemset(t->warena, 0, total));
  t->use_tc = h->use_tc;
  if (t->use_tc) {
    CK(cudaMalloc(&t->wtarena, total));
    CK(cudaMemset(t->wtarena, 0, total));
  }
  CK(cudaMalloc(&t->dwarena, dtot * 4));
  size_t vt = 0;
  t->v_off.resize(P.vecs.size());
  for (size_t i = 0; i < P.vecs.size(); ++i) {
    t->v_off[i] = vt;
    vt += (size_t)train_round_up(P.vecs[i].n, 64);
  }
  t->v_total = vt;
  CK(cudaMalloc(&t->varena, vt * 4));
  CK(cudaMalloc(&t->dvarena, vt * 4));
  if (h->cfg.text_condition) {
    const int TD = h->cfg.text_dim, NKV = int(P.xattn_layers.size()) * 256;
    t->text_tc = t->use_tc && TD % 128 == 0;      // tcgen05 shape rules: K % 64 and N % 128 (TD is both)
    CK(cudaMalloc(&t->kvw, (size_t)NKV * TD * t->esz));
    if (t->text_tc) CK(cudaMalloc(&t->kvwT, (size_t)TD * NKV * 2));
  }
  h->train = t;
  return 0;
}

// text buffers and plans for B scenes of L tokens; grown (never shrunk) like train_capacity's, since L follows the
// longest description of each batch
static int train_text_capacity(ds_handle* h, int B, int L) {
  TrainState* t = h->train;
  const int nl = int(t->plan.xattn_layers.size()), TD = h->cfg.text_dim, NKV = nl * 256;
  if (B > t->x_scenes_cap) {
    cudaFree(t->xctx);
    t->xctx = nullptr;
    CK(cudaMalloc(&t->xctx, (size_t)nl * B * 4096 * 4));
    t->x_scenes_cap = B;
  }
  const int rows = B * L;
  if (rows <= t->x_rows_cap) return 0;
  for (void* p : {t->kv, t->dkv, (void*)t->cross_bf, (void*)t->crossT, (void*)t->trKV, (void*)t->dcross_bf}) cudaFree(p);
  t->kv = t->dkv = nullptr;
  t->cross_bf = t->crossT = t->trKV = t->dcross_bf = nullptr;
  for (TcGemmPlan** p : {&t->tc_kv, &t->tc_kvdw, &t->tc_dcross}) {
    if (*p) tc_plan_destroy(*p);
    *p = nullptr;
  }
  t->x_rows_cap = t->x_rows_pad = 0;
  const int rp = train_round_up(rows, 128);
  auto alloc0 = [&](void** p, size_t bytes) { cudaError_t e = cudaMalloc(p, bytes); if (e == cudaSuccess) e = cudaMemset(*p, 0, bytes); return e; };
  CK(alloc0(&t->kv, (size_t)rp * NKV * t->esz));
  CK(alloc0(&t->dkv, (size_t)rp * NKV * t->esz));
  if (t->bf16) {
    CK(alloc0((void**)&t->cross_bf, (size_t)rp * TD * 2));
    CK(alloc0((void**)&t->dcross_bf, (size_t)rp * TD * 2));
  }
  if (t->text_tc) {
    CK(alloc0((void**)&t->crossT, (size_t)TD * rp * 2));
    CK(alloc0((void**)&t->trKV, (size_t)256 * rp * 2));
    char err[256] = "";
    GemmArgs g;
    memset(&g, 0, sizeof g);
    g.no_pair = 1;      // training GEMMs stay single-CTA (kernels.cuh)
    g.a0 = t->cross_bf; g.lda0 = TD; g.k0 = TD;
    g.w = t->kvw; g.ldw = TD;
    g.d = t->kv; g.ldd = NKV;
    g.M = rp; g.N = NKV;
    if (!(t->tc_kv = tc_plan_create(g, rp, err, sizeof err))) return fail(DS_ERR_CUDA, "train: to_kv plan failed: %s", err);
    // d(to_kv.weight) of one layer = dkv_l^T x context_cross: A = trKV [256, rp], "weights" = crossT [TD, rp]
    memset(&g, 0, sizeof g);
    g.no_pair = 1;
    g.a0 = t->trKV; g.lda0 = rp; g.k0 = rp;
    g.w = t->crossT; g.ldw = rp;
    g.d = t->trKV; g.ldd = 8;             // placeholder (bf16 output unused in atomic mode)
    g.M = 256; g.N = TD;
    if (!(t->tc_kvdw = tc_plan_create(g, 256, err, sizeof err)))
      return fail(DS_ERR_CUDA, "train: to_kv weight-gradient plan failed: %s", err);
    // d(context_cross) = dkv [rows, NKV] x kvw [NKV, TD]: "weights" = kvwT [TD, NKV]
    memset(&g, 0, sizeof g);
    g.no_pair = 1;
    g.a0 = t->dkv; g.lda0 = NKV; g.k0 = NKV;
    g.w = t->kvwT; g.ldw = NKV;
    g.d = t->dcross_bf; g.ldd = TD;
    g.M = rp; g.N = TD;
    if (!(t->tc_dcross = tc_plan_create(g, rp, err, sizeof err)))
      return fail(DS_ERR_CUDA, "train: d(context_cross) plan failed: %s", err);
  }
  t->x_rows_cap = rows;
  t->x_rows_pad = rp;
  return 0;
}

// split-K factor of a dW GEMM with `tiles` output tiles over `kblocks` 64-deep k-blocks: one wave of CTAs, every split
// owning at least one k-block (the kernel derives its k-blocks per split the same way)
static int train_ksplit(int tiles, int kblocks) {
  int ksplit = std::max(1, std::min(148 / std::max(1, tiles), kblocks));
  const int kb_per = (kblocks + ksplit - 1) / ksplit;
  return (kblocks + kb_per - 1) / kb_per;
}

static int train_capacity(ds_handle* h, int n_scenes, int ctx_rows) {
  TrainState* t = h->train;
  const Plan& P = t->plan;
  const int n_obj = h->cfg.num_objects, C = P.C;
  if (n_scenes > t->cap_scenes) {
    for (void* p : t->bufs) cudaFree(p);
    for (void* p : t->gbufs) cudaFree(p);
    t->bufs.assign(P.buf_width.size(), nullptr);
    t->gbufs.assign(P.buf_width.size(), nullptr);
    t->rows_cap = train_round_up(n_scenes * n_obj, 128);
    for (size_t i = 0; i < P.buf_width.size(); ++i) {
      const size_t bytes = (size_t)t->rows_cap * P.buf_width[i] * t->esz;
      CK(cudaMalloc(&t->bufs[i], bytes));
      CK(cudaMemset(t->bufs[i], 0, bytes));
      CK(cudaMalloc(&t->gbufs[i], bytes));
      CK(cudaMemset(t->gbufs[i], 0, bytes));
    }
    const int ntb = int(P.time_blocks.size());
    for (float** p : {&t->emb, &t->z1, &t->h1, &t->temb, &t->st, &t->film, &t->dfilm, &t->dst, &t->dtemb, &t->dh1, &t->x_t,
                      &t->loss_parts}) {
      cudaFree(*p);
      *p = nullptr;
    }
    cudaFree(t->t_idx); cudaFree(t->t_int);
    const size_t B = n_scenes;
    CK(cudaMalloc(&t->emb, B * C * 4));
    CK(cudaMalloc(&t->z1, B * 4 * C * 4));
    CK(cudaMalloc(&t->h1, B * 4 * C * 4));
    CK(cudaMalloc(&t->temb, B * 4 * C * 4));
    CK(cudaMalloc(&t->st, B * 4 * C * 4));
    CK(cudaMalloc(&t->film, B * ntb * 2 * C * 4));
    CK(cudaMalloc(&t->dfilm, B * ntb * 2 * C * 4));
    CK(cudaMalloc(&t->dst, B * 4 * C * 4));
    CK(cudaMalloc(&t->dtemb, B * 4 * C * 4));
    CK(cudaMalloc(&t->dh1, B * 4 * C * 4));
    CK(cudaMalloc(&t->x_t, B * n_obj * P.d * 4));
    CK(cudaMalloc(&t->loss_parts, B * 9 * 4));
    CK(cudaMalloc(&t->t_idx, B * 4));
    CK(cudaMalloc(&t->t_int, B * 4));
    k_iota<<<(n_scenes + 255) / 256, 256>>>(t->t_idx, n_scenes);
    if (t->use_tc) {
      for (auto* p : t->tc_fwd) if (p) tc_plan_destroy(p);
      for (int k = 0; k < 2; ++k) {
        for (auto* p : t->tc_dx[k]) if (p) tc_plan_destroy(p);
        for (auto* p : t->tc_dw[k]) if (p) tc_plan_destroy(p);
        t->tc_dx[k].assign(P.ops.size(), nullptr);
        t->tc_dw[k].assign(P.ops.size(), nullptr);
      }
      t->tc_fwd.assign(P.ops.size(), nullptr);
      cudaFree(t->trA); cudaFree(t->trB);
      int maxw = 0;
      for (int w : P.buf_width) maxw = std::max(maxw, w);
      CK(cudaMalloc(&t->trA, (size_t)maxw * t->rows_cap * 2));
      CK(cudaMalloc(&t->trB, (size_t)maxw * t->rows_cap * 2));
      char err[256] = "";
      auto bp = [&](std::vector<void*>& v, int buf, int col) -> bf16* { return buf < 0 ? nullptr : (bf16*)v[buf] + col; };
      for (size_t i = 0; i < P.ops.size(); ++i) {
        const Op& o = P.ops[i];
        if (o.kind != OP_GEMM) continue;
        const int K = P.wmats[o.w].K, Npad = P.wmats[o.w].N;
        GemmArgs g;
        memset(&g, 0, sizeof g);
        g.no_pair = 1;      // training GEMMs stay single-CTA (kernels.cuh)
        g.a0 = bp(t->bufs, o.in0.buf, o.in0.col); g.lda0 = P.buf_width[o.in0.buf]; g.k0 = o.in0.k;
        g.a1 = bp(t->bufs, o.in1.buf, o.in1.col); g.lda1 = o.in1.buf >= 0 ? P.buf_width[o.in1.buf] : 0;
        g.k1 = o.in1.buf >= 0 ? o.in1.k : 0;
        g.w = t->warena + t->w_off[o.w]; g.ldw = K;
        g.bias = o.b >= 0 ? t->varena + t->v_off[o.b] : nullptr;
        g.d = bp(t->bufs, o.out, o.out_col); g.ldd = P.buf_width[o.out];
        g.res = bp(t->bufs, o.res, 0); g.ldres = o.res >= 0 ? P.buf_width[o.res] : 0;
        g.M = t->rows_cap; g.N = o.N; g.act = o.act;
        t->tc_fwd[i] = tc_plan_create(g, t->rows_cap, err, sizeof err);
        if (!t->tc_fwd[i]) return fail(DS_ERR_CUDA, "train: tcgen05 plan for '%s' failed: %s", o.name.c_str(), err);
        const Slice* ins[2] = {&o.in0, &o.in1};
        int koff = 0;
        for (int k2 = 0; k2 < 2; ++k2) {
          const Slice& in = *ins[k2];
          if (in.buf < 0) continue;
          // dX = dY W : A = dY [M, N], "weights" = W^T rows [koff, koff + k) of [K, Npad]; accumulates in place
          if (in.buf != t->pack_buf && in.k % 128 == 0 && o.N % 64 == 0) {
            memset(&g, 0, sizeof g);
            g.no_pair = 1;      // training GEMMs stay single-CTA (kernels.cuh)
            g.a0 = bp(t->gbufs, o.out, o.out_col); g.lda0 = P.buf_width[o.out]; g.k0 = o.N;
            g.w = (bf16*)(t->wtarena + t->w_off[o.w]) + (size_t)koff * Npad; g.ldw = Npad;
            g.d = bp(t->gbufs, in.buf, in.col); g.ldd = P.buf_width[in.buf];
            g.res = g.d; g.ldres = g.ldd;      // the launcher clears it for first writers
            g.M = t->rows_cap; g.N = in.k;
            t->tc_dx[k2][i] = tc_plan_create(g, t->rows_cap, err, sizeof err);
            if (!t->tc_dx[k2][i]) return fail(DS_ERR_CUDA, "train: dX plan for '%s' failed: %s", o.name.c_str(), err);
          }
          // dW = dY^T X on the transposed copies: A = dY^T [N, rows_cap], "weights" = X^T [k, rows_cap]
          if (in.k % 128 == 0 && o.N % 128 == 0) {
            memset(&g, 0, sizeof g);
            g.no_pair = 1;      // training GEMMs stay single-CTA (kernels.cuh)
            g.a0 = t->trA; g.lda0 = t->rows_cap; g.k0 = t->rows_cap;
            g.w = t->trB; g.ldw = t->rows_cap;
            g.d = t->trA; g.ldd = 8;             // placeholder (bf16 output unused in atomic mode)
            g.M = o.N; g.N = in.k;
            t->tc_dw[k2][i] = tc_plan_create(g, o.N, err, sizeof err);
            if (!t->tc_dw[k2][i]) return fail(DS_ERR_CUDA, "train: dW plan for '%s' failed: %s", o.name.c_str(), err);
            const int tiles = tc_plan_tiles(t->tc_dw[k2][i], o.N);
            int ksplit = std::max(1, 148 / std::max(1, tiles));      // one wave of CTAs: fewer partial sums to reduce
            const int kblocks = t->rows_cap / 64;
            ksplit = std::min(ksplit, kblocks);
            const int kb_per = (kblocks + ksplit - 1) / ksplit;
            ksplit = (kblocks + kb_per - 1) / kb_per;      // every split owns at least one k-block (the kernel derives kb_per the same way)
            tc_plan_set_atomic_out(t->tc_dw[k2][i], t->dwarena + t->dw_off[o.w] + koff, K, ksplit);
          }
          koff += in.k;
        }
      }
    }
    if (t->use_tc) {
      const int W4 = 4 * C, NF = int(P.time_blocks.size()) * 2 * C;
      t->Bp = train_round_up(n_scenes, 128);
      for (auto* p : t->tc_film) if (p) tc_plan_destroy(p);
      for (auto* p : t->tc_dwf) if (p) tc_plan_destroy(p);
      if (t->tc_dst) tc_plan_destroy(t->tc_dst);
      t->tc_film.clear(); t->tc_film_n0.clear(); t->tc_dwf.clear(); t->tc_dst = nullptr;
      for (ds::bf16** p : {&t->st_bf, &t->film_bf, &t->dfilm_bf, &t->dst_bf, &t->wall_bf, &t->wallT_bf, &t->trF, &t->stT}) {
        cudaFree(*p);
        *p = nullptr;
      }
      cudaFree(t->ball); t->ball = nullptr;
      auto alloc0 = [&](ds::bf16** p, size_t n) { cudaError_t e = cudaMalloc(p, n * 2); if (e == cudaSuccess) e = cudaMemset(*p, 0, n * 2); return e; };
      CK(alloc0(&t->st_bf, (size_t)t->Bp * W4));
      CK(alloc0(&t->film_bf, (size_t)t->Bp * NF));
      CK(alloc0(&t->dfilm_bf, (size_t)t->Bp * NF));
      CK(alloc0(&t->dst_bf, (size_t)t->Bp * W4));
      CK(alloc0(&t->wall_bf, (size_t)NF * W4));
      CK(alloc0(&t->wallT_bf, (size_t)W4 * NF));
      CK(alloc0(&t->trF, (size_t)NF * t->Bp));
      CK(alloc0(&t->stT, (size_t)W4 * t->Bp));
      CK(cudaMalloc(&t->ball, (size_t)NF * 4));
      char err[256] = "";
      GemmArgs g;
      for (int n0 = 0; n0 < NF; n0 += 4096) {
        const int nn = std::min(4096, NF - n0);
        memset(&g, 0, sizeof g);
        g.no_pair = 1;      // training GEMMs stay single-CTA (kernels.cuh)
        g.a0 = t->st_bf; g.lda0 = W4; g.k0 = W4;
        g.w = t->wall_bf + (size_t)n0 * W4; g.ldw = W4;
        g.bias = t->ball + n0;
        g.d = t->film_bf + n0; g.ldd = NF;
        g.M = t->Bp; g.N = nn;
        TcGemmPlan* p = tc_plan_create(g, t->Bp, err, sizeof err);
        if (!p) return fail(DS_ERR_CUDA, "train: FiLM projection plan failed: %s", err);
        t->tc_film.push_back(p);
        t->tc_film_n0.push_back(n0);
      }
      memset(&g, 0, sizeof g);
      g.no_pair = 1;      // training GEMMs stay single-CTA (kernels.cuh)
      g.a0 = t->dfilm_bf; g.lda0 = NF; g.k0 = NF;
      g.w = t->wallT_bf; g.ldw = NF;
      g.d = t->dst_bf; g.ldd = W4;
      g.M = t->Bp; g.N = W4;
      t->tc_dst = tc_plan_create(g, t->Bp, err, sizeof err);
      if (!t->tc_dst) return fail(DS_ERR_CUDA, "train: d(time embedding) plan failed: %s", err);
      for (size_t i = 0; i < P.time_blocks.size(); ++i) {
        memset(&g, 0, sizeof g);
        g.no_pair = 1;      // training GEMMs stay single-CTA (kernels.cuh)
        g.a0 = t->trF + i * (size_t)2 * C * t->Bp; g.lda0 = t->Bp; g.k0 = t->Bp;
        g.w = t->stT; g.ldw = t->Bp;
        g.d = t->trF; g.ldd = 8;
        g.M = 2 * C; g.N = W4;
        TcGemmPlan* p = tc_plan_create(g, 2 * C, err, sizeof err);
        if (!p) return fail(DS_ERR_CUDA, "train: FiLM weight-gradient plan failed: %s", err);
        t->tc_dwf.push_back(p);
      }
    }
    t->cap_scenes = n_scenes;
  }
  if (ctx_rows > t->ctx_rows_cap) {
    const int ncb = int(P.ctx_blocks.size()), E = h->cfg.cond_dim;
    for (float** p : {&t->ctx_act, &t->ctx_film, &t->dctx_film, &t->dctx_act}) {
      cudaFree(*p);
      *p = nullptr;
    }
    CK(cudaMalloc(&t->ctx_act, (size_t)ctx_rows * E * 4));
    CK(cudaMalloc(&t->dctx_act, (size_t)ctx_rows * E * 4));
    CK(cudaMalloc(&t->ctx_film, (size_t)ctx_rows * ncb * 2 * C * 4));
    CK(cudaMalloc(&t->dctx_film, (size_t)ctx_rows * ncb * 2 * C * 4));
    t->ctx_rows_cap = ctx_rows;
  }
  return 0;
}

template <typename T>
static int train_step_t(ds_handle* h, const float* flat, const float* x0, const int64_t* t64, const float* noise,
                        const float* context, int ctx_batch, int ctx_shared, int loss_separate, int loss_iou,
                        const float* bounds_host, float grad_scale, float* losses, float* loss_dict, float* grads,
                        float* dcontext, int B, cudaStream_t s) {
  TrainState* t = h->train;
  const Plan& P = t->plan;
  const ds_config& c = h->cfg;
  const int n_obj = c.num_objects, M = B * n_obj, C = P.C, E = c.cond_dim;
  const int ntb = int(P.time_blocks.size()), ncb = int(P.ctx_blocks.size());
  const int ctx_rows = ctx_shared ? n_obj : ctx_batch * n_obj;
  auto F = [&](const std::string& name) { return flat + t->flat_off.at(name); };
  auto G = [&](const std::string& name) { return grads + t->flat_off.at(name); };
  auto ptr = [&](int buf, int col) -> T* { return buf < 0 ? nullptr : (T*)t->bufs[buf] + col; };
  auto gptr = [&](int buf, int col) -> T* { return buf < 0 ? nullptr : (T*)t->gbufs[buf] + col; };
  auto ld = [&](int buf) { return buf < 0 ? 0 : P.buf_width[buf]; };

  for (auto& e : t->ev) if (!e) cudaEventCreate(&e);
  t->ev_valid = false;
  cudaEventRecord(t->ev[0], s);
  // ---- 1. weights: flat fp32 -> packed matrices (weight standardisation folded, storage dtype) and vectors
  for (size_t i = 0; i < P.wmats.size(); ++i) {
    const WRecipe& r = P.wmats[i];
    for (const WPiece& pc : r.pieces)
      launch_pack_piece<T>(F(pc.name), pc.rows, pc.cols, (T*)(t->warena + t->w_off[i]) + (size_t)pc.row_off * r.K + pc.col_off,
                           r.K, r.ws ? 1 : 0,
                           t->use_tc ? (T*)(t->wtarena + t->w_off[i]) + (size_t)pc.col_off * r.N + pc.row_off : nullptr, r.N, s);
  }
  const bool text = c.text_condition != 0;
  const int TD = c.text_dim, NKV = int(P.xattn_layers.size()) * 256, XL = t->cross_L, XR = B * XL;
  for (size_t l = 0; text && l < P.xattn_layers.size(); ++l)
    launch_pack_piece<T>(F(P.xattn_layers[l] + ".fn.fn.to_kv.weight"), 256, TD, (T*)t->kvw + l * 256 * TD, TD, 0,
                         t->text_tc ? (T*)(void*)t->kvwT + l * 256 : nullptr, NKV, s);
  CK(cudaMemsetAsync(t->varena, 0, t->v_total * 4, s));
  for (size_t i = 0; i < P.vecs.size(); ++i)
    for (const VPiece& pc : P.vecs[i].pieces)
      k_vec_add<<<(pc.n + 255) / 256, 256, 0, s>>>(t->varena + t->v_off[i] + pc.off, F(pc.name), pc.n);

  cudaEventRecord(t->ev[1], s);
  // ---- 2. forward
  launch_q_sample(x0, t64, noise, t->x_t, h->sched_dev[S_SQRT_AC], h->sched_dev[S_SQRT_1MAC], B, n_obj * P.d, s);
  launch_t_convert(t64, t->t_int, B, s);
  if (!h->sin_freq) {
    std::vector<float> hf(C / 2);
    sinusoid_freqs_host(C, hf.data());
    CK(cudaMalloc(&h->sin_freq, hf.size() * 4));
    CK(cudaMemcpy(h->sin_freq, hf.data(), hf.size() * 4, cudaMemcpyHostToDevice));
  }
  launch_sinusoid_t(t->emb, h->sin_freq, t->t_int, B, C, s);
  GemmArgs g;
  auto f32gemm = [&](const float* a, int lda, int K, const float* w, const float* b, float* d, int ldd, int N, int rows) {
    memset(&g, 0, sizeof g);
    g.no_pair = 1;      // training GEMMs stay single-CTA (kernels.cuh)
    g.a0 = a; g.lda0 = lda; g.k0 = K; g.w = w; g.ldw = K; g.bias = b; g.d = d; g.ldd = ldd; g.M = rows; g.N = N; g.act = ACT_NONE;
    launch_gemm_f32(g, s);
  };
  // time_mlp = Sequential(SinusoidalPosEmb, Linear, GELU, Linear) (denoise_net.py:417-422); every ResnetBlock applies
  // SiLU then its own Linear(4C -> 2C) (:181-184)
  f32gemm(t->emb, C, C, F("time_mlp.1.weight"), F("time_mlp.1.bias"), t->z1, 4 * C, 4 * C, B);
  launch_act<float>(t->z1, 4 * C, t->h1, 4 * C, B, 4 * C, ACT_GELU, s);
  f32gemm(t->h1, 4 * C, 4 * C, F("time_mlp.3.weight"), F("time_mlp.3.bias"), t->temb, 4 * C, 4 * C, B);
  launch_act<float>(t->temb, 4 * C, t->st, 4 * C, B, 4 * C, ACT_SILU, s);
  const bool film_tc = t->use_tc && !t->tc_film.empty();
  if (film_tc) {
    // the 19 time-FiLM projections [B, 4C] -> [B, 19 x 2C] on the tensor cores: bf16 copies of SiLU(temb) and of the
    // block weights (plus their transposes for d(temb)), fp32 accumulation, result widened back to the fp32 table
    const int W4 = 4 * C, NF = ntb * 2 * C;
    for (int i = 0; i < ntb; ++i) {
      launch_pack_piece<bf16>(F(P.time_blocks[i] + ".mlp.1.weight"), 2 * C, W4, t->wall_bf + (size_t)i * 2 * C * W4, W4, 0,
                              t->wallT_bf + (size_t)i * 2 * C, NF, s);
      CK(cudaMemcpyAsync(t->ball + (size_t)i * 2 * C, F(P.time_blocks[i] + ".mlp.1.bias"), (size_t)2 * C * 4, cudaMemcpyDeviceToDevice, s));
    }
    k_f32_to_bf16<<<((int64_t)B * W4 + 255) / 256, 256, 0, s>>>(t->st, W4, t->st_bf, W4, B, W4);
    for (auto* p : t->tc_film) {
      int e = launch_gemm_tc(p, t->Bp, s);
      if (e) return fail(DS_ERR_CUDA, "train: FiLM projection GEMM failed: %s", cudaGetErrorString((cudaError_t)e));
    }
    k_bf16_to_f32<<<((int64_t)B * NF + 255) / 256, 256, 0, s>>>(t->film_bf, NF, t->film, NF, B, NF);
  } else {
    for (int i = 0; i < ntb; ++i)
      f32gemm(t->st, 4 * C, 4 * C, F(P.time_blocks[i] + ".mlp.1.weight"), F(P.time_blocks[i] + ".mlp.1.bias"),
              t->film + (size_t)i * 2 * C, ntb * 2 * C, 2 * C, B);
  }
  launch_act<float>(context, E, t->ctx_act, E, ctx_rows, E, ACT_SILU, s);
  for (int i = 0; i < ncb; ++i)
    f32gemm(t->ctx_act, E, E, F(P.ctx_blocks[i] + ".mlp.1.weight"), F(P.ctx_blocks[i] + ".mlp.1.bias"),
            t->ctx_film + (size_t)i * 2 * C, ncb * 2 * C, 2 * C, ctx_rows);
  if (text) {
    // k | v of every cross-attention layer in one GEMM, then each layer's text context [B, 4, 32, 32]
    if (t->bf16) {
      k_f32_to_bf16<<<((int64_t)XR * TD + 255) / 256, 256, 0, s>>>(t->cross, TD, t->cross_bf, TD, XR, TD);
      h->launches++;
    }
    if (t->text_tc) {
      int e = launch_gemm_tc(t->tc_kv, XR, s);
      if (e) return fail(DS_ERR_CUDA, "train: to_kv GEMM failed: %s", cudaGetErrorString((cudaError_t)e));
    } else {
      memset(&g, 0, sizeof g);
      g.a0 = t->bf16 ? (const void*)t->cross_bf : (const void*)t->cross; g.lda0 = TD; g.k0 = TD;
      g.w = t->kvw; g.ldw = TD; g.d = t->kv; g.ldd = NKV; g.M = XR; g.N = NKV; g.act = ACT_NONE;
      if constexpr (sizeof(T) == 4) launch_gemm_f32(g, s);
      else launch_gemm_simt<T>(g, true, s);
    }
    for (size_t l = 0; l < P.xattn_layers.size(); ++l)
      launch_xattn_prepare<T>((const T*)t->kv + l * 256, NKV, t->xctx + l * B * 4096, B, XL, s);
    h->launches += 1 + int(P.xattn_layers.size());
  }

  auto film_of = [&](const Op& o) {
    FilmRef f;
    f.base = nullptr; f.mode = FILM_NONE; f.row_stride = 0; f.t = t->t_idx;
    if (o.film == 1) { f.base = t->film + (size_t)o.film_blk * 2 * C; f.mode = FILM_TIME; f.row_stride = (int64_t)ntb * 2 * C; }
    else if (o.film == 2) {
      f.base = t->ctx_film + (size_t)o.film_blk * 2 * C;
      f.mode = ctx_shared ? FILM_OBJECT : FILM_TOKEN;
      f.row_stride = (int64_t)ncb * 2 * C;
    }
    return f;
  };
  for (const Op& o : P.ops) {
    switch (o.kind) {
      case OP_PACK:
        launch_pack_input<T>(t->x_t, (T*)t->bufs[o.out], P.kin_pad, M, P.d, s);
        break;
      case OP_GEMM: {
        memset(&g, 0, sizeof g);
        g.no_pair = 1;      // training GEMMs stay single-CTA (kernels.cuh)
        g.a0 = ptr(o.in0.buf, o.in0.col); g.lda0 = ld(o.in0.buf); g.k0 = o.in0.k;
        g.a1 = ptr(o.in1.buf, o.in1.col); g.lda1 = ld(o.in1.buf); g.k1 = o.in1.buf >= 0 ? o.in1.k : 0;
        g.w = t->warena + t->w_off[o.w]; g.ldw = P.wmats[o.w].K;
        g.bias = o.b >= 0 ? t->varena + t->v_off[o.b] : nullptr;
        g.d = ptr(o.out, o.out_col); g.ldd = ld(o.out);
        g.res = ptr(o.res, 0); g.ldres = ld(o.res);
        g.M = M; g.N = o.N; g.act = o.act;
        if (t->use_tc && t->tc_fwd[&o - &P.ops[0]]) {
          int e = launch_gemm_tc(t->tc_fwd[&o - &P.ops[0]], M, s);
          if (e) return fail(DS_ERR_CUDA, "train: tcgen05 GEMM '%s' failed: %s", o.name.c_str(), cudaGetErrorString((cudaError_t)e));
        } else {
          launch_gemm_simt<T>(g, true, s);
        }
        break;
      }
      case OP_ACT:
        launch_act<T>(ptr(o.in0.buf, o.in0.col), ld(o.in0.buf), ptr(o.out, o.out_col), ld(o.out), M, o.N, o.act, s);
        break;
      case OP_GN:
        if (!launch_gn_fwd_reg<T>(ptr(o.in0.buf, 0), ld(o.in0.buf), ptr(o.out, 0), ld(o.out), t->varena + t->v_off[o.gamma],
                                  t->varena + t->v_off[o.beta], film_of(o), ptr(o.res, 0), ld(o.res), B, n_obj, C, 8, s))
          launch_groupnorm<T>(ptr(o.in0.buf, 0), ld(o.in0.buf), ptr(o.out, 0), ld(o.out), t->varena + t->v_off[o.gamma],
                              t->varena + t->v_off[o.beta], film_of(o), ptr(o.res, 0), ld(o.res), B, n_obj, C, 8, s);
        break;
      case OP_LN:
        launch_layernorm<T>(ptr(o.in0.buf, 0), ld(o.in0.buf), ptr(o.out, 0), ld(o.out), t->varena + t->v_off[o.b],
                            ptr(o.res, 0), ld(o.res), M, C, s);
        break;
      case OP_LINATTN:
        launch_linattn<T>(ptr(o.in0.buf, 0), ld(o.in0.buf), ptr(o.out, 0), ld(o.out), B, n_obj, s);
        break;
      case OP_ATTN:
        launch_softattn<T>(ptr(o.in0.buf, 0), ld(o.in0.buf), ptr(o.out, 0), ld(o.out), B, n_obj, s);
        break;
      case OP_XATTN:
        launch_xattn_apply<T>(ptr(o.in0.buf, 0), ld(o.in0.buf), t->xctx + (size_t)o.xlayer * B * 4096, ptr(o.out, 0), ld(o.out),
                              B, n_obj, s);
        break;
      default:
        return fail(DS_ERR_STATE, "op kind %d has no training path", o.kind);
    }
    h->launches++;
  }

  cudaEventRecord(t->ev[2], s);
  // ---- 3. loss value (per-sample losses + the 9 dict means) and d(loss) / d(model output)
  LossArgs a;
  memset(&a, 0, sizeof a);
  a.n_obj = n_obj; a.d = P.d; a.trans = c.translation_dim; a.size = c.size_dim; a.angle = c.angle_dim;
  a.cls = c.class_dim; a.objn = c.objectness_dim; a.feat = c.objfeat_dim;
  a.mean_type = h->mean_type; a.loss_separate = loss_separate; a.loss_iou = loss_iou;
  a.arrange = c.seperate_all ? 0 : 1;
  if (a.arrange) { a.angle = P.d - a.trans; a.loss_iou = 0; }
  if (bounds_host) memcpy(a.bounds, bounds_host, sizeof(float) * 12);
  const T* outp = (const T*)t->bufs[P.out_buf];
  launch_p_losses<T>(x0, noise, t->x_t, outp, P.dpad, t64, h->sched_dev[S_SQRT_AC], h->sched_dev[S_SQRT_1MAC],
                     h->sched_dev[S_SQRT_RECIP], h->sched_dev[S_SQRT_RECIPM1], h->sched_dev[S_LW], h->sched_dev[S_AC], a,
                     losses, t->loss_parts, B, s);
  launch_loss_dict_mean(t->loss_parts, loss_dict, B, s);
  if (!grads) return 0;
  launch_p_losses_bwd<T>(x0, noise, t->x_t, outp, P.dpad, t64, h->sched_dev[S_SQRT_AC], h->sched_dev[S_SQRT_1MAC],
                         h->sched_dev[S_SQRT_RECIP], h->sched_dev[S_SQRT_RECIPM1], h->sched_dev[S_LW], h->sched_dev[S_AC], a,
                         (T*)t->gbufs[P.out_buf], P.dpad, P.dpad, B, grad_scale, s);

  cudaEventRecord(t->ev[3], s);
  // ---- 4. backward through the step program
  CK(cudaMemsetAsync(t->dwarena, 0, t->dw_total * 4, s));
  CK(cudaMemsetAsync(t->dvarena, 0, t->v_total * 4, s));
  CK(cudaMemsetAsync(grads, 0, (size_t)t->flat_n * 4, s));
  CK(cudaMemsetAsync(t->dctx_film, 0, (size_t)ctx_rows * ncb * 2 * C * 4, s));
  // which column ranges of every gradient buffer have been written so far: the first writer overwrites, later ones
  // accumulate (buffers with several consumers: residual stream, U-Net skips, column-sliced MLP buffers)
  std::vector<std::vector<std::pair<int, int>>> seen(P.buf_width.size());
  auto covered = [&](int buf, int col, int width) {      // is [col, col + width) inside the union of the written ranges?
    int cur = col;
    bool moved = true;
    while (cur < col + width && moved) {
      moved = false;
      for (auto& iv : seen[buf])
        if (iv.first <= cur && cur < iv.second) { cur = iv.second; moved = true; break; }
    }
    return cur >= col + width;
  };
  seen[P.out_buf].push_back({0, P.buf_width[P.out_buf]});
  auto first_write_w = [&](int buf, int col, int width) {      // returns the accumulate flag and marks the range
    if (covered(buf, col, width)) return 1;
    seen[buf].push_back({col, col + width});
    return 0;
  };
  auto first_write = [&](int buf, int col) { return first_write_w(buf, col, col == 0 ? P.buf_width[buf] : 0); };
  // finalisation bookkeeping (host side, at enqueue time): which named gradients are complete in stream order
  std::map<std::string, bool> pending;
  for (auto& kv : t->flat_off) pending[kv.first] = true;
  std::vector<char> bucket_done(t->bucket_events.size(), 0);
  auto advance_buckets = [&]() {      // a bucket is final once no pending gradient intersects its flat range
    for (size_t k = 0; k < t->bucket_events.size(); ++k) {
      if (bucket_done[k]) continue;
      const int64_t lo = t->bucket_bounds[k], hi = t->bucket_bounds[k + 1];
      bool final_ = true;
      for (auto& kv : pending) {
        if (!kv.second) continue;
        const int64_t a0 = t->flat_off.at(kv.first), a1 = a0 + h->plan.expected.at(kv.first);
        if (a0 < hi && a1 > lo) { final_ = false; break; }
      }
      if (final_) {
        cudaEventRecord(t->bucket_events[k], s);
        bucket_done[k] = 1;
      }
    }
  };
  auto unpack_wmat = [&](int w) {
    const WRecipe& r = P.wmats[w];
    for (const WPiece& pc : r.pieces) {
      launch_unpack_piece_grad(t->dwarena + t->dw_off[w] + (size_t)pc.row_off * r.K + pc.col_off, r.K, F(pc.name), pc.rows,
                               pc.cols, G(pc.name), r.ws ? 1 : 0, s);
      pending[pc.name] = false;
    }
  };
  auto unpack_vec = [&](int v) -> int {
    if (v < 0) return 0;
    for (const VPiece& pc : P.vecs[v].pieces) {
      CK(cudaMemcpyAsync(G(pc.name), t->dvarena + t->v_off[v] + pc.off, (size_t)pc.n * 4, cudaMemcpyDeviceToDevice, s));
      pending[pc.name] = false;
    }
    return 0;
  };
  bool dst_started = false, dctx_started = false;
  bool stT_ready = false, crossT_ready = false;
  auto time_block_bwd = [&](int i) {      // FiLM projection of time block i: dW, db, and its share of d(SiLU(temb))
    const float* df = t->dfilm + (size_t)i * 2 * C;
    if (film_tc) {
      const int W4 = 4 * C, NF = ntb * 2 * C;
      if (!stT_ready) {
        launch_transpose_pad<bf16>(t->st_bf, W4, t->stT, t->Bp, B, t->Bp, W4, nullptr, s);
        stT_ready = true;
      }
      dim3 grid((t->Bp + 31) / 32, (2 * C + 31) / 32), block(32, 8);
      k_dfilm_prepare<<<grid, block, 0, s>>>(df, NF, t->dfilm_bf + (size_t)i * 2 * C, NF, t->trF + (size_t)i * 2 * C * t->Bp, t->Bp,
                                             B, 2 * C, G(P.time_blocks[i] + ".mlp.1.bias"));
      const int tiles = tc_plan_tiles(t->tc_dwf[i], 2 * C), kblocks = t->Bp / 64;
      int ksplit = std::max(1, std::min(148 / std::max(1, tiles), kblocks));
      const int kb_per = (kblocks + ksplit - 1) / ksplit;
      ksplit = (kblocks + kb_per - 1) / kb_per;
      tc_plan_set_atomic_out(t->tc_dwf[i], G(P.time_blocks[i] + ".mlp.1.weight"), W4, ksplit);
      launch_gemm_tc(t->tc_dwf[i], 2 * C, s);
      pending[P.time_blocks[i] + ".mlp.1.weight"] = false;
      pending[P.time_blocks[i] + ".mlp.1.bias"] = false;
      return;
    }
    launch_gemm_tn<float, float>(df, ntb * 2 * C, t->st, 4 * C, G(P.time_blocks[i] + ".mlp.1.weight"), 4 * C, B, 2 * C, 4 * C, s);
    launch_colsum<float>(df, ntb * 2 * C, G(P.time_blocks[i] + ".mlp.1.bias"), B, 2 * C, s);
    launch_gemm_nn<float, float, float>(df, ntb * 2 * C, F(P.time_blocks[i] + ".mlp.1.weight"), 4 * C, t->dst, 4 * C, B, 4 * C,
                                        2 * C, dst_started ? 1 : 0, s);
    dst_started = true;
    pending[P.time_blocks[i] + ".mlp.1.weight"] = false;
    pending[P.time_blocks[i] + ".mlp.1.bias"] = false;
  };
  auto ctx_block_bwd = [&](int i) {
    const float* df = t->dctx_film + (size_t)i * 2 * C;
    launch_gemm_tn<float, float>(df, ncb * 2 * C, t->ctx_act, E, G(P.ctx_blocks[i] + ".mlp.1.weight"), E, ctx_rows, 2 * C, E, s);
    launch_colsum<float>(df, ncb * 2 * C, G(P.ctx_blocks[i] + ".mlp.1.bias"), ctx_rows, 2 * C, s);
    if (dcontext) {
      launch_gemm_nn<float, float, float>(df, ncb * 2 * C, F(P.ctx_blocks[i] + ".mlp.1.weight"), E, t->dctx_act, E, ctx_rows, E,
                                          2 * C, dctx_started ? 1 : 0, s);
      dctx_started = true;
    }
    pending[P.ctx_blocks[i] + ".mlp.1.weight"] = false;
    pending[P.ctx_blocks[i] + ".mlp.1.bias"] = false;
  };
  for (int idx = int(P.ops.size()) - 1; idx >= 0; --idx) {
    const Op& o = P.ops[idx];
    if (o.kind == OP_PACK) continue;
    if (!covered(o.out, o.out_col, o.N))
      return fail(DS_ERR_STATE, "op '%s': output gradient was never produced", o.name.c_str());
    switch (o.kind) {
      case OP_GEMM: {
        const T* gD = gptr(o.out, o.out_col);
        const int ldg = ld(o.out), K = P.wmats[o.w].K;
        const T* W = (const T*)(t->warena + t->w_off[o.w]);
        float* dW = t->dwarena + t->dw_off[o.w];
        const Slice* ins[2] = {&o.in0, &o.in1};
        int koff = 0;
        bool bias_done = false, tra_ready = false;
        for (int k2 = 0; k2 < 2; ++k2) {
          const Slice& in = *ins[k2];
          if (in.buf < 0) continue;
          if (t->use_tc && t->tc_dw[k2][idx]) {
            if (!tra_ready) {      // dY^T once per op; its column sums are the bias gradient
              tra_ready = true;
              launch_transpose_pad<bf16>((const bf16*)gD, ldg, t->trA, t->rows_cap, M, t->rows_cap, o.N,
                                         o.b >= 0 ? t->dvarena + t->v_off[o.b] : nullptr, s);
              bias_done = o.b >= 0;
            }
            launch_transpose_pad<bf16>((const bf16*)ptr(in.buf, in.col), ld(in.buf), t->trB, t->rows_cap, M, t->rows_cap, in.k, nullptr, s);
            int e = launch_gemm_tc(t->tc_dw[k2][idx], o.N, s);
            if (e) return fail(DS_ERR_CUDA, "train: dW GEMM '%s' failed: %s", o.name.c_str(), cudaGetErrorString((cudaError_t)e));
          } else {
            launch_gemm_tn<T, T>(gD, ldg, ptr(in.buf, in.col), ld(in.buf), dW + koff, K, M, o.N, in.k, s);
          }
          if (in.buf != t->pack_buf) {
            const int acc = first_write_w(in.buf, in.col, in.k);
            if (t->use_tc && t->tc_dx[k2][idx]) {
              tc_plan_set_residual(t->tc_dx[k2][idx], acc ? (const void*)gptr(in.buf, in.col) : nullptr);
              int e = launch_gemm_tc(t->tc_dx[k2][idx], M, s);
              if (e) return fail(DS_ERR_CUDA, "train: dX GEMM '%s' failed: %s", o.name.c_str(), cudaGetErrorString((cudaError_t)e));
            } else {
              launch_gemm_nn<T, T, T>(gD, ldg, W + koff, K, gptr(in.buf, in.col), ld(in.buf), M, in.k, o.N, acc, s);
            }
          }
          koff += in.k;
        }
        if (o.b >= 0 && !bias_done) launch_colsum<T>(gD, ldg, t->dvarena + t->v_off[o.b], M, o.N, s);
        if (o.res >= 0) launch_add_block<T>(gD, ldg, gptr(o.res, 0), ld(o.res), M, o.N, first_write(o.res, 0), s);
        unpack_wmat(o.w);
        if (unpack_vec(o.b)) return DS_ERR_CUDA;
        break;
      }
      case OP_ACT:
        first_write_w(o.in0.buf, o.in0.col, o.N);
        launch_act_bwd<T>(ptr(o.in0.buf, o.in0.col), ld(o.in0.buf), gptr(o.out, o.out_col), ld(o.out),
                          gptr(o.in0.buf, o.in0.col), ld(o.in0.buf), M, o.N, o.act, s);
        break;
      case OP_GN: {
        FilmRef f = film_of(o);
        float* dfilm = nullptr;
        int64_t dstride = 0;
        if (o.film == 1) { dfilm = t->dfilm + (size_t)o.film_blk * 2 * C; dstride = (int64_t)ntb * 2 * C; }
        else if (o.film == 2) { dfilm = t->dctx_film + (size_t)o.film_blk * 2 * C; dstride = (int64_t)ncb * 2 * C; }
        first_write(o.in0.buf, 0);
        const int racc = o.res >= 0 ? first_write(o.res, 0) : 0;
        launch_gn_bwd<T>(ptr(o.in0.buf, 0), ld(o.in0.buf), gptr(o.out, 0), ld(o.out), gptr(o.in0.buf, 0), ld(o.in0.buf),
                         gptr(o.res, 0), ld(o.res), racc, t->varena + t->v_off[o.gamma], t->varena + t->v_off[o.beta], f,
                         t->dvarena + t->v_off[o.gamma], t->dvarena + t->v_off[o.beta], dfilm, dstride, B, n_obj, C, 8, s);
        if (unpack_vec(o.gamma) || unpack_vec(o.beta)) return DS_ERR_CUDA;
        if (o.film == 1) time_block_bwd(o.film_blk);
        else if (o.film == 2) ctx_block_bwd(o.film_blk);
        break;
      }
      case OP_LN: {
        const int xacc = first_write(o.in0.buf, 0);
        const int racc = o.res >= 0 ? first_write(o.res, 0) : 0;
        launch_ln_bwd<T>(ptr(o.in0.buf, 0), ld(o.in0.buf), gptr(o.out, 0), ld(o.out), gptr(o.in0.buf, 0), ld(o.in0.buf), xacc,
                         gptr(o.res, 0), ld(o.res), racc, t->varena + t->v_off[o.b], t->dvarena + t->v_off[o.b], M, C, s);
        if (unpack_vec(o.b)) return DS_ERR_CUDA;
        break;
      }
      case OP_LINATTN:
        first_write(o.in0.buf, 0);
        launch_linattn_bwd<T>(ptr(o.in0.buf, 0), ld(o.in0.buf), gptr(o.out, 0), ld(o.out), gptr(o.in0.buf, 0), ld(o.in0.buf), B,
                              n_obj, s);
        break;
      case OP_ATTN:
        first_write(o.in0.buf, 0);
        launch_softattn_bwd<T>(ptr(o.in0.buf, 0), ld(o.in0.buf), gptr(o.out, 0), ld(o.out), gptr(o.in0.buf, 0), ld(o.in0.buf), B,
                               n_obj, s);
        break;
      case OP_XATTN: {
        // dq and this layer's d(k | v) [B*L, 256], then d(to_kv.weight) = dkv_l^T x context_cross (final here)
        const int acc = first_write(o.in0.buf, 0);
        T* dkv_l = (T*)t->dkv + (size_t)o.xlayer * 256;
        launch_xattn_bwd<T>(ptr(o.in0.buf, 0), ld(o.in0.buf), gptr(o.out, 0), ld(o.out), (const T*)t->kv + (size_t)o.xlayer * 256,
                            NKV, gptr(o.in0.buf, 0), ld(o.in0.buf), acc, dkv_l, NKV, B, n_obj, XL, s);
        const std::string wn = P.xattn_layers[o.xlayer] + ".fn.fn.to_kv.weight";
        if (t->text_tc) {
          if (!crossT_ready) {
            launch_transpose_pad<bf16>(t->cross_bf, TD, t->crossT, t->x_rows_pad, XR, t->x_rows_pad, TD, nullptr, s);
            crossT_ready = true;
          }
          launch_transpose_pad<bf16>((const bf16*)(void*)dkv_l, NKV, t->trKV, t->x_rows_pad, XR, t->x_rows_pad, 256, nullptr, s);
          tc_plan_set_atomic_out(t->tc_kvdw, G(wn), TD, train_ksplit(tc_plan_tiles(t->tc_kvdw, 256), t->x_rows_pad / 64));
          int e = launch_gemm_tc(t->tc_kvdw, 256, s);
          if (e) return fail(DS_ERR_CUDA, "train: to_kv dW GEMM failed: %s", cudaGetErrorString((cudaError_t)e));
        } else {
          launch_gemm_tn<T, T>(dkv_l, NKV, t->bf16 ? (const T*)(const void*)t->cross_bf : (const T*)(const void*)t->cross, TD,
                               G(wn), TD, XR, 256, TD, s);
        }
        pending[wn] = false;
        break;
      }
      default:
        return fail(DS_ERR_STATE, "op kind %d has no backward", o.kind);
    }
    h->launches++;
    advance_buckets();
  }

  cudaEventRecord(t->ev[4], s);
  // ---- 5. what is left of the conditioning paths: d(SiLU(temb)) from all blocks, the shared time MLP (fp32), d(context)
  if (film_tc) {
    int e = launch_gemm_tc(t->tc_dst, t->Bp, s);      // [B, 19 x 2C] x [19 x 2C, 4C], fp32 accumulation over all blocks
    if (e) return fail(DS_ERR_CUDA, "train: d(time embedding) GEMM failed: %s", cudaGetErrorString((cudaError_t)e));
    k_bf16_to_f32<<<((int64_t)B * 4 * C + 255) / 256, 256, 0, s>>>(t->dst_bf, 4 * C, t->dst, 4 * C, B, 4 * C);
  }
  k_mul_actgrad<<<((int64_t)B * 4 * C + 255) / 256, 256, 0, s>>>(t->dst, t->temb, t->dtemb, (int64_t)B * 4 * C, ACT_SILU);
  launch_gemm_tn<float, float>(t->dtemb, 4 * C, t->h1, 4 * C, G("time_mlp.3.weight"), 4 * C, B, 4 * C, 4 * C, s);
  launch_colsum<float>(t->dtemb, 4 * C, G("time_mlp.3.bias"), B, 4 * C, s);
  launch_gemm_nn<float, float, float>(t->dtemb, 4 * C, F("time_mlp.3.weight"), 4 * C, t->dh1, 4 * C, B, 4 * C, 4 * C, 0, s);
  k_mul_actgrad<<<((int64_t)B * 4 * C + 255) / 256, 256, 0, s>>>(t->dh1, t->z1, t->dst, (int64_t)B * 4 * C, ACT_GELU);      // dst := dz1
  launch_gemm_tn<float, float>(t->dst, 4 * C, t->emb, C, G("time_mlp.1.weight"), C, B, 4 * C, C, s);
  launch_colsum<float>(t->dst, 4 * C, G("time_mlp.1.bias"), B, 4 * C, s);
  for (const char* n : {"time_mlp.1.weight", "time_mlp.1.bias", "time_mlp.3.weight", "time_mlp.3.bias"}) pending[n] = false;
  if (dcontext)
    k_mul_actgrad<<<((int64_t)ctx_rows * E + 255) / 256, 256, 0, s>>>(t->dctx_act, context, dcontext, (int64_t)ctx_rows * E, ACT_SILU);
  if (text && t->dcross) {      // d(context_cross) = sum over layers of dkv_l x W_kv,l: one GEMM with K = NKV
    if (t->text_tc) {
      int e = launch_gemm_tc(t->tc_dcross, XR, s);
      if (e) return fail(DS_ERR_CUDA, "train: d(context_cross) GEMM failed: %s", cudaGetErrorString((cudaError_t)e));
    } else {
      launch_gemm_nn<T, T, T>((const T*)t->dkv, NKV, (const T*)t->kvw, TD, t->bf16 ? (T*)(void*)t->dcross_bf : (T*)(void*)t->dcross,
                              TD, XR, TD, NKV, 0, s);
    }
    if (t->bf16) k_bf16_to_f32<<<((int64_t)XR * TD + 255) / 256, 256, 0, s>>>(t->dcross_bf, TD, t->dcross, TD, XR, TD);
    h->launches++;
  }
  cudaEventRecord(t->ev[5], s);
  // ---- 6. every named gradient is final: release the remaining buckets
  for (auto& kv : pending)
    if (kv.second) return fail(DS_ERR_STATE, "gradient of '%s' was never produced", kv.first.c_str());
  advance_buckets();
  cudaEventRecord(t->ev[6], s);
  t->ev_valid = true;
  CK(cudaGetLastError());
  return 0;
}

extern "C" int64_t ds_train_param_count(ds_handle* h) {
  if (!h) return 0;
  int64_t n = 0;
  for (const std::string& s : h->plan.expected_order) n += h->plan.expected[s];
  return n;
}

extern "C" int ds_train_step(ds_handle* h, const float* flat_params_dev, const float* x0_dev, const int64_t* t_dev,
                             const float* noise_dev, const float* context_dev, int32_t ctx_batch, int32_t ctx_shared,
                             int32_t loss_separate, int32_t loss_iou, const float* bounds_host, float grad_scale,
                             float* losses_dev, float* loss_dict_dev, float* flat_grads_dev, float* dcontext_dev,
                             int32_t batch, void* stream) {
  if (!h || !flat_params_dev || !x0_dev || !t_dev || !noise_dev || !context_dev || !losses_dev || !loss_dict_dev)
    return fail(DS_ERR_INVALID, "null argument");
  if (h->T == 0) return fail(DS_ERR_STATE, "ds_set_schedule() has not been called");
  if (loss_iou && !bounds_host) return fail(DS_ERR_INVALID, "loss_iou needs bounds");
  if (batch <= 0 || (!ctx_shared && ctx_batch != batch)) return fail(DS_ERR_INVALID, "bad batch / context batch");
  if (h->cfg.num_objects > 32) return fail(DS_ERR_INVALID, "native training supports up to 32 objects per scene");
  CK(cudaSetDevice(h->cfg.device));
  int rc = train_init(h);
  if (rc) return rc;
  const int ctx_rows = ctx_shared ? h->cfg.num_objects : ctx_batch * h->cfg.num_objects;
  if ((rc = train_capacity(h, batch, ctx_rows))) return rc;
  if (h->cfg.text_condition) {
    if (!h->train->cross) return fail(DS_ERR_STATE, "text network: ds_train_set_context_cross() has not been called");
    if (h->train->cross_batch != batch)
      return fail(DS_ERR_STATE, "context_cross was set for batch %d, call uses batch %d", h->train->cross_batch, batch);
    if ((rc = train_text_capacity(h, batch, h->train->cross_L))) return rc;
  }
  cudaStream_t s = (cudaStream_t)stream;
  if (h->train->bf16)
    return train_step_t<bf16>(h, flat_params_dev, x0_dev, t_dev, noise_dev, context_dev, ctx_batch, ctx_shared, loss_separate,
                              loss_iou, bounds_host, grad_scale, losses_dev, loss_dict_dev, flat_grads_dev, dcontext_dev, batch, s);
  return train_step_t<float>(h, flat_params_dev, x0_dev, t_dev, noise_dev, context_dev, ctx_batch, ctx_shared, loss_separate,
                             loss_iou, bounds_host, grad_scale, losses_dev, loss_dict_dev, flat_grads_dev, dcontext_dev, batch, s);
}

extern "C" int ds_train_set_buckets(ds_handle* h, const int64_t* bounds, int32_t n_buckets, void* const* events) {
  if (!h || n_buckets < 0 || (n_buckets > 0 && (!bounds || !events))) return fail(DS_ERR_INVALID, "bad argument to ds_train_set_buckets");
  CK(cudaSetDevice(h->cfg.device));
  int rc = train_init(h);
  if (rc) return rc;
  TrainState* t = h->train;
  t->bucket_bounds.assign(bounds, bounds + (n_buckets > 0 ? n_buckets + 1 : 0));
  t->bucket_events.clear();
  for (int i = 0; i < n_buckets; ++i) t->bucket_events.push_back((cudaEvent_t)events[i]);
  if (n_buckets > 0 && (t->bucket_bounds.front() != 0 || t->bucket_bounds.back() != t->flat_n))
    return fail(DS_ERR_INVALID, "bucket bounds must run from 0 to ds_train_param_count()");
  return 0;
}

extern "C" int ds_train_set_context_cross(ds_handle* h, const float* cross_dev, int32_t batch, int32_t L, float* dcross_dev) {
  if (!h) return fail(DS_ERR_INVALID, "null handle");
  if (!h->cfg.text_condition) return fail(DS_ERR_INVALID, "configuration has no text condition");
  if (!cross_dev) {
    if (h->train) {
      h->train->cross = nullptr;
      h->train->dcross = nullptr;
      h->train->cross_batch = h->train->cross_L = 0;
    }
    return 0;
  }
  if (batch <= 0 || L <= 0 || L > 512) return fail(DS_ERR_INVALID, "bad context_cross shape (batch %d, L %d)", batch, L);
  CK(cudaSetDevice(h->cfg.device));
  int rc = train_init(h);
  if (rc) return rc;
  TrainState* t = h->train;
  t->cross = cross_dev;
  t->dcross = dcross_dev;
  t->cross_batch = batch;
  t->cross_L = L;
  return 0;
}

extern "C" int ds_train_phase_ms(ds_handle* h, float* out6) {
  if (!h || !out6 || !h->train || !h->train->ev_valid) return fail(DS_ERR_STATE, "no completed training step with gradients");
  CK(cudaEventSynchronize(h->train->ev[6]));
  for (int i = 0; i < 6; ++i) CK(cudaEventElapsedTime(out6 + i, h->train->ev[i], h->train->ev[i + 1]));
  return 0;
}

extern "C" int ds_sumsq(const float* g_dev, int64_t n, float* out_dev, void* stream) {
  if (!g_dev || !out_dev || n < 0) return fail(DS_ERR_INVALID, "bad argument to ds_sumsq");
  launch_sumsq(g_dev, n, out_dev, (cudaStream_t)stream);
  CK(cudaGetLastError());
  return 0;
}

extern "C" int ds_adam_step(float* params_dev, const float* grads_dev, float* exp_avg_dev, float* exp_avg_sq_dev, int64_t n,
                            float lr, float beta1, float beta2, float eps, int32_t step, const float* sumsq_dev,
                            float max_norm, void* stream) {
  if (!params_dev || !grads_dev || !exp_avg_dev || !exp_avg_sq_dev || n < 0 || step < 1)
    return fail(DS_ERR_INVALID, "bad argument to ds_adam_step");
  launch_adam(params_dev, grads_dev, exp_avg_dev, exp_avg_sq_dev, n, lr, beta1, beta2, eps, step, sumsq_dev, max_norm,
              (cudaStream_t)stream);
  CK(cudaGetLastError());
  return 0;
}
