// Engine: owns packed weights, FiLM tables, activation buffers and the step program; implements the
// C ABI of include/diffuscene_b200.h.  There is no CPU compute path in this file: every op is a
// kernel launch from kernels.cuh, and ds_create() fails without a device.
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <string.h>

#include <algorithm>
#include <map>
#include <string>
#include <vector>

#include "kernels.cuh"
#include "plan.h"

#include "engine_internal.h"

static thread_local char g_err[1024] = "";
int fail(int code, const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof g_err, fmt, ap);
  va_end(ap);
  return code;
}
void drop_graph(ds_handle* h) {
  if (h->gexec) cudaGraphExecDestroy(h->gexec);
  h->gexec = nullptr;
  h->gkey = ds_handle::GraphKey();
  h->plan_gen++;
}

static int round_up(int a, int b) { return (a + b - 1) / b * b; }

// ------------------------------------------------------------------------------------------------
// op execution
// ------------------------------------------------------------------------------------------------
static FilmRef film_ref(ds_handle* h, const Op& o) {
  const Plan& P = h->plan;
  const int C = P.C;
  FilmRef f;
  f.base = nullptr; f.mode = FILM_NONE; f.row_stride = 0; f.t = h->t_dev;
  if (o.film == 1) {
    f.base = h->time_table + (size_t)o.film_blk * 2 * C;
    f.mode = FILM_TIME;
    f.row_stride = (int64_t)P.time_blocks.size() * 2 * C;
  } else if (o.film == 2) {
    f.base = h->ctx_table ? h->ctx_table + (size_t)o.film_blk * 2 * C : nullptr;
    f.mode = h->ctx_shared ? FILM_OBJECT : FILM_TOKEN;
    f.row_stride = (int64_t)P.ctx_blocks.size() * 2 * C;
  }
  return f;
}

template <typename T>
static int run_op(ds_handle* h, int idx, int n_scenes, cudaStream_t s) {
  const Plan& P = h->plan;
  const Op& o = P.ops[idx];
  const int n_obj = h->cfg.num_objects, M = n_scenes * n_obj, C = P.C;
  auto ptr = [&](int buf, int col) -> T* { return buf < 0 ? nullptr : (T*)h->bufs[buf] + col; };
  auto ld = [&](int buf) { return buf < 0 ? 0 : P.buf_width[buf]; };
  switch (o.kind) {
    case OP_PACK:
      return DS_ERR_STATE;   // handled by the caller (needs the x pointer)
    case OP_LN_QKV_ATTN: {
      if (!h->use_tc || !h->atp[idx]) return fail(DS_ERR_STATE, "fused attention op without the tcgen05 backend");
      int e = launch_ln_qkv_attn(h->atp[idx], M, s);
      if (e) return fail(DS_ERR_CUDA, "fused LayerNorm + to_qkv + attention launch '%s' failed: %s", o.name.c_str(),
                         cudaGetErrorString((cudaError_t)e));
      break;
    }
    case OP_GEMM_LN: {
      if (!h->use_tc || !h->lnp[idx]) return fail(DS_ERR_STATE, "fused LayerNorm op without the tcgen05 backend");
      int e = launch_gemm_ln(h->lnp[idx], M, s);
      if (e) return fail(DS_ERR_CUDA, "tcgen05 GEMM+LayerNorm launch '%s' failed: %s", o.name.c_str(),
                         cudaGetErrorString((cudaError_t)e));
      break;
    }
    case OP_GEMM_GN:
      if (!h->use_tc) return fail(DS_ERR_STATE, "fused GroupNorm op without the tcgen05 backend");
      // fallthrough
    case OP_GEMM: {
      if (h->use_tc) {
        if (o.kind == OP_GEMM_GN) tc_plan_set_uniform_t(h->tc[idx], h->t_uniform);
        int e = launch_gemm_tc(h->tc[idx], M, s);
        if (e) return fail(DS_ERR_CUDA, "tcgen05 GEMM launch '%s' failed: %s", o.name.c_str(),
                           cudaGetErrorString((cudaError_t)e));
      } else {
        GemmArgs g;
        memset(&g, 0, sizeof g);
        g.a0 = ptr(o.in0.buf, o.in0.col); g.lda0 = ld(o.in0.buf); g.k0 = o.in0.k;
        g.a1 = ptr(o.in1.buf, o.in1.col); g.lda1 = ld(o.in1.buf); g.k1 = o.in1.buf >= 0 ? o.in1.k : 0;
        g.w = h->warena + h->w_off[o.w]; g.ldw = P.wmats[o.w].K;
        g.bias = o.b >= 0 ? h->varena + h->v_off[o.b] : nullptr;
        g.d = ptr(o.out, o.out_col); g.ldd = ld(o.out);
        g.res = ptr(o.res, 0); g.ldres = ld(o.res);
        g.M = M; g.N = o.N; g.act = o.act;
        launch_gemm_simt<T>(g, !h->bf16_mode, s);
      }
      break;
    }
    case OP_GN: {
      FilmRef f = film_ref(h, o);
      launch_groupnorm<T>(ptr(o.in0.buf, 0), ld(o.in0.buf), ptr(o.out, 0), ld(o.out), h->varena + h->v_off[o.gamma],
                          h->varena + h->v_off[o.beta], f, ptr(o.res, 0), ld(o.res), n_scenes, n_obj, C, 8, s);
      break;
    }
    case OP_LN:
      launch_layernorm<T>(ptr(o.in0.buf, 0), ld(o.in0.buf), ptr(o.out, 0), ld(o.out), h->varena + h->v_off[o.b],
                          ptr(o.res, 0), ld(o.res), M, C, s);
      break;
    case OP_LINATTN:
      launch_linattn<T>(ptr(o.in0.buf, 0), ld(o.in0.buf), ptr(o.out, 0), ld(o.out), n_scenes, n_obj, s);
      break;
    case OP_ATTN:
      launch_softattn<T>(ptr(o.in0.buf, 0), ld(o.in0.buf), ptr(o.out, 0), ld(o.out), n_scenes, n_obj, s);
      break;
    case OP_XATTN:
      launch_xattn_apply<T>(ptr(o.in0.buf, 0), ld(o.in0.buf), h->xctx + (size_t)o.xlayer * h->xctx_batch * 4096,
                            ptr(o.out, 0), ld(o.out), n_scenes, n_obj, s);
      break;
  }
  h->launches++;
  return 0;
}

// all ops of one denoiser forward on x [n_scenes, N, d] fp32 (device); result in plan.out_buf
template <typename T>
static int run_forward_t(ds_handle* h, const float* x, int n_scenes, cudaStream_t s) {
  const Plan& P = h->plan;
  const int M = n_scenes * h->cfg.num_objects;
  for (size_t i = 0; i < P.ops.size(); ++i) {
    if (P.ops[i].kind == OP_PACK) {
      launch_pack_input<T>(x, (T*)h->bufs[P.ops[i].out], P.kin_pad, M, P.d, s);
      h->launches++;
    } else {
      int rc = run_op<T>(h, int(i), n_scenes, s);
      if (rc) return rc;
    }
  }
  return 0;
}
static int run_forward(ds_handle* h, const float* x, int n_scenes, cudaStream_t s) {
  return h->bf16_mode ? run_forward_t<bf16>(h, x, n_scenes, s) : run_forward_t<float>(h, x, n_scenes, s);
}

// ------------------------------------------------------------------------------------------------
// capacity / buffers
// ------------------------------------------------------------------------------------------------
static void free_buffers(ds_handle* h) {
  drop_graph(h);
  for (void* p : h->bufs) cudaFree(p);
  h->bufs.clear();
  for (auto* p : h->tc) if (p) tc_plan_destroy(p);
  h->tc.clear();
  for (auto* p : h->lnp) if (p) ln_plan_destroy(p);
  h->lnp.clear();
  for (auto* p : h->atp) if (p) attn_qkv_plan_destroy(p);
  h->atp.clear();
  cudaFree(h->t_dev); h->t_dev = nullptr;
  cudaFree(h->x_state); h->x_state = nullptr;
  cudaFree(h->x_tmp); h->x_tmp = nullptr;
  cudaFree(h->t64_tmp); h->t64_tmp = nullptr;
  cudaFree(h->loss_parts); h->loss_parts = nullptr;
  h->cap_scenes = 0;
}

// which kernel variant a GEMM op runs on (0: row-major tcgen05 kernel, 2: channels-on-lanes GroupNorm, 3: ... plain)
static int gemm_variant(const ds_handle* h, const Op& o) {
  if (o.kind == OP_GEMM_GN) return h->gnt ? 2 : 1;
  // plain GEMMs: the channels-on-lanes kernel wins where the epilogue dominates (K <= 128: to_out) or where the
  // row-major kernel would fall back to 128-wide tiles (N % 256 != 0: to_qkv); the MMA-bound shapes keep the
  // row-major kernel, whose 128 x 256 tiles feed the tensor pipe better than 128 x 192 (measured, profiles/)
  if (o.kind == OP_GEMM && h->gnt_plain && tc_gnt_plain_supported(h->cfg.num_objects, o.N)) {
    const int K = o.in0.k + (o.in1.buf >= 0 ? o.in1.k : 0);
    if (K <= 128 || o.N % 256 != 0) return 3;
  }
  return 0;
}

static int ensure_capacity(ds_handle* h, int n_scenes) {
  if (n_scenes <= 0) return fail(DS_ERR_INVALID, "batch must be positive");
  if (!h->committed) return fail(DS_ERR_STATE, "ds_commit_weights() has not been called");
  if (n_scenes <= h->cap_scenes) return 0;
  free_buffers(h);
  const Plan& P = h->plan;
  const int n_obj = h->cfg.num_objects;
  h->rows_cap = round_up(n_scenes * n_obj, 128);
  h->bufs.resize(P.buf_width.size(), nullptr);
  for (size_t i = 0; i < P.buf_width.size(); ++i) {
    size_t bytes = (size_t)h->rows_cap * P.buf_width[i] * h->esz;
    CK(cudaMalloc(&h->bufs[i], bytes));
    CK(cudaMemset(h->bufs[i], 0, bytes));
  }
  CK(cudaMalloc(&h->t_dev, sizeof(int) * n_scenes));
  CK(cudaMemset(h->t_dev, 0, sizeof(int) * n_scenes));
  size_t xs = (size_t)n_scenes * n_obj * P.d * sizeof(float);
  CK(cudaMalloc(&h->x_state, xs));
  CK(cudaMalloc(&h->x_tmp, xs));
  CK(cudaMalloc(&h->t64_tmp, sizeof(int64_t) * n_scenes));
  CK(cudaMalloc(&h->loss_parts, sizeof(float) * 9 * n_scenes));
  h->tc.assign(P.ops.size(), nullptr);
  h->lnp.assign(P.ops.size(), nullptr);
  h->atp.assign(P.ops.size(), nullptr);
  if (h->use_tc) {
    for (size_t i = 0; i < P.ops.size(); ++i) {
      const Op& o = P.ops[i];
      if (o.kind == OP_LN_QKV_ATTN) {
        char err[256] = "";
        h->atp[i] = attn_qkv_plan_create((bf16*)h->bufs[o.in0.buf] + o.in0.col, P.buf_width[o.in0.buf], h->warena + h->w_off[o.w],
                                         P.wmats[o.w].K, h->attn_cs + (size_t)o.w * 384, (bf16*)h->bufs[o.out], P.buf_width[o.out],
                                         n_obj, P.wmats[o.w].K, h->rows_cap, err, sizeof err);
        if (!h->atp[i]) return fail(DS_ERR_CUDA, "fused attention plan for op '%s' failed: %s", o.name.c_str(), err);
        continue;
      }
      if (o.kind != OP_GEMM && o.kind != OP_GEMM_GN && o.kind != OP_GEMM_LN) continue;
      auto ptr = [&](int buf, int col) -> bf16* { return buf < 0 ? nullptr : (bf16*)h->bufs[buf] + col; };
      GemmArgs g;
      memset(&g, 0, sizeof g);
      if (o.kind == OP_GEMM_LN) {
        g.a0 = ptr(o.in0.buf, o.in0.col); g.lda0 = P.buf_width[o.in0.buf]; g.k0 = o.in0.k;
        g.w = h->warena + h->w_off[o.w]; g.ldw = P.wmats[o.w].K;
        g.bias = o.b >= 0 ? h->varena + h->v_off[o.b] : nullptr;
        g.gamma = h->varena + h->v_off[o.gamma];
        g.d = ptr(o.out, o.out_col); g.ldd = P.buf_width[o.out];
        g.res = ptr(o.res, 0); g.ldres = o.res >= 0 ? P.buf_width[o.res] : 0;
        g.M = h->rows_cap; g.N = o.N;
        char err[256] = "";
        h->lnp[i] = ln_plan_create(g, h->rows_cap, err, sizeof err);
        if (!h->lnp[i]) return fail(DS_ERR_CUDA, "tcgen05 GEMM+LayerNorm plan for op '%s' failed: %s", o.name.c_str(), err);
        continue;
      }
      g.gn = gemm_variant(h, o);
      g.n_obj = n_obj;
      if (o.kind == OP_GEMM_GN) {
        g.film_C = P.C;
        g.gamma = h->varena + h->v_off[o.gamma];
        g.beta = h->varena + h->v_off[o.beta];
        g.film = film_ref(h, o);
      }
      g.a0 = ptr(o.in0.buf, o.in0.col); g.lda0 = P.buf_width[o.in0.buf]; g.k0 = o.in0.k;
      g.a1 = ptr(o.in1.buf, o.in1.col); g.lda1 = o.in1.buf >= 0 ? P.buf_width[o.in1.buf] : 0;
      g.k1 = o.in1.buf >= 0 ? o.in1.k : 0;
      g.w = h->warena + h->w_off[o.w]; g.ldw = P.wmats[o.w].K;
      g.bias = o.b >= 0 ? h->varena + h->v_off[o.b] : nullptr;
      g.d = ptr(o.out, o.out_col); g.ldd = P.buf_width[o.out];
      g.res = ptr(o.res, 0); g.ldres = o.res >= 0 ? P.buf_width[o.res] : 0;
      g.M = h->rows_cap; g.N = o.N; g.act = o.act;
      char err[256] = "";
      h->tc[i] = tc_plan_create(g, h->rows_cap, err, sizeof err);
      if (!h->tc[i]) return fail(DS_ERR_CUDA, "tcgen05 plan for op '%s' failed: %s", o.name.c_str(), err);
    }
  }
  h->cap_scenes = n_scenes;
  return 0;
}

// ------------------------------------------------------------------------------------------------
// weights
// ------------------------------------------------------------------------------------------------
static const std::vector<float>* find_w(ds_handle* h, const std::string& name, int64_t numel, int* rc) {
  auto it = h->host_w.find(name);
  if (it == h->host_w.end()) {
    *rc = fail(DS_ERR_MISSING_WEIGHT, "weight '%s' was never loaded", name.c_str());
    return nullptr;
  }
  if ((int64_t)it->second.size() != numel) {
    *rc = fail(DS_ERR_INVALID, "weight '%s' has %lld elements, expected %lld", name.c_str(),
               (long long)it->second.size(), (long long)numel);
    return nullptr;
  }
  return &it->second;
}

static void to_bf16_host(const float* src, uint16_t* dst, size_t n) {
  for (size_t i = 0; i < n; ++i) {
    uint32_t u;
    memcpy(&u, src + i, 4);
    if ((u & 0x7fffffffu) > 0x7f800000u) { dst[i] = uint16_t((u >> 16) | 0x40); continue; }   // NaN
    uint32_t lsb = (u >> 16) & 1u;
    u += 0x7fffu + lsb;                                                                          // RNE
    dst[i] = uint16_t(u >> 16);
  }
}

static int upload_f32(float** dst, const float* src, size_t n) {
  if (*dst) cudaFree(*dst);
  *dst = nullptr;
  CK(cudaMalloc(dst, n * sizeof(float)));
  CK(cudaMemcpy(*dst, src, n * sizeof(float), cudaMemcpyHostToDevice));
  return 0;
}

static int build_time_table(ds_handle* h) {
  const Plan& P = h->plan;
  const int C = P.C, T = h->cfg.num_timesteps, ntb = int(P.time_blocks.size());
  cudaStream_t s = h->own_stream;
  float *emb = nullptr, *h1 = nullptr, *h2 = nullptr;
  CK(cudaMalloc(&emb, (size_t)T * C * 4));
  CK(cudaMalloc(&h1, (size_t)T * 4 * C * 4));
  CK(cudaMalloc(&h2, (size_t)T * 4 * C * 4));
  if (h->time_table) cudaFree(h->time_table);
  CK(cudaMalloc(&h->time_table, (size_t)T * ntb * 2 * C * 4));
  {      // per-handle frequency vector (handles on different devices never share device memory)
    std::vector<float> hf(C / 2);
    sinusoid_freqs_host(C, hf.data());
    int rc = upload_f32(&h->sin_freq, hf.data(), hf.size());
    if (rc) return rc;
  }
  launch_sinusoid(emb, h->sin_freq, T, C, s);
  GemmArgs g;
  memset(&g, 0, sizeof g);
  g.a0 = emb; g.lda0 = C; g.k0 = C; g.w = h->time_w1; g.ldw = C; g.bias = h->time_b1; g.d = h1; g.ldd = 4 * C;
  g.M = T; g.N = 4 * C; g.act = ACT_GELU;
  launch_gemm_f32(g, s);
  // every consumer applies SiLU first (ResnetBlock.mlp = Sequential(SiLU, Linear), denoise_net.py:181-184)
  g.a0 = h1; g.lda0 = 4 * C; g.k0 = 4 * C; g.w = h->time_w3; g.ldw = 4 * C; g.bias = h->time_b3; g.d = h2;
  g.act = ACT_SILU;
  launch_gemm_f32(g, s);
  g.a0 = h2; g.w = h->time_wall; g.bias = h->time_ball; g.d = h->time_table; g.ldd = ntb * 2 * C; g.N = ntb * 2 * C;
  g.act = ACT_NONE;
  launch_gemm_f32(g, s);
  h->launches += 4;
  CK(cudaStreamSynchronize(s));
  cudaFree(emb); cudaFree(h1); cudaFree(h2);
  return 0;
}

extern "C" int ds_commit_weights(ds_handle* h) {
  if (!h) return fail(DS_ERR_INVALID, "null handle");
  CK(cudaSetDevice(h->cfg.device));
  const Plan& P = h->plan;
  const int C = P.C;
  int rc = 0;
  // ---- packed GEMM weights ----
  size_t total = 0;
  h->w_off.resize(P.wmats.size());
  for (size_t i = 0; i < P.wmats.size(); ++i) {
    h->w_off[i] = total;
    total += ((size_t)P.wmats[i].N * P.wmats[i].K * h->esz + 255) / 256 * 256;
  }
  std::vector<char> host(total, 0);
  std::vector<float> mat;
  std::vector<float> attn_cs_host(P.wmats.size() * 384, 0.f);
  std::vector<char> gnt_w(P.wmats.size(), 0);       // weight matrices consumed by fused GroupNorm ops
  std::vector<char> row_major_w(P.wmats.size(), 0);
  for (const Op& o : P.ops) {
    if (o.kind == OP_GEMM_LN || o.kind == OP_LN_QKV_ATTN) { row_major_w[o.w] = 1; continue; }
    if (o.kind != OP_GEMM && o.kind != OP_GEMM_GN) continue;
    if (gemm_variant(h, o) >= 2) gnt_w[o.w] = 1;
    else row_major_w[o.w] = 1;
  }
  for (size_t i = 0; i < P.wmats.size(); ++i)
    if (gnt_w[i] && row_major_w[i]) return fail(DS_ERR_STATE, "weight matrix %d is shared by both GEMM layouts", int(i));
  for (size_t i = 0; i < P.wmats.size(); ++i) {
    const WRecipe& r = P.wmats[i];
    mat.assign((size_t)r.N * r.K, 0.f);
    for (const WPiece& pc : r.pieces) {
      const std::vector<float>* src = find_w(h, pc.name, (int64_t)pc.rows * pc.cols, &rc);
      if (!src) return rc;
      for (int rr = 0; rr < pc.rows; ++rr) {
        const float* srow = src->data() + (size_t)rr * pc.cols;
        float* drow = mat.data() + (size_t)(pc.row_off + rr) * r.K + pc.col_off;
        if (r.ws) {
          // weight standardisation, fp32 like the reference (denoise_net.py:86-89), eps 1e-5, biased variance
          double mean = 0;
          for (int c = 0; c < pc.cols; ++c) mean += srow[c];
          mean /= pc.cols;
          double var = 0;
          for (int c = 0; c < pc.cols; ++c) var += (srow[c] - mean) * (srow[c] - mean);
          var /= pc.cols;
          const float fm = float(mean), rs = 1.0f / sqrtf(float(var) + 1e-5f);
          for (int c = 0; c < pc.cols; ++c) drow[c] = (srow[c] - fm) * rs;
        } else {
          memcpy(drow, srow, sizeof(float) * pc.cols);
        }
      }
    }
    if (!r.scale_k.empty()) {      // a LayerNorm gain folded into the columns of the following conv (k_ln_qkv_attn)
      const std::vector<float>* gk = find_w(h, r.scale_k, r.K, &rc);
      if (!gk) return rc;
      for (int rr = 0; rr < r.N; ++rr)
        for (int c = 0; c < r.K; ++c) mat[(size_t)rr * r.K + c] *= (*gk)[c];
      if (r.N <= 384 && h->bf16_mode) {
        // column sums of the ROUNDED weights: the kernel subtracts mean * cs from an accumulator built from them
        std::vector<uint16_t> tmp(mat.size());
        to_bf16_host(mat.data(), tmp.data(), mat.size());
        for (int rr = 0; rr < r.N; ++rr) {
          double acc = 0;
          for (int c = 0; c < r.K; ++c) {
            uint32_t u = uint32_t(tmp[(size_t)rr * r.K + c]) << 16;
            float f;
            memcpy(&f, &u, 4);
            acc += f;
          }
          attn_cs_host[i * 384 + rr] = float(acc);
        }
      }
    }
    if (gnt_w[i]) {      // row order the channels-on-lanes kernel expects (see tc_gnt_row)
      std::vector<float> pm(mat.size());
      for (int rr = 0; rr < r.N; ++rr) memcpy(pm.data() + (size_t)rr * r.K, mat.data() + (size_t)tc_gnt_row(rr) * r.K, sizeof(float) * r.K);
      mat.swap(pm);
    }
    if (h->bf16_mode) to_bf16_host(mat.data(), (uint16_t*)(host.data() + h->w_off[i]), mat.size());
    else memcpy(host.data() + h->w_off[i], mat.data(), mat.size() * 4);
  }
  if (h->warena) cudaFree(h->warena);
  h->warena = nullptr;
  CK(cudaMalloc(&h->warena, total));
  CK(cudaMemcpy(h->warena, host.data(), total, cudaMemcpyHostToDevice));
  if ((rc = upload_f32(&h->attn_cs, attn_cs_host.data(), attn_cs_host.size()))) return rc;
  // ---- fp32 vectors ----
  size_t vt = 0;
  h->v_off.resize(P.vecs.size());
  for (size_t i = 0; i < P.vecs.size(); ++i) {
    h->v_off[i] = vt;
    vt += (size_t)round_up(P.vecs[i].n, 64);
  }
  std::vector<float> hv(vt, 0.f);
  for (size_t i = 0; i < P.vecs.size(); ++i)
    for (const VPiece& pc : P.vecs[i].pieces) {
      const std::vector<float>* src = find_w(h, pc.name, pc.n, &rc);
      if (!src) return rc;
      for (int k = 0; k < pc.n; ++k) hv[h->v_off[i] + pc.off + k] += (*src)[k];
    }
  rc = upload_f32(&h->varena, hv.data(), vt);
  if (rc) return rc;
  // ---- time path (fp32) ----
  const std::vector<float>* w;
  if (!(w = find_w(h, "time_mlp.1.weight", (int64_t)4 * C * C, &rc))) return rc;
  if ((rc = upload_f32(&h->time_w1, w->data(), w->size()))) return rc;
  if (!(w = find_w(h, "time_mlp.1.bias", 4 * C, &rc))) return rc;
  if ((rc = upload_f32(&h->time_b1, w->data(), w->size()))) return rc;
  if (!(w = find_w(h, "time_mlp.3.weight", (int64_t)16 * C * C, &rc))) return rc;
  if ((rc = upload_f32(&h->time_w3, w->data(), w->size()))) return rc;
  if (!(w = find_w(h, "time_mlp.3.bias", 4 * C, &rc))) return rc;
  if ((rc = upload_f32(&h->time_b3, w->data(), w->size()))) return rc;
  {
    const int ntb = int(P.time_blocks.size());
    std::vector<float> wall((size_t)ntb * 2 * C * 4 * C), ball((size_t)ntb * 2 * C);
    for (int i = 0; i < ntb; ++i) {
      if (!(w = find_w(h, P.time_blocks[i] + ".mlp.1.weight", (int64_t)2 * C * 4 * C, &rc))) return rc;
      memcpy(wall.data() + (size_t)i * 2 * C * 4 * C, w->data(), w->size() * 4);
      if (!(w = find_w(h, P.time_blocks[i] + ".mlp.1.bias", 2 * C, &rc))) return rc;
      memcpy(ball.data() + (size_t)i * 2 * C, w->data(), w->size() * 4);
    }
    if ((rc = upload_f32(&h->time_wall, wall.data(), wall.size()))) return rc;
    if ((rc = upload_f32(&h->time_ball, ball.data(), ball.size()))) return rc;
  }
  {
    const int ncb = int(P.ctx_blocks.size()), E = h->cfg.cond_dim;
    std::vector<float> wall((size_t)ncb * 2 * C * E), ball((size_t)ncb * 2 * C);
    for (int i = 0; i < ncb; ++i) {
      if (!(w = find_w(h, P.ctx_blocks[i] + ".mlp.1.weight", (int64_t)2 * C * E, &rc))) return rc;
      memcpy(wall.data() + (size_t)i * 2 * C * E, w->data(), w->size() * 4);
      if (!(w = find_w(h, P.ctx_blocks[i] + ".mlp.1.bias", 2 * C, &rc))) return rc;
      memcpy(ball.data() + (size_t)i * 2 * C, w->data(), w->size() * 4);
    }
    if ((rc = upload_f32(&h->ctx_wall, wall.data(), wall.size()))) return rc;
    if ((rc = upload_f32(&h->ctx_ball, ball.data(), ball.size()))) return rc;
  }
  for (float* p : h->kv_w) cudaFree(p);
  h->kv_w.assign(P.xattn_layers.size(), nullptr);
  for (size_t i = 0; i < P.xattn_layers.size(); ++i) {
    if (!(w = find_w(h, P.xattn_layers[i] + ".fn.fn.to_kv.weight", (int64_t)256 * h->cfg.text_dim, &rc))) return rc;
    if ((rc = upload_f32(&h->kv_w[i], w->data(), w->size()))) return rc;
  }
  if ((rc = build_time_table(h))) return rc;
  h->committed = true;
  h->ctx_set = false;      // FiLM projections depend on the weights
  h->xctx_batch = 0;
  // tensor maps point into the old weight arena
  int cap = h->cap_scenes;
  free_buffers(h);
  if (cap > 0) return ensure_capacity(h, cap);
  return 0;
}

// ------------------------------------------------------------------------------------------------
// lifetime
// ------------------------------------------------------------------------------------------------
extern "C" const char* ds_last_error(void) { return g_err; }
extern "C" const char* ds_version(void) { return "diffuscene_b200 0.1 (sm_100a)"; }

extern "C" int ds_create(const ds_config* cfg, ds_handle** out) {
  if (!cfg || !out) return fail(DS_ERR_INVALID, "null argument");
  *out = nullptr;
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(DS_ERR_NO_DEVICE, "no CUDA device: diffuscene_b200 has no CPU fallback");
  }
  if (cfg->device < 0 || cfg->device >= ndev) return fail(DS_ERR_INVALID, "device %d out of range", cfg->device);
  CK(cudaSetDevice(cfg->device));
  cudaDeviceProp prop;
  CK(cudaGetDeviceProperties(&prop, cfg->device));
  if (prop.major != 10)
    return fail(DS_ERR_NO_DEVICE, "device %d is sm_%d%d; this library is built for sm_100a only", cfg->device,
                prop.major, prop.minor);
  ds_handle* h = new ds_handle();
  h->cfg = *cfg;
  if (!build_plan(*cfg, false, &h->plan)) {
    int rc = fail(DS_ERR_INVALID, "%s", h->plan.error.c_str());
    delete h;
    return rc;
  }
  h->bf16_mode = cfg->precision == DS_PREC_BF16;
  h->esz = h->bf16_mode ? 2 : 4;
  if (cfg->gemm_backend == DS_GEMM_TCGEN05 && !h->bf16_mode) {
    delete h;
    return fail(DS_ERR_INVALID, "the tcgen05 backend needs DS_PREC_BF16");
  }
  h->use_tc = h->bf16_mode && cfg->gemm_backend != DS_GEMM_SIMT;
  if (h->use_tc) {
    char err[256] = "";
    if (!tc_runtime_available(err, sizeof err)) {
      delete h;
      return fail(DS_ERR_CUDA, "%s", err);
    }
  }
  // fuse_level 2: the fused conv + GroupNorm ops use the channels-on-lanes tcgen05 kernel where it applies
  h->gnt = h->use_tc && cfg->fuse_level >= 2 && tc_gnt_supported(cfg->num_objects, h->plan.C);
  h->gnt_plain = h->gnt && cfg->fuse_level >= 3;
  cudaError_t e = cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking);
  if (e != cudaSuccess) {
    delete h;
    return fail(DS_ERR_CUDA, "cudaStreamCreate: %s", cudaGetErrorString(e));
  }
  init_pointwise_attrs();
  cudaMalloc(&h->state_dev, sizeof(StepState));
  cudaMemset(h->state_dev, 0, sizeof(StepState));
  *out = h;
  return 0;
}

extern "C" int ds_destroy(ds_handle* h) {
  if (!h) return 0;
  cudaSetDevice(h->cfg.device);
  drop_graph(h);
  if (h->train) train_state_destroy(h->train);
  h->train = nullptr;
  free_buffers(h);
  cudaFree(h->warena); cudaFree(h->varena); cudaFree(h->attn_cs);
  cudaFree(h->time_w1); cudaFree(h->time_b1); cudaFree(h->time_w3); cudaFree(h->time_b3);
  cudaFree(h->time_wall); cudaFree(h->time_ball); cudaFree(h->time_table); cudaFree(h->sin_freq);
  cudaFree(h->ctx_wall); cudaFree(h->ctx_ball); cudaFree(h->ctx_table);
  for (float* p : h->kv_w) cudaFree(p);
  cudaFree(h->xctx);
  for (int i = 0; i < S_COUNT; ++i) cudaFree(h->sched_dev[i]);
  cudaFree(h->coef_dev); cudaFree(h->state_dev);
  if (h->own_stream) cudaStreamDestroy(h->own_stream);
  delete h;
  return 0;
}

extern "C" int ds_load_weight(ds_handle* h, const char* name, const float* host_data, int64_t numel) {
  if (!h || !name || !host_data || numel <= 0) return fail(DS_ERR_INVALID, "bad argument to ds_load_weight");
  auto it = h->plan.expected.find(name);
  if (it == h->plan.expected.end()) return fail(DS_ERR_INVALID, "unexpected weight name '%s'", name);
  if (it->second != numel)
    return fail(DS_ERR_INVALID, "weight '%s': %lld elements given, %lld expected", name, (long long)numel,
                (long long)it->second);
  h->host_w[name].assign(host_data, host_data + numel);
  return 0;
}
extern "C" int ds_expected_weight_count(ds_handle* h) { return h ? int(h->plan.expected_order.size()) : 0; }
extern "C" int ds_expected_weight(ds_handle* h, int index, const char** name, int64_t* numel) {
  if (!h || index < 0 || index >= (int)h->plan.expected_order.size()) return fail(DS_ERR_INVALID, "index out of range");
  const std::string& n = h->plan.expected_order[index];
  if (name) *name = n.c_str();
  if (numel) *numel = h->plan.expected[n];
  return 0;
}

// ------------------------------------------------------------------------------------------------
// schedule / conditioning
// ------------------------------------------------------------------------------------------------
extern "C" int ds_set_schedule(ds_handle* h, const ds_schedule* s) {
  if (!h || !s) return fail(DS_ERR_INVALID, "null argument");
  if (s->T != h->cfg.num_timesteps)
    return fail(DS_ERR_INVALID, "schedule T=%d differs from the configured num_timesteps=%d", s->T,
                h->cfg.num_timesteps);
  if (s->mean_type < 0 || s->mean_type > 2) return fail(DS_ERR_INVALID, "bad mean_type");
  const float* src[9] = {s->sqrt_ac, s->sqrt_1mac, s->sqrt_recip_ac, s->sqrt_recipm1_ac, s->coef1, s->coef2,
                         s->sigma, s->alphas_cumprod, s->loss_weight};
  CK(cudaSetDevice(h->cfg.device));
  for (int i = 0; i < 9; ++i) {
    if (!src[i]) return fail(DS_ERR_INVALID, "schedule array %d is null", i);
    h->sched_host[i].assign(src[i], src[i] + s->T);
  }
  h->sched_host[S_NEG_1MAC].resize(s->T);
  h->sched_host[S_NEG_RECIPM1].resize(s->T);
  h->sched_host[S_ZERO].assign(s->T, 0.f);
  h->sched_host[S_ONE].assign(s->T, 1.f);
  for (int t = 0; t < s->T; ++t) {
    h->sched_host[S_NEG_1MAC][t] = -s->sqrt_1mac[t];
    h->sched_host[S_NEG_RECIPM1][t] = -s->sqrt_recipm1_ac[t];
  }
  for (int i = 0; i < S_COUNT; ++i) {
    int rc = upload_f32(&h->sched_dev[i], h->sched_host[i].data(), s->T);
    if (rc) return rc;
  }
  h->T = s->T;
  h->mean_type = s->mean_type;
  return 0;
}

extern "C" int ds_set_context(ds_handle* h, const float* context_dev, int32_t batch, int32_t shared, void* stream) {
  if (!h || !context_dev) return fail(DS_ERR_INVALID, "null argument");
  if (!h->committed) return fail(DS_ERR_STATE, "ds_commit_weights() first");
  CK(cudaSetDevice(h->cfg.device));
  cudaStream_t s = stream ? (cudaStream_t)stream : h->own_stream;
  const Plan& P = h->plan;
  const int C = P.C, E = h->cfg.cond_dim, ncb = int(P.ctx_blocks.size());
  const int rows = shared ? h->cfg.num_objects : batch * h->cfg.num_objects;
  if (rows <= 0) return fail(DS_ERR_INVALID, "bad context batch");
  if (rows > h->ctx_rows) {
    drop_graph(h);
    cudaFree(h->ctx_table);
    h->ctx_table = nullptr;
    CK(cudaMalloc(&h->ctx_table, (size_t)rows * ncb * 2 * C * 4));
    h->ctx_rows = rows;
  }
  float* act = nullptr;
  CK(cudaMallocAsync(&act, (size_t)rows * E * 4, s));
  launch_silu_f32(context_dev, act, (int64_t)rows * E, s);
  GemmArgs g;
  memset(&g, 0, sizeof g);
  g.a0 = act; g.lda0 = E; g.k0 = E; g.w = h->ctx_wall; g.ldw = E; g.bias = h->ctx_ball; g.d = h->ctx_table;
  g.ldd = ncb * 2 * C; g.M = rows; g.N = ncb * 2 * C; g.act = ACT_NONE;
  launch_gemm_f32(g, s);
  CK(cudaFreeAsync(act, s));
  h->launches += 2;
  if ((shared != 0) != h->ctx_shared || !h->ctx_set) drop_graph(h);     // FiLM mode is baked into the captured launches
  h->ctx_shared = shared != 0;
  h->ctx_batch = shared ? 0 : batch;
  h->ctx_set = true;
  for (size_t i = 0; i < h->tc.size(); ++i)     // fused epilogues carry the table pointer / mode
    if (h->tc[i] && P.ops[i].kind == OP_GEMM_GN && P.ops[i].film == 2) tc_plan_set_film(h->tc[i], film_ref(h, P.ops[i]));
  if (!stream) CK(cudaStreamSynchronize(s));
  return 0;
}

extern "C" int ds_set_context_cross(ds_handle* h, const float* cross_dev, int32_t batch, int32_t L, void* stream) {
  if (!h) return fail(DS_ERR_INVALID, "null handle");
  if (!h->cfg.text_condition) return fail(DS_ERR_INVALID, "configuration has no text condition");
  if (!h->committed) return fail(DS_ERR_STATE, "ds_commit_weights() first");
  if (!cross_dev) { h->xctx_batch = 0; return 0; }
  if (batch <= 0 || L <= 0 || L > 512) return fail(DS_ERR_INVALID, "bad context_cross shape");
  CK(cudaSetDevice(h->cfg.device));
  cudaStream_t s = stream ? (cudaStream_t)stream : h->own_stream;
  const int nl = int(h->plan.xattn_layers.size()), TD = h->cfg.text_dim;
  if (batch != h->xctx_cap) {
    drop_graph(h);
    cudaFree(h->xctx);
    h->xctx = nullptr;
    CK(cudaMalloc(&h->xctx, (size_t)nl * batch * 4096 * 4));
    h->xctx_cap = batch;
  }
  float* kv = nullptr;
  CK(cudaMallocAsync(&kv, (size_t)batch * L * 256 * 4, s));
  for (int l = 0; l < nl; ++l) {
    GemmArgs g;
    memset(&g, 0, sizeof g);
    g.a0 = cross_dev; g.lda0 = TD; g.k0 = TD; g.w = h->kv_w[l]; g.ldw = TD; g.d = kv; g.ldd = 256;
    g.M = batch * L; g.N = 256; g.act = ACT_NONE;
    launch_gemm_f32(g, s);
    launch_xattn_prepare<float>(kv, 256, h->xctx + (size_t)l * batch * 4096, batch, L, s);
    CK(cudaGetLastError());
    h->launches += 2;
  }
  CK(cudaFreeAsync(kv, s));
  h->xctx_batch = batch;
  if (!stream) CK(cudaStreamSynchronize(s));
  return 0;
}

static int check_ready(ds_handle* h, int batch) {
  if (!h->ctx_set) return fail(DS_ERR_STATE, "ds_set_context() has not been called since the last weight commit");
  if (!h->ctx_shared && h->ctx_batch != batch)
    return fail(DS_ERR_STATE, "context was set for batch %d, call uses batch %d", h->ctx_batch, batch);
  if (h->cfg.text_condition && h->xctx_batch != batch)
    return fail(DS_ERR_STATE, "context_cross was set for batch %d, call uses batch %d", h->xctx_batch, batch);
  return 0;
}

// ------------------------------------------------------------------------------------------------
// forward
// ------------------------------------------------------------------------------------------------
static int unpack_out(ds_handle* h, float* out, int n_scenes, cudaStream_t s) {
  const Plan& P = h->plan;
  const int M = n_scenes * h->cfg.num_objects;
  if (h->bf16_mode) launch_unpack_output<bf16>((const bf16*)h->bufs[P.out_buf], P.dpad, out, M, P.d, s);
  else launch_unpack_output<float>((const float*)h->bufs[P.out_buf], P.dpad, out, M, P.d, s);
  h->launches++;
  return 0;
}

extern "C" int ds_denoise_forward(ds_handle* h, const float* x_t_dev, const int64_t* t_dev, float* out_dev,
                                  int32_t batch, void* stream) {
  if (!h || !x_t_dev || !t_dev || !out_dev) return fail(DS_ERR_INVALID, "null argument");
  CK(cudaSetDevice(h->cfg.device));
  int rc = ensure_capacity(h, batch);
  if (rc) return rc;
  if ((rc = check_ready(h, batch))) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  launch_t_convert(t_dev, h->t_dev, batch, s);
  h->launches++;
  if ((rc = run_forward(h, x_t_dev, batch, s))) return rc;
  unpack_out(h, out_dev, batch, s);
  CK(cudaGetLastError());
  return 0;
}

extern "C" int ds_denoise_forward_host(ds_handle* h, const float* x_t, const int64_t* t, float* out, int32_t batch) {
  if (!h || !x_t || !t || !out) return fail(DS_ERR_INVALID, "null argument");
  CK(cudaSetDevice(h->cfg.device));
  int rc = ensure_capacity(h, batch);
  if (rc) return rc;
  cudaStream_t s = h->own_stream;
  size_t xs = (size_t)batch * h->cfg.num_objects * h->plan.d * sizeof(float);
  CK(cudaMemcpyAsync(h->x_tmp, x_t, xs, cudaMemcpyHostToDevice, s));
  CK(cudaMemcpyAsync(h->t64_tmp, t, sizeof(int64_t) * batch, cudaMemcpyHostToDevice, s));
  if ((rc = ds_denoise_forward(h, h->x_tmp, h->t64_tmp, h->x_state, batch, s))) return rc;
  CK(cudaMemcpyAsync(out, h->x_state, xs, cudaMemcpyDeviceToHost, s));
  CK(cudaStreamSynchronize(s));
  return 0;
}

// ------------------------------------------------------------------------------------------------
// sampling
// ------------------------------------------------------------------------------------------------
extern "C" int ds_traj_count(int32_t T, int32_t freq) {
  if (freq <= 0) return 0;
  int n = 0;
  for (int t = T - 1; t >= 0; --t)
    if (t % freq == 0 || t == T - 1) ++n;
  return n;
}

static void model_coefs(ds_handle* h, int t, float* a_x, float* a_o) {
  if (h->mean_type == DS_MEAN_V) { *a_x = h->sched_host[S_SQRT_AC][t]; *a_o = -h->sched_host[S_SQRT_1MAC][t]; }
  else if (h->mean_type == DS_MEAN_EPS) { *a_x = h->sched_host[S_SQRT_RECIP][t]; *a_o = -h->sched_host[S_SQRT_RECIPM1][t]; }
  else { *a_x = 0.f; *a_o = 1.f; }
}

static int step_body(ds_handle* h, const ds_sample_args* a, cudaStream_t s) {
  const Plan& P = h->plan;
  struct Uni { ds_handle* h; Uni(ds_handle* x) : h(x) { h->t_uniform = 1; } ~Uni() { h->t_uniform = 0; } } uni(h);
  const int B = a->batch, n_obj = h->cfg.num_objects;
  launch_begin_step(h->coef_dev, h->state_dev, h->t_dev, h->x_state, a->partial_dev, a->partial_noise_dev, B, n_obj,
                    P.d, a->partial_dev ? a->num_partial : 0, s);
  h->launches++;
  int rc = run_forward(h, h->x_state, B, s);
  if (rc) return rc;
  const int clip = a->ddim ? 1 : a->clip_denoised;
  if (h->bf16_mode)
    launch_step_update<bf16>(h->coef_dev, h->state_dev, h->x_state, (const bf16*)h->bufs[P.out_buf], P.dpad,
                             a->noise_dev, B, n_obj, P.d, clip, s);
  else
    launch_step_update<float>(h->coef_dev, h->state_dev, h->x_state, (const float*)h->bufs[P.out_buf], P.dpad,
                              a->noise_dev, B, n_obj, P.d, clip, s);
  h->launches++;
  return 0;
}

extern "C" int ds_sample_loop(ds_handle* h, const ds_sample_args* a, float* out_dev, void* stream) {
  if (!h || !a || !out_dev) return fail(DS_ERR_INVALID, "null argument");
  if (h->T == 0) return fail(DS_ERR_STATE, "ds_set_schedule() has not been called");
  CK(cudaSetDevice(h->cfg.device));
  const int B = a->batch;
  if (a->chunk_scenes > 0 && B > a->chunk_scenes && !a->noise_dev && !a->partial_dev && a->traj_freq <= 0 &&
      h->ctx_shared && !h->cfg.text_condition) {
    // sub-batches run the full loop back to back; Philox streams are keyed by the global scene index, so the
    // result is identical to the unchunked run
    const size_t per = (size_t)h->cfg.num_objects * h->plan.d;
    for (int c0 = 0; c0 < B; c0 += a->chunk_scenes) {
      ds_sample_args sub = *a;
      sub.batch = std::min(a->chunk_scenes, B - c0);
      sub.chunk_scenes = 0;
      sub.scene_offset = a->scene_offset + c0;
      if (a->x_init_dev) sub.x_init_dev = a->x_init_dev + (size_t)c0 * per;
      int rc = ds_sample_loop(h, &sub, out_dev + (size_t)c0 * per, stream);
      if (rc) return rc;
    }
    return 0;
  }
  int rc = ensure_capacity(h, B);
  if (rc) return rc;
  if ((rc = check_ready(h, B))) return rc;
  const Plan& P = h->plan;
  const int n_obj = h->cfg.num_objects, T = h->T;
  if (a->partial_dev && (a->num_partial <= 0 || a->num_partial > n_obj))
    return fail(DS_ERR_INVALID, "num_partial out of range");
  // the loop is captured into a CUDA graph: needs a capturable (non-legacy) stream
  cudaStream_t s = stream ? (cudaStream_t)stream : h->own_stream;

  // ---- per-step coefficient table ----
  std::vector<StepCoef> coef;
  std::vector<int> ts;
  if (!a->ddim) {
    int n = a->num_steps > 0 ? a->num_steps : T;
    if (n > T) return fail(DS_ERR_INVALID, "num_steps > T");
    for (int t = n - 1; t >= 0; --t) {
      StepCoef c;
      model_coefs(h, t, &c.a_x, &c.a_o);
      c.c_0 = h->sched_host[S_COEF1][t];
      c.c_x = h->sched_host[S_COEF2][t];
      c.c_z = h->sched_host[S_SIGMA][t];
      c.q_a = h->sched_host[S_SQRT_AC][t];
      c.q_b = h->sched_host[S_SQRT_1MAC][t];
      c.t = t;
      coef.push_back(c);
      ts.push_back(t);
    }
  } else {
    const int S = a->num_steps > 0 ? a->num_steps : 50;
    std::vector<int> times(S + 1);
    if (a->ddim_times) {
      for (int i = 0; i <= S; ++i) times[i] = a->ddim_times[i];
    } else {
      // torch.linspace(-1, T-1, S+1).int() reversed (diffusion_ddpm.py:407-408)
      for (int i = 0; i <= S; ++i) times[S - i] = int(-1.0 + double(T) * double(i) / double(S));
    }
    for (int i = 0; i < S; ++i) {
      const int t = times[i], tn = times[i + 1];
      if (t < 0 || t >= T || tn >= T) return fail(DS_ERR_INVALID, "bad DDIM time pair (%d, %d)", t, tn);
      StepCoef c;
      model_coefs(h, t, &c.a_x, &c.a_o);
      c.q_a = h->sched_host[S_SQRT_AC][t];
      c.q_b = h->sched_host[S_SQRT_1MAC][t];
      c.t = t;
      if (tn < 0) {
        c.c_0 = 1.f; c.c_x = 0.f; c.c_z = 0.f;
      } else {
        const double al = h->sched_host[S_AC][t], an = h->sched_host[S_AC][tn];
        const double sr = h->sched_host[S_SQRT_RECIP][t], srm1 = h->sched_host[S_SQRT_RECIPM1][t];
        const double sigma = a->ddim_eta * sqrt((1 - al / an) * (1 - an) / (1 - al));
        const double cc = sqrt(1 - an - sigma * sigma);
        c.c_0 = float(sqrt(an) - cc / srm1);      // x0 coefficient after substituting eps = (sr*x - x0)/srm1
        c.c_x = float(cc * sr / srm1);
        c.c_z = float(sigma);
      }
      coef.push_back(c);
      ts.push_back(t);
    }
  }
  const int n_steps = int(coef.size());
  if (n_steps > h->coef_cap) {
    cudaFree(h->coef_dev);
    h->coef_dev = nullptr;
    CK(cudaMalloc(&h->coef_dev, sizeof(StepCoef) * n_steps));
    h->coef_cap = n_steps;
  }
  CK(cudaMemcpyAsync(h->coef_dev, coef.data(), sizeof(StepCoef) * n_steps, cudaMemcpyHostToDevice, s));
  StepState st0;
  st0.step = 0; st0.done = 0; st0.seed = a->seed; st0.scene_offset = a->scene_offset;
  CK(cudaMemcpyAsync(h->state_dev, &st0, sizeof(StepState), cudaMemcpyHostToDevice, s));
  CK(cudaStreamSynchronize(s));      // coef / st0 are locals

  const size_t xs = (size_t)B * n_obj * P.d * sizeof(float);
  if (a->x_init_dev) CK(cudaMemcpyAsync(h->x_state, a->x_init_dev, xs, cudaMemcpyDeviceToDevice, s));
  else {
    launch_randn(h->x_state, B, n_obj * P.d, a->seed, a->scene_offset, 2u, s);
    h->launches++;
  }

  cudaGraphExec_t gexec = nullptr;
  int64_t launches_per_step = 0;
  if (a->use_graph) {
    ds_handle::GraphKey key;
    key.batch = B; key.clip = a->ddim ? 1 : a->clip_denoised; key.num_partial = a->partial_dev ? a->num_partial : 0;
    key.plan_gen = h->plan_gen; key.noise = a->noise_dev; key.partial = a->partial_dev;
    key.partial_noise = a->partial_noise_dev; key.stream = s;
    if (!h->gexec || !(h->gkey == key)) {
      if (h->gexec) { cudaGraphExecDestroy(h->gexec); h->gexec = nullptr; }
      cudaGraph_t graph = nullptr;
      int64_t l0 = h->launches;
      CK(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
      rc = step_body(h, a, s);
      cudaError_t ce = cudaStreamEndCapture(s, &graph);
      if (rc) { if (graph) cudaGraphDestroy(graph); return rc; }
      if (ce != cudaSuccess) return fail(DS_ERR_CUDA, "graph capture failed: %s", cudaGetErrorString(ce));
      ce = cudaGraphInstantiate(&h->gexec, graph, 0);
      cudaGraphDestroy(graph);
      if (ce != cudaSuccess) { h->gexec = nullptr; return fail(DS_ERR_CUDA, "cudaGraphInstantiate: %s", cudaGetErrorString(ce)); }
      h->g_launches = h->launches - l0;
      h->launches = l0;
      h->gkey = key;
      h->graph_builds++;
    }
    gexec = h->gexec;
    launches_per_step = h->g_launches;
  }
  int snap = 0;
  for (int i = 0; i < n_steps; ++i) {
    if (gexec) {
      CK(cudaGraphLaunch(gexec, s));
      h->launches += launches_per_step;
    } else if ((rc = step_body(h, a, s))) {
      return rc;
    }
    if (a->traj_freq > 0 && a->traj_dev && (ts[i] % a->traj_freq == 0 || i == 0)) {
      CK(cudaMemcpyAsync(a->traj_dev + (size_t)snap * B * n_obj * P.d, h->x_state, xs, cudaMemcpyDeviceToDevice, s));
      ++snap;
    }
  }
  if (a->partial_dev) {
    // paste the clean partial scene (diffusion_ddpm.py:471-473)
    CK(cudaMemcpy2DAsync(h->x_state, (size_t)n_obj * P.d * 4, a->partial_dev, (size_t)a->num_partial * P.d * 4,
                         (size_t)a->num_partial * P.d * 4, B, cudaMemcpyDeviceToDevice, s));
  }
  CK(cudaMemcpyAsync(out_dev, h->x_state, xs, cudaMemcpyDeviceToDevice, s));
  cudaError_t le = cudaGetLastError();
  if (gexec || !stream) CK(cudaStreamSynchronize(s));      // the caller's injected buffers may go away after the call
  if (le != cudaSuccess) return fail(DS_ERR_CUDA, "sampling loop: %s", cudaGetErrorString(le));
  if (tc_error_flag()) return fail(DS_ERR_CUDA, "tcgen05 pipeline timeout (code %d)", tc_error_flag());
  return 0;
}

extern "C" int ds_sample_loop_host(ds_handle* h, const ds_sample_args* a, float* out_host) {
  if (!h || !a || !out_host) return fail(DS_ERR_INVALID, "null argument");
  CK(cudaSetDevice(h->cfg.device));
  int rc = ensure_capacity(h, a->batch);
  if (rc) return rc;
  size_t xs = (size_t)a->batch * h->cfg.num_objects * h->plan.d * sizeof(float);
  if ((rc = ds_sample_loop(h, a, h->x_tmp, h->own_stream))) return rc;
  CK(cudaMemcpyAsync(out_host, h->x_tmp, xs, cudaMemcpyDeviceToHost, h->own_stream));
  CK(cudaStreamSynchronize(h->own_stream));
  return 0;
}

extern "C" int ds_p_sample_step(ds_handle* h, const float* x_t_dev, const int64_t* t_dev, const float* noise_dev,
                                int32_t clip_denoised, float* out_dev, int32_t batch, void* stream) {
  if (!h || !x_t_dev || !t_dev || !noise_dev || !out_dev) return fail(DS_ERR_INVALID, "null argument");
  if (h->T == 0) return fail(DS_ERR_STATE, "ds_set_schedule() has not been called");
  CK(cudaSetDevice(h->cfg.device));
  int rc = ensure_capacity(h, batch);
  if (rc) return rc;
  if ((rc = check_ready(h, batch))) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const Plan& P = h->plan;
  launch_t_convert(t_dev, h->t_dev, batch, s);
  h->launches++;
  if ((rc = run_forward(h, x_t_dev, batch, s))) return rc;
  const float *ax, *ao;
  if (h->mean_type == DS_MEAN_V) { ax = h->sched_dev[S_SQRT_AC]; ao = h->sched_dev[S_NEG_1MAC]; }
  else if (h->mean_type == DS_MEAN_EPS) { ax = h->sched_dev[S_SQRT_RECIP]; ao = h->sched_dev[S_NEG_RECIPM1]; }
  else { ax = h->sched_dev[S_ZERO]; ao = h->sched_dev[S_ONE]; }
  if (h->bf16_mode)
    launch_p_sample<bf16>(x_t_dev, (const bf16*)h->bufs[P.out_buf], P.dpad, h->t_dev, noise_dev, out_dev, ax, ao,
                          h->sched_dev[S_COEF1], h->sched_dev[S_COEF2], h->sched_dev[S_SIGMA], batch,
                          h->cfg.num_objects, P.d, clip_denoised, s);
  else
    launch_p_sample<float>(x_t_dev, (const float*)h->bufs[P.out_buf], P.dpad, h->t_dev, noise_dev, out_dev, ax, ao,
                           h->sched_dev[S_COEF1], h->sched_dev[S_COEF2], h->sched_dev[S_SIGMA], batch,
                           h->cfg.num_objects, P.d, clip_denoised, s);
  h->launches++;
  CK(cudaGetLastError());
  return 0;
}

extern "C" int ds_q_sample(ds_handle* h, const float* x0_dev, const int64_t* t_dev, const float* noise_dev,
                           float* out_dev, int32_t batch, void* stream) {
  if (!h || !x0_dev || !t_dev || !noise_dev || !out_dev) return fail(DS_ERR_INVALID, "null argument");
  if (h->T == 0) return fail(DS_ERR_STATE, "ds_set_schedule() has not been called");
  CK(cudaSetDevice(h->cfg.device));
  launch_q_sample(x0_dev, t_dev, noise_dev, out_dev, h->sched_dev[S_SQRT_AC], h->sched_dev[S_SQRT_1MAC], batch,
                  h->cfg.num_objects * h->plan.d, (cudaStream_t)stream);
  h->launches++;
  CK(cudaGetLastError());
  return 0;
}

extern "C" int ds_p_losses(ds_handle* h, const float* x0_dev, const int64_t* t_dev, const float* noise_dev,
                           int32_t loss_separate, int32_t loss_iou, const float* bounds_host, float* losses_dev,
                           float* loss_dict_dev, int32_t batch, void* stream) {
  if (!h || !x0_dev || !t_dev || !noise_dev || !losses_dev || !loss_dict_dev)
    return fail(DS_ERR_INVALID, "null argument");
  if (h->T == 0) return fail(DS_ERR_STATE, "ds_set_schedule() has not been called");
  if (loss_iou && !bounds_host) return fail(DS_ERR_INVALID, "loss_iou needs bounds");
  CK(cudaSetDevice(h->cfg.device));
  int rc = ensure_capacity(h, batch);
  if (rc) return rc;
  if ((rc = check_ready(h, batch))) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  const Plan& P = h->plan;
  const ds_config& c = h->cfg;
  launch_q_sample(x0_dev, t_dev, noise_dev, h->x_tmp, h->sched_dev[S_SQRT_AC], h->sched_dev[S_SQRT_1MAC], batch,
                  c.num_objects * P.d, s);
  launch_t_convert(t_dev, h->t_dev, batch, s);
  h->launches += 2;
  if ((rc = run_forward(h, h->x_tmp, batch, s))) return rc;
  LossArgs a;
  memset(&a, 0, sizeof a);
  a.n_obj = c.num_objects; a.d = P.d; a.trans = c.translation_dim; a.size = c.size_dim; a.angle = c.angle_dim;
  a.cls = c.class_dim; a.objn = c.objectness_dim; a.feat = c.objfeat_dim;
  a.mean_type = h->mean_type; a.loss_separate = loss_separate; a.loss_iou = loss_iou;
  a.arrange = c.seperate_all ? 0 : 1;
  if (a.arrange) { a.angle = P.d - a.trans; a.loss_iou = 0; }
  if (bounds_host) memcpy(a.bounds, bounds_host, sizeof(float) * 12);
  if (h->bf16_mode)
    launch_p_losses<bf16>(x0_dev, noise_dev, h->x_tmp, (const bf16*)h->bufs[P.out_buf], P.dpad, t_dev,
                          h->sched_dev[S_SQRT_AC], h->sched_dev[S_SQRT_1MAC], h->sched_dev[S_SQRT_RECIP],
                          h->sched_dev[S_SQRT_RECIPM1], h->sched_dev[S_LW], h->sched_dev[S_AC], a, losses_dev,
                          h->loss_parts, batch, s);
  else
    launch_p_losses<float>(x0_dev, noise_dev, h->x_tmp, (const float*)h->bufs[P.out_buf], P.dpad, t_dev,
                           h->sched_dev[S_SQRT_AC], h->sched_dev[S_SQRT_1MAC], h->sched_dev[S_SQRT_RECIP],
                           h->sched_dev[S_SQRT_RECIPM1], h->sched_dev[S_LW], h->sched_dev[S_AC], a, losses_dev,
                           h->loss_parts, batch, s);
  launch_loss_dict_mean(h->loss_parts, loss_dict_dev, batch, s);
  h->launches += 2;
  CK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// post-processing: object retrieval (stateless; any sm_100 device)
// ------------------------------------------------------------------------------------------------
extern "C" int ds_retrieve_objects(const int32_t* class_start_dev, int32_t n_classes, const float* cat_feat_dev,
                                   const float* cat_size_dev, int32_t feat_dim, int32_t size_dim,
                                   const int64_t* q_label_dev, const float* q_feat_dev, const float* q_size_dev,
                                   int32_t num_queries, int32_t mode, int64_t* out_index_dev, void* stream) {
  if (!class_start_dev || !q_label_dev || !out_index_dev || n_classes <= 0 || num_queries < 0 || mode < 0 || mode > 2)
    return fail(DS_ERR_INVALID, "bad argument to ds_retrieve_objects");
  if (mode != 2 && (!cat_feat_dev || !q_feat_dev || feat_dim <= 0)) return fail(DS_ERR_INVALID, "feature arrays needed");
  if (mode != 1 && (!cat_size_dev || !q_size_dev || size_dim <= 0)) return fail(DS_ERR_INVALID, "size arrays needed");
  int ndev = 0;
  if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
    cudaGetLastError();
    return fail(DS_ERR_NO_DEVICE, "no CUDA device: diffuscene_b200 has no CPU fallback");
  }
  if (num_queries == 0) return 0;
  launch_retrieve(class_start_dev, n_classes, cat_feat_dev, cat_size_dev, feat_dim, size_dim, q_label_dev, q_feat_dev,
                  q_size_dev, num_queries, mode, out_index_dev, (cudaStream_t)stream);
  CK(cudaGetLastError());
  return 0;
}

// ------------------------------------------------------------------------------------------------
// introspection
// ------------------------------------------------------------------------------------------------
extern "C" int ds_plan_describe(const ds_config* cfg, char* buf, int64_t buf_len) {
  if (!cfg || !buf || buf_len <= 0) return fail(DS_ERR_INVALID, "bad argument");
  Plan p;
  if (!build_plan(*cfg, false, &p)) return fail(DS_ERR_INVALID, "%s", p.error.c_str());
  std::string s = describe_plan(p);
  s += "weights:\n";
  for (auto& n : p.expected_order) s += n + " " + std::to_string(p.expected[n]) + "\n";
  int64_t n = std::min<int64_t>((int64_t)s.size(), buf_len - 1);
  memcpy(buf, s.data(), n);
  buf[n] = 0;
  return int(n);
}

extern "C" int ds_plan_export_json(const ds_config* cfg, int32_t no_reuse, char* buf, int64_t buf_len) {
  if (!cfg || !buf || buf_len <= 0) return fail(DS_ERR_INVALID, "bad argument");
  Plan p;
  if (!build_plan(*cfg, no_reuse != 0, &p)) return fail(DS_ERR_INVALID, "%s", p.error.c_str());
  std::string s = export_plan_json(p);
  if ((int64_t)s.size() + 1 > buf_len) return fail(DS_ERR_INVALID, "buffer too small (%lld needed)", (long long)s.size() + 1);
  memcpy(buf, s.data(), s.size());
  buf[s.size()] = 0;
  return int(s.size());
}

extern "C" int ds_enable_taps(ds_handle* h, int32_t on) {
  if (!h) return fail(DS_ERR_INVALID, "null handle");
  if ((on != 0) == h->taps) return 0;
  CK(cudaSetDevice(h->cfg.device));
  Plan np;
  if (!build_plan(h->cfg, on != 0, &np)) return fail(DS_ERR_INVALID, "%s", np.error.c_str());
  free_buffers(h);
  h->plan = np;
  h->taps = on != 0;
  if (h->committed) return ds_commit_weights(h);   // vector / matrix ids are stable, buffers are not
  return 0;
}

extern "C" int ds_read_tap(ds_handle* h, const char* name, float* host_out, int64_t capacity, int32_t* rows,
                           int32_t* width) {
  if (!h || !name || !host_out) return fail(DS_ERR_INVALID, "null argument");
  if (!h->taps) return fail(DS_ERR_STATE, "taps are not enabled");
  CK(cudaSetDevice(h->cfg.device));
  const Plan& P = h->plan;
  for (const Op& o : P.ops) {
    if (o.name != name || o.out < 0) continue;
    const int w = P.buf_width[o.out], r = h->cap_scenes * h->cfg.num_objects;
    if ((int64_t)r * w > capacity) return fail(DS_ERR_INVALID, "tap buffer too small");
    CK(cudaDeviceSynchronize());
    if (h->bf16_mode) {
      std::vector<uint16_t> tmp((size_t)r * w);
      CK(cudaMemcpy(tmp.data(), h->bufs[o.out], tmp.size() * 2, cudaMemcpyDeviceToHost));
      for (size_t i = 0; i < tmp.size(); ++i) {
        uint32_t u = uint32_t(tmp[i]) << 16;
        memcpy(host_out + i, &u, 4);
      }
    } else {
      CK(cudaMemcpy(host_out, h->bufs[o.out], (size_t)r * w * 4, cudaMemcpyDeviceToHost));
    }
    if (rows) *rows = r;
    if (width) *width = w;
    return 0;
  }
  return fail(DS_ERR_INVALID, "no op named '%s'", name);
}

extern "C" int64_t ds_launch_count(ds_handle* h) { return h ? h->launches : 0; }
extern "C" int64_t ds_graph_build_count(ds_handle* h) { return h ? h->graph_builds : 0; }
extern "C" int32_t ds_gnt_weight_row(int32_t stored_row) { return tc_gnt_row(stored_row); }

extern "C" int ds_profile_ops(ds_handle* h, int32_t batch, char* names_buf, int64_t names_len, float* usec,
                              int32_t cap) {
  if (!h || !names_buf || !usec) return fail(DS_ERR_INVALID, "null argument");
  CK(cudaSetDevice(h->cfg.device));
  int rc = ensure_capacity(h, batch);
  if (rc) return rc;
  if ((rc = check_ready(h, batch))) return rc;
  const Plan& P = h->plan;
  cudaStream_t s = h->own_stream;
  const int n = int(P.ops.size());
  std::vector<cudaEvent_t> ev(n + 1);
  for (auto& e : ev) cudaEventCreate(&e);
  CK(cudaMemsetAsync(h->x_state, 0, (size_t)batch * h->cfg.num_objects * P.d * 4, s));
  std::vector<float> acc(n, 0.f);
  const int reps = 5;
  for (int rep = 0; rep < reps + 1; ++rep) {
    cudaEventRecord(ev[0], s);
    for (int i = 0; i < n; ++i) {
      if (P.ops[i].kind == OP_PACK) {
        if (h->bf16_mode) launch_pack_input<bf16>(h->x_state, (bf16*)h->bufs[P.ops[i].out], P.kin_pad,
                                                  batch * h->cfg.num_objects, P.d, s);
        else launch_pack_input<float>(h->x_state, (float*)h->bufs[P.ops[i].out], P.kin_pad,
                                      batch * h->cfg.num_objects, P.d, s);
      } else {
        rc = h->bf16_mode ? run_op<bf16>(h, i, batch, s) : run_op<float>(h, i, batch, s);
        if (rc) return rc;
      }
      cudaEventRecord(ev[i + 1], s);
    }
    CK(cudaStreamSynchronize(s));
    if (rep == 0) continue;    // warm-up
    for (int i = 0; i < n; ++i) {
      float ms = 0;
      cudaEventElapsedTime(&ms, ev[i], ev[i + 1]);
      acc[i] += ms * 1000.f / reps;
    }
  }
  for (auto& e : ev) cudaEventDestroy(e);
  std::string names;
  for (int i = 0; i < n && i < cap; ++i) {
    usec[i] = acc[i];
    names += P.ops[i].name + "\n";
  }
  int64_t m = std::min<int64_t>((int64_t)names.size(), names_len - 1);
  memcpy(names_buf, names.data(), m);
  names_buf[m] = 0;
  return n;
}

// Bring-up aid: one tcgen05 GEMM (optionally with the GroupNorm epilogue, n_obj > 0) with per-role cycle counters.
// trace_host receives [148][8] uint64 (see gemm_tc.cu for the slot meaning); reps launches are timed with events.
extern "C" int ds_test_gemm_trace(const void* a_dev, const void* w_dev, const float* bias_dev, const void* res_dev,
                                  void* d_dev, int32_t M, int32_t N, int32_t K, int32_t n_obj, const float* gamma_dev,
                                  const float* beta_dev, int32_t reps, unsigned long long* trace_host, float* usec) {
  GemmArgs g;
  memset(&g, 0, sizeof g);
  g.a0 = a_dev; g.lda0 = K; g.k0 = K; g.w = w_dev; g.ldw = K; g.bias = bias_dev; g.d = d_dev; g.ldd = N;
  g.res = res_dev; g.ldres = N; g.M = M; g.N = N;
  // n_obj < 0: the channels-on-lanes variant (the caller passes the weight rows in tc_gnt_row order)
  // ... and n_obj < 0 with gamma == NULL: the same kernel as a plain GEMM (act passed in `reps` bits 8.. for the probe)
  if (n_obj != 0) {
    g.gn = n_obj < 0 ? (gamma_dev ? 2 : 3) : 1; g.n_obj = n_obj < 0 ? -n_obj : n_obj; g.film_C = N; g.gamma = gamma_dev;
    g.beta = beta_dev; g.film.mode = FILM_NONE;
    if (g.gn == 3) { g.act = reps >> 8; reps &= 0xff; }
  }
  char err[256] = "";
  TcGemmPlan* p = tc_plan_create(g, M, err, sizeof err);
  if (!p) return fail(DS_ERR_CUDA, "%s", err);
  unsigned long long* tr = nullptr;
  CK(cudaMalloc(&tr, 256 * 8 * sizeof(unsigned long long)));
  CK(cudaMemset(tr, 0, 256 * 8 * sizeof(unsigned long long)));
  cudaEvent_t e0, e1;
  cudaEventCreate(&e0); cudaEventCreate(&e1);
  int le = 0;
  for (int i = 0; i < 3; ++i) le |= launch_gemm_tc(p, M, 0);
  if (le) {       // launch errors are not sticky: without this check a refused launch reads as a 1 us kernel
    cudaFree(tr);
    tc_plan_destroy(p);
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    return fail(DS_ERR_CUDA, "trace GEMM launch failed: %s", cudaGetErrorString((cudaError_t)le));
  }
  cudaEventRecord(e0, 0);
  for (int i = 0; i < reps; ++i) launch_gemm_tc(p, M, 0);
  cudaEventRecord(e1, 0);
  cudaError_t se = cudaDeviceSynchronize();
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  if (usec) *usec = ms * 1000.f / reps;
  tc_plan_set_trace(p, tr);
  launch_gemm_tc(p, M, 0);
  se = cudaDeviceSynchronize();
  if (trace_host) cudaMemcpy(trace_host, tr, 256 * 8 * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
  cudaFree(tr);
  tc_plan_destroy(p);
  cudaEventDestroy(e0); cudaEventDestroy(e1);
  if (se != cudaSuccess) return fail(DS_ERR_CUDA, "trace GEMM failed: %s (code %d)", cudaGetErrorString(se), tc_error_flag());
  return 0;
}

extern "C" int ds_test_gemm_bf16(int backend, const void* a_dev, const void* w_dev, const float* bias_dev, void* d_dev,
                                 int32_t M, int32_t N, int32_t K, int32_t act, void* stream) {
  GemmArgs g;
  memset(&g, 0, sizeof g);
  g.a0 = a_dev; g.lda0 = K; g.k0 = K; g.w = w_dev; g.ldw = K; g.bias = bias_dev; g.d = d_dev; g.ldd = N;
  g.M = M; g.N = N; g.act = act;
  cudaStream_t s = (cudaStream_t)stream;
  if (backend == DS_GEMM_TCGEN05) {
    char err[256] = "";
    TcGemmPlan* p = tc_plan_create(g, M, err, sizeof err);
    if (!p) return fail(DS_ERR_CUDA, "%s", err);
    int e = launch_gemm_tc(p, M, s);
    cudaError_t se = cudaStreamSynchronize(s);
    tc_plan_destroy(p);
    if (e) return fail(DS_ERR_CUDA, "launch failed: %s", cudaGetErrorString((cudaError_t)e));
    if (se != cudaSuccess)
      return fail(DS_ERR_CUDA, "tcgen05 GEMM failed: %s (pipeline code %d)", cudaGetErrorString(se), tc_error_flag());
    return 0;
  }
  launch_gemm_simt<bf16>(g, false, s);
  CK(cudaStreamSynchronize(s));
  return 0;
}
