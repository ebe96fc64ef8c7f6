/*
 * diffuscene_b200 -- C ABI of the B200-native DiffuScene denoising hot path.
 *
 * The reference (tangjiapeng/DiffuScene) is pure Python/PyTorch and has no FFI of its own; this
 * header is the boundary a maintainer binds with ctypes (see INTEGRATION.md).  Each entry point
 * names the reference interface it replaces (paths relative to the reference repository root).
 *
 * Conventions
 *   - plain C types only; no torch / CUDA types in signatures (streams travel as void*).
 *   - "dev" pointers are device (HBM) pointers borrowed from the caller; "host" pointers are host
 *     memory.  Nothing is allocated inside the hot calls once a batch size has been seen.
 *   - every function returns 0 on success or a negative ds_status; ds_last_error() gives the text.
 *   - a handle is bound to one device and is not thread-safe; distinct handles are independent.
 *   - there is NO CPU fallback: without a CUDA device ds_create() fails with DS_ERR_NO_DEVICE
 *     (ds_plan_describe() is the only compute-free introspection call that works without one).
 */
#ifndef DIFFUSCENE_B200_H_
#define DIFFUSCENE_B200_H_

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define DS_API __attribute__((visibility("default")))
#else
#define DS_API
#endif

typedef struct ds_handle ds_handle;

enum ds_status {
  DS_OK = 0,
  DS_ERR_INVALID = -1,      /* bad argument / unsupported configuration            */
  DS_ERR_NO_DEVICE = -2,    /* no CUDA device or not sm_100                        */
  DS_ERR_CUDA = -3,         /* a CUDA runtime / driver call failed                 */
  DS_ERR_STATE = -4,        /* call order violated (weights / schedule / context)  */
  DS_ERR_MISSING_WEIGHT = -5
};

enum ds_precision {
  DS_PREC_FP32 = 0,   /* parity mode: fp32 storage + fp32 FMA GEMMs (rtol 1e-3 / atol 1e-4 vs reference) */
  DS_PREC_BF16 = 1    /* throughput mode: bf16 storage, tcgen05 tensor-core GEMMs, fp32 accumulate/norms */
};

enum ds_gemm_backend {
  DS_GEMM_AUTO = 0,   /* tcgen05 for bf16, SIMT for fp32 */
  DS_GEMM_SIMT = 1,   /* CUDA-core GEMM for either precision (debug / cross-check) */
  DS_GEMM_TCGEN05 = 2
};

enum ds_mean_type { DS_MEAN_EPS = 0, DS_MEAN_X0 = 1, DS_MEAN_V = 2 };

/* Mirrors the reference's `net_kwargs` for Unet1D (scene_synthesis/networks/denoise_net.py:336-362)
 * plus the engine knobs.  dim_mults must be all ones (every shipped config). */
typedef struct ds_config {
  int32_t dim;              /* hidden width C (512)                                   */
  int32_t channels;         /* point_dim when seperate_all == 0                        */
  int32_t seperate_all;     /* 1: per-attribute encoder / decoder MLPs                 */
  int32_t objectness_dim, class_dim, translation_dim, size_dim, angle_dim, objfeat_dim;
  int32_t cond_dim;         /* context_dim + instanclass_dim: width of `context`       */
  int32_t text_condition;   /* 1: LinearAttentionCross layers present                  */
  int32_t text_dim;
  int32_t n_stages;         /* len(dim_mults), 4                                       */
  int32_t num_objects;      /* N: objects per scene (12 bedroom / 21 living)           */
  int32_t num_timesteps;    /* T of the diffusion schedule (time FiLM table rows)      */
  int32_t precision;        /* ds_precision                                            */
  int32_t gemm_backend;     /* ds_gemm_backend                                         */
  int32_t device;           /* CUDA device ordinal                                     */
  int32_t fuse_level;       /* 0: one kernel per op; 1: fused GEMM epilogues; 2: + the
                               channels-on-lanes conv+GroupNorm GEMM where supported;
                               3: + epilogue-bound plain GEMMs on that kernel;
                               4: + to_out + LayerNorm + residual of the attention wrappers
                                  as one GEMM with a LayerNorm epilogue;
                               5: + LayerNorm + to_qkv + linear-attention core as one kernel (N = 12) */
  int32_t train;            /* 1: training step program -- one op per reference layer (no fused epilogues, activations
                               as their own ops), every intermediate kept for the backward pass (ds_train_*)   */
  int32_t reserved[6];
} ds_config;

/* ---- lifetime ----------------------------------------------------------------------------- */
/* Replaces Unet1D.__init__ + DiffusionPoint.__init__ (denoise_net.py:336-482, diffusion_ddpm.py:721-731). */
DS_API int ds_create(const ds_config* cfg, ds_handle** out);
DS_API int ds_destroy(ds_handle* h);
DS_API const char* ds_last_error(void);
DS_API const char* ds_version(void);

/* ---- weights ------------------------------------------------------------------------------
 * Replaces nn.Module.load_state_dict (scene_synthesis/networks/__init__.py:62-66).  Names are the
 * reference state-dict keys with the "diffusion.model." prefix removed ("downs.0.1.block1.proj.weight").
 * Data is fp32, host memory, C-contiguous, `numel` elements.  ds_commit_weights() folds the weight
 * standardisation (denoise_net.py:78-91), packs for the selected precision, uploads, and rebuilds the
 * time-FiLM table (time_mlp + the per-block Linear of denoise_net.py:181-200 for every t in [0, T)). */
DS_API int ds_load_weight(ds_handle* h, const char* name, const float* host_data, int64_t numel);
DS_API int ds_commit_weights(ds_handle* h);
/* Number of parameter tensors the configuration expects and the i-th expected name / numel. */
DS_API int ds_expected_weight_count(ds_handle* h);
DS_API int ds_expected_weight(ds_handle* h, int index, const char** name, int64_t* numel);

/* ---- diffusion schedule -------------------------------------------------------------------
 * Replaces the table set of GaussianDiffusion.__init__ (diffusion_ddpm.py:168-203).  Each array has T
 * fp32 entries (host).  sigma[t] = (t != 0) * exp(0.5 * model_log_variance[t]) (:314-323, :348-350). */
typedef struct ds_schedule {
  int32_t T;
  int32_t mean_type;                 /* ds_mean_type */
  const float* sqrt_ac;              /* sqrt_alphas_cumprod              */
  const float* sqrt_1mac;            /* sqrt_one_minus_alphas_cumprod    */
  const float* sqrt_recip_ac;        /* sqrt_recip_alphas_cumprod        */
  const float* sqrt_recipm1_ac;      /* sqrt_recipm1_alphas_cumprod      */
  const float* coef1;                /* posterior_mean_coef1             */
  const float* coef2;                /* posterior_mean_coef2             */
  const float* sigma;                /* see above                        */
  const float* alphas_cumprod;
  const float* loss_weight;          /* p_losses weight per t (:194-203) */
} ds_schedule;
DS_API int ds_set_schedule(ds_handle* h, const ds_schedule* s);

/* ---- conditioning -------------------------------------------------------------------------
 * `context` is the [B, N, cond_dim] tensor handed to Unet1D.forward (denoise_net.py:507, built at
 * diffusion_scene_layout_ddpm.py:172-207).  shared != 0: one [N, cond_dim] block used for every scene
 * (the unconditional configs, where it is positional_embedding broadcast over the batch).
 * Device pointers, fp32.  Precomputes the 9 context-FiLM projections (they do not depend on x_t or t). */
DS_API int ds_set_context(ds_handle* h, const float* context_dev, int32_t batch, int32_t shared, void* stream);
/* `context_cross` [B, L, text_dim] fp32 device (diffusion_scene_layout_ddpm.py:210-221); precomputes the
 * k/v side of every LinearAttentionCross (denoise_net.py:284-293). Pass NULL to clear. */
DS_API int ds_set_context_cross(ds_handle* h, const float* cross_dev, int32_t batch, int32_t L, void* stream);

/* ---- denoiser forward ---------------------------------------------------------------------
 * Replaces DiffusionPoint._denoise / Unet1D.forward (diffusion_ddpm.py:748-756, denoise_net.py:507-593).
 * x_t [B, N, d] fp32, t [B] int64, out [B, N, d] fp32 -- all device pointers. */
DS_API int ds_denoise_forward(ds_handle* h, const float* x_t_dev, const int64_t* t_dev, float* out_dev,
                       int32_t batch, void* stream);
/* Same call with HOST buffers: copies in, runs, copies out, synchronises. */
DS_API int ds_denoise_forward_host(ds_handle* h, const float* x_t, const int64_t* t, float* out, int32_t batch);

/* ---- sampling -----------------------------------------------------------------------------
 * Replaces GaussianDiffusion.p_sample_loop / _trajectory / _complete / ddim (diffusion_ddpm.py:355-476)
 * and p_sample (:339-352).  One CUDA graph per step, replayed T times; t lives on the device. */
typedef struct ds_sample_args {
  int32_t batch;
  int32_t clip_denoised;        /* clamp x0 estimate to [-1, 1] (:310-311)                          */
  int32_t num_steps;            /* 0: full schedule T;  DDIM: number of sampling steps              */
  int32_t ddim;                 /* 0: ancestral DDPM (:355-371); 1: DDIM (:401-444 formula)         */
  float   ddim_eta;
  uint64_t seed;                /* Philox seed when no noise is injected                             */
  uint64_t scene_offset;        /* global index of scene 0 (keeps RNG streams independent of sharding) */
  const float* x_init_dev;      /* optional [B,N,d] x_T; NULL: drawn from Philox                     */
  const float* noise_dev;       /* optional injected noise [num_steps, B, N, d], step order T-1..0   */
  const float* partial_dev;     /* completion: clean [B, P, d] (p_sample_loop_complete :447-476)     */
  int32_t num_partial;          /* P                                                                 */
  const float* partial_noise_dev;/* optional injected q_sample noise [num_steps, B, P, d]            */
  int32_t traj_freq;            /* >0: snapshot when t % freq == 0 or t == T-1 (:394)                */
  float* traj_dev;              /* [n_snap, B, N, d] (excluding x_T); n_snap from ds_traj_count      */
  int32_t use_graph;            /* 1: CUDA-graph the step (default); 0: plain launches               */
  const int32_t* ddim_times;    /* optional host array [num_steps+1], descending, last = -1 (:407-409) */
  int32_t chunk_scenes;         /* >0: run the whole loop for sub-batches of this many scenes, one after the other,
                                   so that a sub-batch's activations stay L2-resident (Philox noise path only) */
  int32_t reserved[5];
} ds_sample_args;
DS_API int ds_sample_loop(ds_handle* h, const ds_sample_args* a, float* out_dev, void* stream);
DS_API int ds_sample_loop_host(ds_handle* h, const ds_sample_args* a, float* out_host);
DS_API int ds_traj_count(int32_t T, int32_t freq);
/* One reverse step with explicit per-sample t (p_sample, diffusion_ddpm.py:339-352). */
DS_API int ds_p_sample_step(ds_handle* h, const float* x_t_dev, const int64_t* t_dev, const float* noise_dev,
                     int32_t clip_denoised, float* out_dev, int32_t batch, void* stream);

/* ---- training-side forward pieces ---------------------------------------------------------
 * q_sample (diffusion_ddpm.py:276-286) and the p_losses value (:520-652, loss.py:7-102): per-sample
 * losses [B] and the 9 means of the reference loss dict (order: bbox, trans, size, angle, class, object,
 * objfeat, liou, bbox_iou).  bounds = {trans_min[3], trans_max[3], size_min[3], size_max[3]} or NULL. */
DS_API int ds_q_sample(ds_handle* h, const float* x0_dev, const int64_t* t_dev, const float* noise_dev,
                float* out_dev, int32_t batch, void* stream);
DS_API int ds_p_losses(ds_handle* h, const float* x0_dev, const int64_t* t_dev, const float* noise_dev,
                int32_t loss_separate, int32_t loss_iou, const float* bounds_host,
                float* losses_dev, float* loss_dict_dev, int32_t batch, void* stream);

/* ---- native training step ---------------------------------------------------------------------
 * Replaces what `loss.backward()` + `optimizer.step()` do in train_on_batch
 * (scene_synthesis/networks/diffusion_scene_layout_ddpm.py:456-473) for the denoiser: forward of p_losses
 * (diffusion_ddpm.py:520-652) with every intermediate kept, then the hand-written backward pass of every layer of
 * Unet1D (denoise_net.py:78-593: weight-standardised convs, GroupNorm + FiLM + SiLU blocks, LayerNorms, linear /
 * softmax attention, the time-embedding MLP and all FiLM projections) and of the loss (MSE terms + IoU regulariser).
 * Parameters and gradients are ONE flat fp32 device buffer each, laid out in ds_expected_weight() order
 * (ds_train_param_count() floats).  grad_scale multiplies d(mean-over-batch loss); pass 1 / world_size to get the
 * data-parallel mean after a sum all-reduce.  context [ctx_shared ? N : B*N, cond_dim] is the conditioning input of
 * Unet1D.forward; dcontext_dev (optional, same shape) receives its gradient (it continues into
 * positional_embedding / the condition MLPs on the caller's side).  flat_grads_dev == NULL: forward + loss only.
 * Uses the handle's schedule (ds_set_schedule) and precision.  Networks with text cross-attention (text_condition)
 * need ds_train_set_context_cross() for the same batch first: their to_kv projections run from flat_params_dev on
 * every step, and d(to_kv.weight) lands in flat_grads_dev like every other gradient. */
DS_API int64_t ds_train_param_count(ds_handle* h);
DS_API int ds_train_step(ds_handle* h, const float* flat_params_dev, const float* x0_dev, const int64_t* t_dev,
                         const float* noise_dev, const float* context_dev, int32_t ctx_batch, int32_t ctx_shared,
                         int32_t loss_separate, int32_t loss_iou, const float* bounds_host, float grad_scale,
                         float* losses_dev, float* loss_dict_dev, float* flat_grads_dev, float* dcontext_dev,
                         int32_t batch, void* stream);
/* Text condition of the following ds_train_step calls: context_cross [batch, L, text_dim] fp32 device (the input of
 * every LinearAttentionCross's to_kv, denoise_net.py:261-297), 1 <= L <= 512.  dcross_dev (optional, same shape)
 * receives d(loss)/d(context_cross) on every ds_train_step that computes gradients; it continues into fc_text_f on
 * the caller's side.  Pointers are borrowed until the next call; cross_dev == NULL clears.  A ds_train_step on a text
 * network without it, or with a different batch, fails with DS_ERR_STATE; a network without text condition gives
 * DS_ERR_INVALID. */
DS_API int ds_train_set_context_cross(ds_handle* h, const float* cross_dev, int32_t batch, int32_t L, float* dcross_dev);
/* Overlap of the data-parallel gradient all-reduce with the backward pass: bucket k is the flat range
 * [bounds[k], bounds[k + 1]) (bounds[0] = 0, bounds[n] = ds_train_param_count()); ds_train_step records events[k] (a
 * cudaEvent_t owned by the caller) on its stream as soon as every gradient inside the bucket is final -- the backward
 * pass finalises the buffer from its end towards its start -- so the caller's communication stream can wait on the
 * event and all-reduce that bucket while the rest of the backward pass still runs.  n_buckets = 0 clears. */
DS_API int ds_train_set_buckets(ds_handle* h, const int64_t* bounds, int32_t n_buckets, void* const* events);
/* Device time of the phases of the last ds_train_step with gradients, milliseconds (profiling aid; synchronises):
 * weight packing, forward, loss + d(loss)/d(output), backward through the step program, conditioning paths,
 * gradient unpacking (weight-standardisation adjoint). */
DS_API int ds_train_phase_ms(ds_handle* h, float* out6);
/* out[0] += sum(g^2) (device scalar; the caller zeroes it) -- the global gradient norm of clip_grad_norm_. */
DS_API int ds_sumsq(const float* g_dev, int64_t n, float* out_dev, void* stream);
/* torch.optim.Adam (weight decay 0, networks/__init__.py:15-34) on flat buffers.  sumsq_dev (optional): device
 * scalar holding the squared L2 norm of ALL gradients; with max_norm > 0 the clip coefficient
 * min(1, max_norm / (norm + 1e-6)) of clip_grad_norm_ is applied to the gradient on the fly. */
DS_API int ds_adam_step(float* params_dev, const float* grads_dev, float* exp_avg_dev, float* exp_avg_sq_dev, int64_t n,
                        float lr, float beta1, float beta2, float eps, int32_t step, const float* sumsq_dev,
                        float max_norm, void* stream);

/* ---- post-processing: object retrieval -----------------------------------------------------
 * Replaces ThreedFutureDataset.get_closest_furniture_to_objfeats_and_size (mode 0), _to_objfeats (mode 1) and
 * _to_box (mode 2) (scene_synthesis/datasets/threed_future_dataset.py:28-77) for a whole batch of generated objects:
 * out[q] = index of the catalogue entry of class q_label[q] minimising (size mse, feature mse) lexicographically
 * (mode 0; np.lexsort((mses_feat, mses_size))), the feature mse (1) or the size mse (2); ties -> lowest index;
 * -1 when the class has no entry.  The catalogue is grouped by class (stable order inside a class):
 * class_start[c] .. class_start[c + 1] is the entry range of class c (n_classes + 1 ints).  cat_feat
 * [n_entries, feat_dim], cat_size [n_entries, size_dim], q_feat [Q, feat_dim], q_size [Q, size_dim] fp32; all
 * device pointers.  Distances are accumulated in numpy's float32 order, so indices are bit-exact.  Stateless. */
DS_API int ds_retrieve_objects(const int32_t* class_start_dev, int32_t n_classes, const float* cat_feat_dev,
                               const float* cat_size_dev, int32_t feat_dim, int32_t size_dim,
                               const int64_t* q_label_dev, const float* q_feat_dev, const float* q_size_dev,
                               int32_t num_queries, int32_t mode, int64_t* out_index_dev, void* stream);

/* ---- introspection / debugging ------------------------------------------------------------ */
/* Human-readable op list of the step program (works without a device when h == NULL: builds the plan
 * for `cfg` on the host only).  Returns bytes written (excluding NUL) or a negative status. */
DS_API int ds_plan_describe(const ds_config* cfg, char* buf, int64_t buf_len);
/* The same plan (ops, buffer table, weight-packing recipes) as JSON, for host-side verification of the
 * program against the oracle without a GPU.  no_reuse != 0: one buffer per op output. */
DS_API int ds_plan_export_json(const ds_config* cfg, int32_t no_reuse, char* buf, int64_t buf_len);
/* After a forward with taps enabled, copy the named intermediate [B*N, width] to host as fp32. */
DS_API int ds_enable_taps(ds_handle* h, int32_t on);
DS_API int ds_read_tap(ds_handle* h, const char* name, float* host_out, int64_t capacity, int32_t* rows, int32_t* width);
/* Kernel launches issued by this handle since creation (ours only; no library kernels exist). */
DS_API int64_t ds_launch_count(ds_handle* h);
/* How many times ds_sample_loop had to capture + instantiate its step graph (it is cached across calls whose
 * batch / flags / injected-buffer pointers agree; seeds and shard offsets live in device memory). */
DS_API int64_t ds_graph_build_count(ds_handle* h);
/* Weight layout of the channels-on-lanes GEMM (fuse_level >= 2): the output channel whose weights are stored in row
 * `stored_row` of a packed [N, K] matrix.  Host-only (no device needed); identity for the row-major kernels. */
DS_API int32_t ds_gnt_weight_row(int32_t stored_row);
/* Per-op device time of one forward (CUDA events around each op; profiling aid, not a bench number).
 * Writes up to `cap` entries of (name, microseconds). Returns op count. */
DS_API int ds_profile_ops(ds_handle* h, int32_t batch, char* names_buf, int64_t names_len, float* usec, int32_t cap);
/* Standalone GEMM for unit tests: D[M,N] = A[M,K] * W[N,K]^T (+bias), bf16 in / bf16 out via the selected
 * backend. Device pointers. */
DS_API int ds_test_gemm_bf16(int backend, const void* a_dev, const void* w_dev, const float* bias_dev, void* d_dev,
                      int32_t M, int32_t N, int32_t K, int32_t act, void* stream);

/* Bring-up / profiling aid: one tcgen05 GEMM (GroupNorm epilogue when n_obj > 0) timed with CUDA events over
 * `reps` launches, plus per-role cycle counters of one traced launch: trace_host[256][8] uint64.
 * n_obj < 0 selects the channels-on-lanes kernel for |n_obj| objects per scene; the caller then passes the weight
 * rows in that kernel's order (stored row 32b+l = channel 32b + 8(l%4) + l/4).  With gamma_dev == NULL it runs as a
 * plain GEMM whose activation (0 none, 1 GELU, 2 SiLU) travels in bits 8.. of `reps`. */
DS_API int ds_test_gemm_trace(const void* a_dev, const void* w_dev, const float* bias_dev, const void* res_dev,
                              void* d_dev, int32_t M, int32_t N, int32_t K, int32_t n_obj, const float* gamma_dev,
                              const float* beta_dev, int32_t reps, unsigned long long* trace_host, float* usec);

#ifdef __cplusplus
}
#endif
#endif /* DIFFUSCENE_B200_H_ */
