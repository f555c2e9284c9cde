/* nerfies_b200.h - C ABI of the B200-native deformable-NeRF render hot path.
 *
 * The reference (google/nerfies) is pure Python/JAX and has no FFI; the seam a
 * replacement plugs into is the Python call surface listed in SURVEY.md §8(b).
 * Each entry point below names the reference callable it replaces
 * (file:line in /root/reference).  The Python host side
 * (nerfies_b200/models.py, evaluation.py) binds these with ctypes and keeps the
 * reference's names / pytree keys / shapes on top.
 *
 * Conventions
 *  - every pointer is a DEVICE pointer on the current CUDA device unless the
 *    function name ends in _host; tensors are contiguous, row-major, float32;
 *    ids are uint32;
 *  - calls enqueue work on `stream` (a cudaStream_t passed as void*) and return
 *    without synchronising (the *_host variant synchronises before returning);
 *  - the caller owns every input/output buffer and keeps it alive until the
 *    stream has passed the call; the library owns only its workspace, allocated
 *    in nfb_create; nothing is allocated on the hot path;
 *  - return value 0 = success, < 0 = error (message via nfb_last_error());
 *  - the tensor-core kernels never hang or trap on an internal protocol error:
 *    a bounded mbarrier wait raises a process-wide abort flag (mapped host
 *    memory), the kernel drains, and the _host entry point / every later call
 *    returns an error ("a tcgen05 kernel aborted ..."); results of that launch
 *    are invalid;
 *  - a handle is not thread-safe: one handle per GPU per process/rank.  Its workspace
 *    is shared by its calls: consecutive calls on one stream are ordered by the
 *    stream; when a call arrives on a different stream than the previous one the
 *    library makes the new stream wait for the previous call's work (one event).
 *    Concurrent launches from one handle on two streams are therefore serialised,
 *    not run in parallel - use one handle per stream for that.
 */
#ifndef NERFIES_B200_H_
#define NERFIES_B200_H_

#ifdef __cplusplus
extern "C" {
#endif

typedef struct nfb_handle nfb_handle;

/* Activation selectors: configs.py:27-32 registers exactly these for gin. */
enum nfb_activation {
  NFB_ACT_NONE = 0, NFB_ACT_RELU = 1, NFB_ACT_ELU = 2, NFB_ACT_LEAKY_RELU = 3,
  NFB_ACT_TANH = 4, NFB_ACT_SIGMOID = 5, NFB_ACT_SOFTPLUS = 6
};
enum nfb_warp_type { NFB_WARP_NONE = 0, NFB_WARP_TRANSLATION = 1, NFB_WARP_SE3 = 2 };
/* warp_metadata_encoder_type (configs.py:103; warping.py:109-123, 250-260):
 * GLO   = GloEncoder on metadata['warp'] ids;
 * TIME  = modules.TimeEncoder (modules.py:297-322) on metadata['time'], annealed by
 *         warp_extra['time_alpha'];
 * BLEND = (1 - time_alpha) * glo(id) + time_alpha * TimeEncoder(float(id)) (warping.py:128-133). */
enum nfb_warp_encoder { NFB_WARP_ENC_GLO = 0, NFB_WARP_ENC_TIME = 1, NFB_WARP_ENC_BLEND = 2 };
/* Arithmetic of the MLP GEMMs.  Everything else is always fp32. */
enum nfb_precision {
  NFB_PREC_FP32 = 0,     /* fp32 FFMA on CUDA cores: general (any width / activation / condition) */
  NFB_PREC_BF16 = 1,     /* bf16 operands, fp32 accumulate, tcgen05 tensor cores: fastest, ~1e-2  */
  NFB_PREC_FP16X3 = 2    /* fp32 emulated on tcgen05 by three fp16 MMA chains into one fp32
                          * accumulator (x_hi W_hi + x_lo W_hi + x_hi W_lo, hi = fp16(v),
                          * lo = fp16(v - hi): 22 significant bits per operand): the
                          * tensor-core mode that holds the 1e-4 parity gate.  Activations
                          * beyond fp16's range (|v| > 65504) saturate.  (Round 1 reserved this
                          * value as "bf16x3"; a bf16 split leaves 2^-17 per operand, not enough.) */
};

/* Mirrors the NerfModel attributes that shape the forward pass
 * (nerfies/models.py:76-120; filled from ModelConfig, nerfies/configs.py:37-105). */
typedef struct nfb_config {
  int num_coarse_samples;        /* ModelConfig.num_coarse_samples              */
  int num_fine_samples;          /* ModelConfig.num_fine_samples (0: no fine)   */
  int num_nerf_point_freqs;      /* SinusoidalEncoder F for points (models.py:148) */
  int num_nerf_viewdir_freqs;    /* ... for viewdirs (models.py:151)            */
  int num_warp_freqs;            /* AnnealedSinusoidalEncoder F (warping.py:245) */
  int nerf_trunk_depth, nerf_trunk_width;
  int nerf_rgb_branch_depth, nerf_rgb_branch_width;
  unsigned nerf_skips_mask;      /* bit i set <=> i in nerf_skips (modules.py:47) */
  int alpha_channels, rgb_channels;   /* must be 1 and 3                        */
  int warp_field_type;           /* nfb_warp_type; NONE when use_warp is False  */
  int warp_trunk_depth, warp_trunk_width;   /* SE3Field/TranslationField MLP    */
  unsigned warp_skips_mask;
  int num_warp_features, num_appearance_features, num_camera_features;
  int num_warp_embeddings, num_appearance_embeddings, num_camera_embeddings;
  int use_viewdirs, use_appearance_metadata, use_camera_metadata;
  int use_trunk_condition, use_alpha_condition, use_rgb_condition;
  int activation;                /* hidden activation of NerfMLP (nfb_activation) */
  int sigma_activation;          /* models.py:277                               */
  int use_white_background, use_linear_disparity, use_sample_at_infinity;
  float near_plane, far_plane;   /* NerfModel.near / .far                       */
  int precision;                 /* nfb_precision                               */
  /* warp-field variants (warping.py:84-123, 233-260, 242-243, 339-352) */
  int warp_metadata_encoder;     /* nfb_warp_encoder: glo | time | blend (TranslationField only) */
  int time_encoder_num_freqs;    /* warp_kwargs['metadata_encoder_num_freqs'] (TimeEncoder posenc) */
  int warp_use_pivot;            /* SE3Field(use_pivot=True): branches_p          */
  int warp_use_translation;      /* SE3Field(use_translation=True): branches_t    */
} nfb_config;

/* Flags for the render entry points. */
#define NFB_FLAG_COARSE_ONLY 1u  /* stop after the coarse level                 */
#define NFB_FLAG_NO_WARP     2u  /* use_warp=False call-time override (models.py:321) */
#define NFB_FLAG_METADATA_ENCODED 4u /* metadata_encoded=True (models.py:198-213,251;
                                      * warping.py:186-187): warp_id / app_id / cam_id are
                                      * reinterpreted as const float* per-ray embeddings of
                                      * shape (B, num_warp_features) / (B, num_appearance_features) /
                                      * (B, num_camera_features) and used instead of the GLO
                                      * table rows.  Device entry points only. */

/* Lifetime.  Replaces construct_nerf's model construction (models.py:424-463);
 * max_rays bounds B of every later call (workspace is sized once, here). */
int nfb_create(const nfb_config* cfg, int max_rays, nfb_handle** out);
void nfb_destroy(nfb_handle* h);

/* Parameter interface.  The expected tensors, in order, with their Flax names
 * ("warp_field/trunk/hidden_0/kernel", ... SURVEY.md §8a R12) and (rows, cols);
 * Dense kernels are (in, out), biases (1, out), embeddings (num, features). */
int nfb_param_count(const nfb_handle* h);
int nfb_param_info(const nfb_handle* h, int index, char* name, int name_capacity,
                   long long* rows, long long* cols);
/* Copies/repacks the fp32 tensors (device pointers, order of nfb_param_info)
 * into the library's padded layouts.  Replaces passing {'params': params} to
 * model.apply (models.py:289; eval.py:331). */
int nfb_set_params(nfb_handle* h, const float* const* tensors,
                   const long long* numels, int count, void* stream);

/* NerfModel.__call__ (nerfies/models.py:289-375): coarse level, hierarchical
 * resampling, fine level.
 *   origins, directions, viewdirs : (B,3); viewdirs NULL = directions (:326-329)
 *   warp_id, appearance_id, camera_id : (B) uint32 = metadata[...][:,0]; NULL
 *       allowed when the model does not use that metadata
 *   warp_alpha : warp_extra['alpha'] (model_utils.py:31-33)
 *   t_rand (B,Nc), u_rand (B,Nf) : the uniform draws of the stratified path
 *       (model_utils.py:65,162); NULL = deterministic path (:67-70, :164-165)
 *   out_coarse, out_fine : (B,6) = rgb[3], depth, med_depth, acc
 *   w_coarse (B,Nc), w_fine (B,Nc+Nf), z_fine (B,Nc+Nf) : optional outputs */
int nfb_render_forward(nfb_handle* h, int num_rays, const float* origins,
                       const float* directions, const float* viewdirs,
                       const unsigned* warp_id, const unsigned* appearance_id,
                       const unsigned* camera_id, float warp_alpha,
                       const float* t_rand, const float* u_rand, unsigned flags,
                       float* out_coarse, float* out_fine, float* w_coarse,
                       float* w_fine, float* z_fine, void* stream);

/* warp_extra['time_alpha'] (model_utils.py:31-33; modules.py:317-320) for the
 * TIME / BLEND warp metadata encoders; persists on the handle until changed
 * (default 0).  With NFB_WARP_ENC_TIME the `warp_id` argument of the render / warp
 * entry points is reinterpreted as const float* metadata['time'] (B). */
int nfb_set_time_alpha(nfb_handle* h, float time_alpha);

/* Same call with HOST buffers: stages inputs through pinned memory, H2D,
 * renders, D2H, synchronises.  This is what render_image's model_fn does per
 * chunk in the reference (evaluation.py:85-93: shard -> model_fn -> unshard). */
int nfb_render_forward_host(nfb_handle* h, int num_rays, const float* origins,
                            const float* directions, const float* viewdirs,
                            const unsigned* warp_id,
                            const unsigned* appearance_id,
                            const unsigned* camera_id, float warp_alpha,
                            unsigned flags, float* out_coarse, float* out_fine,
                            void* stream);

/* NerfModel.render_samples (nerfies/models.py:230-287) for one level
 * (0 = coarse MLP, 1 = fine MLP) on caller-supplied z_vals (B,S), points =
 * origins + z * directions.  out (B,6); optional weights (B,S), per-sample
 * sigmoid(rgb)/sigma (B,S,4) and warped_points (B,S,3). */
int nfb_render_samples(nfb_handle* h, int level, int num_rays, int num_samples,
                       const float* z_vals, const float* origins,
                       const float* directions, const float* viewdirs,
                       const unsigned* warp_id, const unsigned* appearance_id,
                       const unsigned* camera_id, float warp_alpha,
                       unsigned flags, float* out, float* weights,
                       float* samples, float* warped_points, void* stream);

/* model_utils.sample_pdf (nerfies/model_utils.py:190-215) with the caller prep
 * of models.py:353-357: bins = midpoints of z_coarse, weights = w_coarse[1:-1];
 * z_fine = sort(concat(z_coarse, inverse-CDF samples)). */
int nfb_sample_pdf(nfb_handle* h, int num_rays, const float* z_coarse,
                   const float* w_coarse, const float* u_rand, float* z_fine,
                   void* stream);

/* model_utils.sample_along_rays z_vals (nerfies/model_utils.py:56-70). */
int nfb_coarse_z_vals(nfb_handle* h, int num_rays, const float* t_rand,
                      float* z_coarse, void* stream);

/* warp_field.apply on free points (nerfies/warping.py:355-389, 160-199; called
 * by training.py:122-131): points (P,3), warp_id (P) -> warped (P,3). */
int nfb_warp_forward(nfb_handle* h, int num_points, const float* points,
                     const unsigned* warp_id, float warp_alpha, unsigned flags,
                     float* warped, void* stream);
/* flags: NFB_FLAG_METADATA_ENCODED = warp_field.apply(..., metadata_encoded=True)
 * (warping.py:186-187, 378): warp_id is (P, num_warp_features) float embeddings. */

/* ---- training tier (SURVEY §8(f) #1) ----------------------------------------------
 * jax.value_and_grad of the photometric loss of training.train_step
 * (training.py:171-175, 214-244, 263-264): loss = mean((rgb_coarse - target)^2) +
 * mean((rgb_fine - target)^2) over the batch, differentiated w.r.t. every model
 * parameter through NerfModel.__call__ (z_fine is a constant: lax.stop_gradient,
 * model_utils.py:211).  fp32, layer-wise with a tape in device memory, hand-written
 * SIMT GEMMs (csrc/train.cuh); uses the parameters of the last nfb_set_params.
 *   rgb_target (B,3); chunk_rays: rays per tape chunk (<= 0: 256);
 *   grads[i]: device tensor of the i-th parameter of nfb_param_info, rows*cols floats,
 *             ACCUMULATED into (+=): zero them first for a plain gradient;
 *   loss_out (device, 2 floats): the coarse and the fine loss.
 * Every warp metadata encoder trains; NFB_FLAG_METADATA_ENCODED is not supported.  `warp_id`:
 *   'glo'   (B) uint32 GLO ids;
 *   'time'  (B) float32 metadata['time'], as for nfb_render_forward (reinterpreted pointer);
 *   'blend' (B) uint32 GLO ids; the TimeEncoder sees float(id).
 * The 'time' / 'blend' encoders read warp_extra['time_alpha'] from nfb_set_time_alpha: the
 * TimeEncoder's window is cosine_easing_window(F, time_alpha) for 'time' and fully open for
 * 'blend', whose embedding is (1 - time_alpha) glo + time_alpha time (warping.py:128-133). */
int nfb_train_value_and_grad(nfb_handle* h, int num_rays, const float* origins,
                             const float* directions, const float* viewdirs,
                             const unsigned* warp_id, const unsigned* appearance_id,
                             const unsigned* camera_id, float warp_alpha,
                             const float* t_rand, const float* u_rand, unsigned flags,
                             const float* rgb_target, int chunk_rays, float* const* grads,
                             const long long* numels, int count, float* loss_out, void* stream);

/* Regularisers of training.train_step (training.py:138-147, 71-135, 176-212, 246-257). */
enum { NFB_ELASTIC_LOG_SVALS = 0, NFB_ELASTIC_SVALS = 1, NFB_ELASTIC_JTJ = 2, NFB_ELASTIC_DIV = 3,
       NFB_ELASTIC_DET = 4, NFB_ELASTIC_LOG_DET = 5 };
typedef struct nfb_train_reg {
  int use_elastic_loss;            /* training.py:143; applies to the coarse level (training.py:242-244) */
  int elastic_reduce_method;       /* 0 = 'median' (the median-depth sample of each ray), 1 = 'weight' */
  int elastic_loss_type;           /* NFB_ELASTIC_* = compute_elastic_loss's loss_type ('nr' unsupported) */
  float elastic_loss_weight;       /* ScalarParams.elastic_loss_weight */
  int use_warp_reg_loss;           /* training.py:147, both levels */
  float warp_reg_loss_weight, warp_reg_loss_alpha, warp_reg_loss_scale;
  int use_background_loss;         /* training.py:146 */
  int num_background_points;
  const float* background_points;        /* device (P,3): batch['background_points'] */
  const unsigned* background_warp_ids;   /* device (P) uint32 ids for EVERY encoder: the reference draws
                                            random.choice(key, model.warp_ids) and the 'time' encoder sees
                                            float(id) with alpha = time_alpha (training.py:121-131) */
  const float* background_noise;         /* device (P,3) or NULL: noise_std * random.normal(key, points.shape) */
  float background_loss_weight;          /* ScalarParams.background_loss_weight */
} nfb_train_reg;

/* nfb_train_value_and_grad plus the regularisers (reg may be NULL).  loss_out: 16 device floats
 *   [0] rgb loss coarse  [1] rgb loss fine  [2] loss/elastic  [3] residual/elastic
 *   [4] metric/jacobian_det  [5] metric/jacobian_div  [6] metric/jacobian_curl (means over the rows whose
 *   Jacobian the loss uses: the reference averages these three over every coarse sample, training.py:214-222)
 *   [7] loss/warp_reg coarse  [8] residual/warp_reg coarse  [9] loss/warp_reg fine  [10] residual fine
 *   [11] background loss (unweighted mean)  [12] mean |warped - x| of the background points.
 * The gradient is that of  rgb_coarse + rgb_fine + elastic_loss_weight * [2] + warp_reg_loss_weight *
 * ([7] + [9]) + background_loss_weight * [11]  (training.py:176-212, 228-259).  Replaces
 * jax.value_and_grad(_loss_fn) (training.py:263-264) with every regulariser of train_step. */
int nfb_train_value_and_grad_reg(nfb_handle* h, int B, const float* origins, const float* directions,
                                 const float* viewdirs, const unsigned* warp_id, const unsigned* app_id,
                                 const unsigned* cam_id, float warp_alpha, const float* t_rand,
                                 const float* u_rand, unsigned flags, const float* rgb_target,
                                 int chunk_rays, const nfb_train_reg* reg, float* const* grads,
                                 const long long* numels, int count, float* loss_out, void* stream);

/* Jacobian of the warp field at free points: jacobian_out (P,3,3), J[i][j] = d warped_i / d point_j
 * (jax.jacfwd(self.warp, argnums=0), warping.py:196-198, 385-387); warped_out (P,3) nullable.
 * warp_id (P) as for nfb_warp_forward: GLO ids, float32 timestamps for the 'time' encoder; the metadata
 * embedding is a constant of the Jacobian.  The warp MLP must use relu.  fp32, any precision mode of the
 * handle (layer-wise tape kernels). */
int nfb_warp_jacobian(nfb_handle* h, int P, const float* points, const unsigned* warp_id, float warp_alpha,
                      float* warped_out, float* jacobian_out, void* stream);

/* flax.optim.Adam.apply_gradient (training.py:268; beta1 0.9, beta2 0.999, eps 1e-8, no
 * weight decay are the Flax defaults the reference uses, train.py:219) on flat device
 * vectors of n floats; `step` counts from 1 (bias correction 1 - beta^step).  No handle. */
int nfb_adam_step(float* params, const float* grads, float* m, float* v, long long n,
                  float learning_rate, float beta1, float beta2, float eps, long long step,
                  void* stream);

/* Measurement aid (bench.py's roofline): when enabled, every launch of the field
 * kernel (the dominant kernel) is bracketed by cudaEvents on its launch stream.
 * nfb_field_time_ms synchronises on the events of the most recent launch of
 * `level` (0 coarse, 1 fine) and returns its duration in ms (< 0 on error). */
int nfb_set_profiling(nfb_handle* h, int enabled);
float nfb_field_time_ms(nfb_handle* h, int level);

/* ---- camera -> rays (SURVEY §8(f) row 3) ------------------------------------
 * Mirrors the fields of nerfies.camera.Camera (camera.py:110-137). */
typedef struct nfb_camera {
  float orientation[9];           /* world-to-camera rotation, row-major        */
  float position[3];
  float focal_length;
  float principal_point[2];
  float skew;
  float pixel_aspect_ratio;
  float radial_distortion[3];     /* k1 k2 k3                                   */
  float tangential_distortion[2]; /* p1 p2                                      */
  int image_size[2];              /* (width, height)                            */
} nfb_camera;

/* Replaces datasets/core.py:50-75 camera_to_rays (camera.py:317-321 pixel centres
 * + camera.py:244-269 pixels_to_rays) for the pixels [first_pixel,
 * first_pixel + count) of the frame in row-major order: origins (count,3) =
 * camera position, directions (count,3) unit, pixels (count,2) centres.
 * origins and pixels may be NULL.  Needs no handle. */
int nfb_camera_rays(const nfb_camera* cam, long long first_pixel, long long count,
                    float* origins, float* directions, float* pixels, void* stream);

/* Replaces Camera.pixels_to_rays (camera.py:244-269) for arbitrary float32 pixel
 * positions (n,2) -> unit world-space directions (n,3). */
int nfb_pixels_to_rays(const nfb_camera* cam, const float* pixels, long long n,
                       float* directions, void* stream);

/* Debug aid: block 0 of the tensor-core field kernel appends (tag, clock64)
 * pairs to `buffer` (device, 1 + 2*capacity int64; buffer[0] = record count,
 * zero it first).  NULL disables tracing.  Only builds compiled with -DNFB_TRACE
 * carry the tracer; others return -1 for a non-NULL buffer. */
int nfb_set_trace(nfb_handle* h, long long* buffer, int capacity);

/* Test hook for the abort path described in the conventions above: while enabled,
 * the MMA issuer of the bf16 tcgen05 kernel first waits on an mbarrier that never
 * completes, so the launch must time out, drain and raise the abort flag
 * (tests/test_edge_cases_gpu.py).  The process cannot run further tensor-core
 * launches afterwards.  No reference analogue. */
int nfb_debug_provoke_timeout(nfb_handle* h, int enabled);

/* The asynchronous entry points (nfb_render_forward, nfb_render_samples, nfb_warp_forward, ...) return
 * before their kernels finish, so a tensor-core kernel's protocol time-out (see the conventions above)
 * is only seen by a LATER call.  nfb_check_abort reports it for the work already submitted: with
 * synchronize != 0 it first waits for `stream`; returns 0 or < 0 (nfb_last_error).  nfb_reset_abort
 * waits for the device and clears the process-wide flag, after which launches are accepted again.
 * No reference analogue. */
int nfb_check_abort(void* stream, int synchronize);
int nfb_reset_abort(void);

/* Hardware self-test of the tcgen05 building blocks (UMMA descriptors, 128-byte
 * swizzle, TMEM, bulk-copy ring): C[128,N] = bf16(A[128,K]) x bf16(W[K,N]), fp32
 * accumulate.  K <= 320, N <= 256; device pointers. */
int nfb_selftest_gemm(int K, int N, const float* A, const float* W, float* C,
                      void* stream);

/* Micro-benchmark of the tensor pipe (mode 0: chain of tcgen05.mma M=128,N=n) or
 * of TMEM reads (mode 1: tcgen05.ld by `nwarps` warps).  out (host, 3 int64):
 * cycles, work items, issue cycles. */
int nfb_selftest_microbench(int mode, int n, int reps, int nwarps, long long* out);

/* CTA-pair (tcgen05 cta_group::2, a 2-CTA cluster) variant of nfb_selftest_gemm:
 * C (256 x N) = bf16(A (256 x K)) x bf16(W (K x N)) times `reps`, N in {64,128,256},
 * K <= 320.  out (host, 2 x int64, nullable): cycles seen by the leader CTA from
 * the first MMA issue to completion, and the number of MMAs (M=256, K=16) issued.
 * Hardware self-test / micro-benchmark for the planned 2-CTA field kernel; no
 * reference analogue. */
int nfb_selftest_gemm2(int K, int N, const float* A, const float* W, float* C, int reps,
                       long long* out, void* stream);

/* A-operand-in-TMEM form of tcgen05.mma, as the fp16x3 field kernel uses it:
 * C (128 x N) = A (128 x K) W (K x N) as three fp16 chains (A_hi W_hi + A_lo W_hi +
 * A_hi W_lo, fp32 accumulate), both fp16 images of A written to tensor memory with
 * tcgen05.st, W from shared memory.  K <= 256, N <= 256; `reps` repeats the chains
 * (the result is divided by reps).  out (host, 2 x int64, nullable): cycles from the
 * first issue to completion, number of MMAs.  Hardware self-test; no reference analogue. */
int nfb_selftest_gemm3(int K, int N, const float* A, const float* W, float* C, int reps,
                       long long* out, void* stream);

/* Number of CUDA kernels this handle has launched so far (bench accounting). */
long long nfb_kernel_launches(const nfb_handle* h);
/* Thread-local description of the last error returned on this thread. */
const char* nfb_last_error(void);
/* "nerfies_b200 <version> sm_100a" */
const char* nfb_version(void);

#ifdef __cplusplus
}
#endif
#endif  /* NERFIES_B200_H_ */
