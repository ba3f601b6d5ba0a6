/* mipnerf_b200.h — C ABI of libmipnerf_b200.so: the B200 (sm_100a) Mip-NeRF per-ray hot path.
 *
 * The reference (hjxwhy/mipnerf_pl) has no FFI layer: its boundary for this path is the Python
 * call surface `MipNerf.forward` (models/mip_nerf.py:172-248) and the free functions it reaches in
 * models/mip.py.  Each entry point below names the reference function it replaces.  The host-side
 * mirror that binds these symbols (ctypes) is mipnerf_pl_b200/_cabi.py; INTEGRATION.md shows the
 * stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every pointer is a DEVICE pointer to row-major fp32 unless stated otherwise; the library never
 *     allocates or frees device memory and keeps no state besides the thread-local error string;
 *   - `stream` is a cudaStream_t passed as void*; all calls are asynchronous on it (no sync inside);
 *   - return value: 0 on success, negative MIPNERF_B200_E* on failure (`mipnerf_b200_last_error()`
 *     gives the text).  There is no CPU fallback anywhere behind this ABI.
 */
#ifndef MIPNERF_B200_H_
#define MIPNERF_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define MIPNERF_B200_ABI_VERSION 4

#define MIPNERF_B200_OK 0
#define MIPNERF_B200_EINVAL (-1)       /* bad argument (NULL pointer, negative size, ...)            */
#define MIPNERF_B200_EUNSUPPORTED (-2) /* config outside what the kernels implement                  */
#define MIPNERF_B200_ECUDA (-3)        /* a CUDA runtime call or launch failed                       */
#define MIPNERF_B200_EWORKSPACE (-4)   /* workspace smaller than mipnerf_b200_workspace_bytes()      */

/* Arithmetic the MLP contraction runs in (everything else on the path is always fp32).
 * FP32 takes any config check_config accepts.  The tensor-core precisions take the reference's shipped architecture:
 * 8x256 trunk with the skip after layer 4, one 128-wide view layer, num_samples = 128, use_viewdirs, min_deg_point = 0,
 * max_deg_point 1..16 and deg_view 1..4 (narrower encodings are zero-padded into the operand image by
 * mipnerf_b200_pack_weights); the tensor-core TRAINING step and mipnerf_b200_mlp_forward need max_deg_point = 16 and
 * deg_view = 4.  Anything else answers MIPNERF_B200_EUNSUPPORTED (mipnerf_b200_packed_weights_bytes() == 0). */
#define MIPNERF_B200_FP32 0 /* CUDA-core FFMA, fp32 operands: the 1e-4 parity mode                   */
#define MIPNERF_B200_BF16 1 /* tcgen05 kind::f16, bf16 operands, fp32 accumulate in TMEM             */
#define MIPNERF_B200_FP16 2 /* tcgen05 kind::f16, fp16 operands, fp32 accumulate in TMEM             */
/* Split-operand tensor-core modes: every GEMM operand x is carried as hi = fl16(x), lo = fl16(x - hi) and each
 * K step issues hi.hi + lo.hi + hi.lo into the same fp32 TMEM accumulator (3x the MMAs).  FP16X3 keeps 22
 * significant operand bits (|x| < 65504) and is the tensor-core mode that meets the reference's fp32 result
 * to 1e-4 (models/mip_nerf.py:94-110 computes every nn.Linear in fp32); BF16X3 keeps 16 bits with fp32's range. */
#define MIPNERF_B200_FP16X3 3
#define MIPNERF_B200_BF16X3 4

/* One torch.nn.Linear: weight [out_features, in_features] row-major, bias [out_features]. */
typedef struct mipnerf_b200_linear {
  const float* weight;
  const float* bias;
  int32_t in_features;
  int32_t out_features;
} mipnerf_b200_linear;

/* Constructor arguments of MipNerf that change the arithmetic (models/mip_nerf.py:117-141). */
typedef struct mipnerf_b200_config {
  int32_t num_samples; /* per level; CUDA path needs num_samples % 32 == 0 and <= 256               */
  int32_t num_levels;
  int32_t min_deg_point, max_deg_point, deg_view;
  int32_t use_viewdirs, disparity, disable_integration;
  float resample_padding, density_bias, rgb_padding;
  int32_t net_depth, net_width, net_depth_condition, net_width_condition, skip_index;
  int32_t num_rgb_channels, num_density_channels; /* must be 3 and 1                                */
  float density_noise; /* std of the Gaussian noise added to raw density when randomized (models/mip_nerf.py:232-233) */
} mipnerf_b200_config;

/* MLP parameters in state_dict order (models/mip_nerf.py:19-73):
 * layers.0 .. layers.{net_depth-1}, density_layer, extra_layer, view_layers.0 .. , color_layer.
 * `packed` is the optional tensor-core operand image written by mipnerf_b200_pack_weights. */
typedef struct mipnerf_b200_weights {
  const mipnerf_b200_linear* linears;
  int32_t num_linears;
  int32_t packed_precision; /* MIPNERF_B200_BF16/FP16 the image was packed for, or -1              */
  const void* packed;
  size_t packed_bytes;
} mipnerf_b200_weights;

/* Rays namedtuple fields used by forward (datasets/datasets.py:13-16; lossmult is not read). */
typedef struct mipnerf_b200_rays {
  const float* origins;    /* [B,3] */
  const float* directions; /* [B,3] not normalised */
  const float* viewdirs;   /* [B,3] */
  const float* radii;      /* [B,1] */
  const float* near;       /* [B,1] */
  const float* far;        /* [B,1] */
  int64_t num_rays;
} mipnerf_b200_rays;

/* One element of the list MipNerf.forward returns (models/mip_nerf.py:246). */
typedef struct mipnerf_b200_level_out {
  float* comp_rgb;  /* [B,3]            */
  float* distance;  /* [B]              */
  float* acc;       /* [B]              */
  float* weights;   /* [B,N]   nullable */
  float* t_samples; /* [B,N+1] nullable */
  int64_t* inds;    /* [B,N+1] nullable; searchsorted indices of the resampler (levels >= 1)       */
  /* INPUT, nullable: [B,N] standard-normal draws replacing torch.randn of models/mip_nerf.py:233 for this level.
   * Read only when randomized != 0 and cfg->density_noise > 0; required then by the entry points that take injected
   * noise (t_rand / u_jitter), ignored by the _rng entry points (in-kernel Philox + Box-Muller, stream 32 + level). */
  const float* density_normal;
} mipnerf_b200_level_out;

/* In-kernel random numbers for randomized=True: Philox4x32-10 keyed by `seed`; the draw of (ray, index, stream) is a
 * pure function of (seed, offset, ray's position in the call), so results do not depend on chunking.  Advance `offset`
 * by one per call for fresh noise (the role of torch's generator offset). */
typedef struct mipnerf_b200_rng {
  uint64_t seed;
  uint64_t offset;
} mipnerf_b200_rng;

const char* mipnerf_b200_last_error(void);
int mipnerf_b200_abi_version(void);

/* Bytes of scratch `mipnerf_b200_forward` / `mipnerf_b200_mlp_forward` need for `num_rays` rays. */
size_t mipnerf_b200_workspace_bytes(const mipnerf_b200_config* cfg, int64_t num_rays, int precision);

/* Size of / builder for the tensor-core operand image of the MLP weights (device -> device). */
size_t mipnerf_b200_packed_weights_bytes(const mipnerf_b200_config* cfg, int precision);
int mipnerf_b200_pack_weights(const mipnerf_b200_config* cfg, const mipnerf_b200_weights* w,
                              int precision, void* packed_out, size_t packed_bytes, void* stream);

/* MipNerf.forward (models/mip_nerf.py:172-248).  `t_rand` [B,N+1] in [0,1) and `u_jitter`
 * [B,N+1] in [0, 1/(N+1)-eps) replace torch.rand / uniform_ (models/mip.py:159, :201-202) when
 * `randomized` != 0 (both required then).  `outs` has cfg->num_levels entries. */
int mipnerf_b200_forward(const mipnerf_b200_config* cfg, const mipnerf_b200_weights* w,
                         const mipnerf_b200_rays* rays, int randomized, const float* t_rand,
                         const float* u_jitter, int white_bkgd, int precision,
                         mipnerf_b200_level_out* outs, void* workspace, size_t workspace_bytes,
                         void* stream);

/* Same, drawing the uniforms of randomized mode INSIDE the kernels that consume them (no torch.rand launch, no
 * [B,N+1] arrays in HBM): stream 0 = the stratified draws of sample_along_rays (models/mip.py:159), stream 1+l =
 * the inverse-CDF jitter of level l (models/mip.py:201-202, scaled to [0, 1/(N+1) - eps)). */
int mipnerf_b200_forward_rng(const mipnerf_b200_config* cfg, const mipnerf_b200_weights* w,
                             const mipnerf_b200_rays* rays, const mipnerf_b200_rng* rng, int white_bkgd,
                             int precision, mipnerf_b200_level_out* outs, void* workspace,
                             size_t workspace_bytes, void* stream);

/* The uniforms those kernels draw: out[num_rays, ncols] for `stream_id` (0: t_rand in [0,1); >= 1: u_jitter in
 * [0, 1/ncols - eps)).  forward(t_rand = stream 0, u_jitter = stream 1+level) reproduces forward_rng bit for bit. */
int mipnerf_b200_philox_uniform(const mipnerf_b200_rng* rng, int stream_id, int64_t num_rays, int ncols, float* out,
                                void* stream);
/* The standard normals the _rng entry points add (times cfg->density_noise) to the raw density of level `level`
 * (models/mip_nerf.py:232-233): out[num_rays, num_samples].  Passed as outs[level].density_normal to the injected-
 * noise entry points they reproduce the in-kernel draws bit for bit. */
int mipnerf_b200_philox_normal(const mipnerf_b200_rng* rng, int level, int64_t num_rays, int num_samples, float* out,
                               void* stream);

/* distloss (models/mip.py:8-20), forward value per ray: weights [B,N], samples [B,N+1] (sorted) ->
 * per_ray_loss [B] = (1/3) sum_i d_i w_i^2 + sum_ij w_i w_j |m_i - m_j|; the reference's scalar is its mean. */
int mipnerf_b200_distloss(const float* weights, const float* samples, int64_t num_rays, int num_samples,
                          float* per_ray_loss, void* stream);

/* ---- training step (SURVEY.md §8f N2) -------------------------------------------------------------
 * Gradient buffers, one per entry of mipnerf_b200_weights.linears (same order and shapes). */
typedef struct mipnerf_b200_linear_grad {
  float* weight_grad; /* [out_features, in_features] */
  float* bias_grad;   /* [out_features]              */
} mipnerf_b200_linear_grad;

/* The loss of MipNeRFSystem.training_step (models/nerf_system.py:95-121):
 *   loss = sum_l  level_mse_mult[l] * sum_r mask_r |comp_rgb_l,r - target_r|^2 / mask_sum
 *               + level_dist_mult[l] * dist_scale * sum_r distloss_l,r
 * (reference: mse_mult = {coarse_loss_mult, 1}, dist_mult = {0.01*coarse_loss_mult, 0.01},
 * mask = rays.lossmult or ones, dist_scale = 1/B: the .mean() of models/mip.py:16,19).
 * `mask_sum` and `dist_scale` are over the GLOBAL batch so that ray shards of one batch (chunks, ranks)
 * produce gradients that simply add up. */
typedef struct mipnerf_b200_loss {
  const float* target_rgb;      /* [B,3] device                                                      */
  const float* lossmult;        /* [B] device, or NULL for a mask of ones                            */
  const float* mask_sum;        /* device scalar                                                     */
  float dist_scale;
  const float* level_mse_mult;  /* HOST [num_levels]                                                 */
  const float* level_dist_mult; /* HOST [num_levels]                                                 */
  float* per_ray_sqerr;         /* [num_levels, B] device, nullable: mask_r |comp_rgb - target|^2    */
  float* per_ray_distloss;      /* [num_levels, B] device, nullable                                  */
} mipnerf_b200_loss;

size_t mipnerf_b200_train_workspace_bytes(const mipnerf_b200_config* cfg, int64_t num_rays);

/* MipNerf.forward (outputs in `outs`, as mipnerf_b200_forward) followed by the backward pass of the loss
 * above into `grads` (overwritten, or added to when `accumulate` != 0).  Replaces
 * `loss = training_step(...); loss.backward()` (models/nerf_system.py:95-121 + autograd).  Fenceposts carry
 * no gradient (stop_resample_grad=True semantics, models/mip.py:250-264).  precision FP32: every GEMM in fp32 FFMA
 * (the parity mode); BF16 / FP16: forward and dgrad GEMMs on tcgen05 with 16-bit operands, wgrad / heads / rendering
 * in fp32 (default 8x256 architecture only). */
int mipnerf_b200_forward_backward(const mipnerf_b200_config* cfg, const mipnerf_b200_weights* weights,
                                  const mipnerf_b200_rays* rays, int randomized, const float* t_rand,
                                  const float* u_jitter, int white_bkgd, int precision,
                                  const mipnerf_b200_loss* loss, mipnerf_b200_level_out* outs,
                                  const mipnerf_b200_linear_grad* grads, int num_grads, int accumulate,
                                  void* workspace, size_t workspace_bytes, void* stream);
/* randomized=True training step with the in-kernel generator (what a training loop calls every step). */
int mipnerf_b200_forward_backward_rng(const mipnerf_b200_config* cfg, const mipnerf_b200_weights* weights,
                                      const mipnerf_b200_rays* rays, const mipnerf_b200_rng* rng, int white_bkgd,
                                      int precision, const mipnerf_b200_loss* loss, mipnerf_b200_level_out* outs,
                                      const mipnerf_b200_linear_grad* grads, int num_grads, int accumulate,
                                      void* workspace, size_t workspace_bytes, void* stream);
/* The same with (seed, offset) read from DEVICE memory (`rng_state` = uint64_t[2]) when the kernels run, so that a
 * CUDA graph that captured this call draws fresh numbers after the caller advances rng_state[1]: the draws equal
 * forward_backward_rng's for the same values.  BF16 / FP16 fused step only (EUNSUPPORTED otherwise). */
int mipnerf_b200_forward_backward_rng_state(const mipnerf_b200_config* cfg, const mipnerf_b200_weights* weights,
                                            const mipnerf_b200_rays* rays, const uint64_t* rng_state, int white_bkgd,
                                            int precision, const mipnerf_b200_loss* loss, mipnerf_b200_level_out* outs,
                                            const mipnerf_b200_linear_grad* grads, int num_grads, int accumulate,
                                            void* workspace, size_t workspace_bytes, void* stream);

/* Stand-alone tensor-core linear layer  y[m,n] = act(x[m,k] . weight[n,k]^T + bias)  (tcgen05, 16-bit operands, fp32
 * accumulate; n in {128,256}, k in {96,128,256}): the GEMM the training step uses for its forward and dgrad passes in
 * BF16 / FP16 mode.  `scratch` receives the packed weight image (n * ceil(k/64) * 128 bytes). */
int mipnerf_b200_linear_tc(const float* x, const float* weight, const float* bias, float* y, int64_t m, int n,
                           int k, int relu, int precision, void* scratch, size_t scratch_bytes, void* stream);

/* Stand-alone tensor-core weight gradient of one nn.Linear (what loss.backward() accumulates into layer.weight.grad /
 * layer.bias.grad, models/nerf_system.py:108-111):  dw[n, k1+k2] = dy[m,n]^T . [x1[m,k1] | x2[m / x2_row_div, k2]],
 * db[n] = column sums of dy; n in {128,256}, 16-bit operands rounded while staging, fp32 accumulation, per-slice
 * partials reduced in a fixed order (bit-reproducible).  x2 may be NULL (k2 = 0). */
size_t mipnerf_b200_wgrad_tc_scratch_bytes(int n, int k);
int mipnerf_b200_wgrad_tc(const float* dy, int n, const float* x1, int k1, const float* x2, int k2, int x2_row_div,
                          int64_t m, float* dw, float* db, int precision, void* scratch, size_t scratch_bytes,
                          void* stream);

/* torch.optim.Adam.step() for one flat fp32 tensor (models/nerf_system.py:70-72; amsgrad off, no weight
 * decay): `step` is the 1-based step count after this update; the gradient is read as grad * grad_scale
 * (1/world_size after a sum all-reduce). */
int mipnerf_b200_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                           double lr, double beta1, double beta2, double eps, int64_t step, double grad_scale,
                           void* stream);
/* The same update for `count` tensors that share lr / betas / eps / step (one optimiser group) in ONE launch; the
 * arrays are host arrays of device pointers / element counts. */
int mipnerf_b200_adam_step_multi(int count, float* const* params, const float* const* grads, float* const* exp_avg,
                                 float* const* exp_avg_sq, const int64_t* sizes, double lr, double beta1, double beta2,
                                 double eps, int64_t step, double grad_scale, void* stream);
/* adam_step_multi with the step count on the device: the update number is t = *step + 1 and the step size lr_t / bc1_t
 * and sqrt(bc2_t) are read from the DEVICE tables step_size[t] / bc2_sqrt[t] (t clamped to 1 .. table_len - 1), which
 * the caller fills with the double-precision math of adam_step_multi; *step is not changed. */
int mipnerf_b200_adam_step_multi_table(int count, float* const* params, const float* const* grads,
                                       float* const* exp_avg, float* const* exp_avg_sq, const int64_t* sizes,
                                       const float* step_size, const float* bc2_sqrt, int64_t table_len,
                                       const int64_t* step, double beta1, double beta2, double eps, double grad_scale,
                                       void* stream);
/* End of a device-driven training step: ring[(*step % ring_len) * 2 + {0, 1}] = {*loss, *psnr} (ring_len may be 0),
 * then *step += 1 and rng_state[1] += 1.  All pointers are device pointers. */
int mipnerf_b200_train_step_advance(int64_t* step, uint64_t* rng_state, const float* loss, const float* psnr,
                                    float* ring, int ring_len, void* stream);

/* Pinhole rays of rows [row0,row0+rows) of an H x W frame generated on the device, replacing the
 * host NumPy loaders (datasets/datasets.py:214-263, render_video.py:29-105).  `c2w_host` is a HOST
 * pointer to the row-major [3,4] camera-to-world matrix; outputs are [rows*W, 3|1] device buffers. */
int mipnerf_b200_generate_rays(const float* c2w_host, int height, int width, float focal, float near,
                               float far, int row0, int rows, float* origins, float* directions,
                               float* viewdirs, float* radii, float* near_out, float* far_out,
                               void* stream);

/* eval_errors (utils/metrics.py:190-197) of one rendered frame: pred / target [H, W, C] fp32 row-major (the layout
 * render_image produces) -> out[0] = PSNR = -10 log10(mean squared error) (utils/metrics.py:182-188), out[1] = mean
 * SSIM with the reference's 11x11 Gaussian window (sigma 1.5, zero padding, C1 = 0.01^2, C2 = 0.03^2; :44-126),
 * out[2] = the mean squared error.  `scratch`: mipnerf_b200_image_metrics_scratch_bytes() bytes. */
size_t mipnerf_b200_image_metrics_scratch_bytes(int height, int width, int channels);
int mipnerf_b200_image_metrics(const float* pred, const float* target, int height, int width, int channels,
                               void* scratch, size_t scratch_bytes, float* out, void* stream);

/* Training rays from pixel ids, scene resident in HBM (replaces the per-pixel host arrays of
 * datasets/datasets.py:116-168, 216-263 and the DataLoader's H2D copies, SURVEY.md §8f N4):
 *   cam_table [num_images, 24] = pix2cam (3x3 row-major, maps (x+.5, y+.5, 1) to a camera direction) |
 *                                cam2world (3x4 row-major) | lossmult | near | far
 *   offsets [num_images+1] first atlas row of each image; widths [num_images]; atlas [P,3] target colours
 *   pixel_ids [count] atlas rows (ids outside [0, offsets[num_images]) are clamped to the first / last row)
 *   -> the seven Rays fields ([count,3|1]) and rgb [count,3] (nullable). */
int mipnerf_b200_rays_from_pixels(const float* cam_table, const int64_t* offsets, const int32_t* widths,
                                  int num_images, const int64_t* pixel_ids, int64_t count, const float* atlas,
                                  float* origins, float* directions, float* viewdirs, float* radii,
                                  float* lossmult, float* near_out, float* far_out, float* rgb, void* stream);
/* A uniformly random batch of `count` training rays drawn on the device, then rays_from_pixels on it: the id of ray i is
 * floor(x * num_pixels / 2^32), x the first 32-bit output of Philox4x32-10 keyed like the in-kernel draws by
 * rng_state = DEVICE uint64_t[2] (seed, offset) with counter (ray_base + i, stream 64, offset).  1 <= num_pixels <= 2^32;
 * each id's probability is within 2^-32 of 1/num_pixels.  Ids past offsets[num_images] (num_pixels larger than the
 * atlas) are clamped to its last row.  pixel_ids [count] (nullable) receives the ids. */
int mipnerf_b200_sample_pixels(const float* cam_table, const int64_t* offsets, const int32_t* widths, int num_images,
                               int64_t num_pixels, const uint64_t* rng_state, int64_t ray_base, int64_t count,
                               const float* atlas, int64_t* pixel_ids, float* origins, float* directions,
                               float* viewdirs, float* radii, float* lossmult, float* near_out, float* far_out,
                               float* rgb, void* stream);

/* ---- per-stage entry points (unit parity against the functions of models/mip.py) ---- */

/* sample_along_rays (models/mip.py:127-165): t_samples [B,N+1], means/covs [B,N,3] (nullable). */
int mipnerf_b200_sample_along_rays(const mipnerf_b200_rays* rays, int num_samples, int randomized,
                                   int disparity, const float* t_rand, float* t_samples,
                                   float* means, float* covs, void* stream);

/* cast_rays, cone + diagonal (models/mip.py:81-103): t_samples [B,N+1] -> means, covs [B,N,3]. */
int mipnerf_b200_cast_rays(const mipnerf_b200_rays* rays, const float* t_samples, int num_samples,
                           float* means, float* covs, void* stream);

/* integrated_pos_enc, diagonal (models/mip.py:322-350): means, covs [M,3] -> out [M, 6*(max-min)]. */
int mipnerf_b200_integrated_pos_enc(const float* means, const float* covs, int64_t num_points,
                                    int min_deg, int max_deg, float* out, void* stream);

/* pos_enc (models/mip.py:353-363): x [B,3] -> out [B, 6*(max-min) (+3)]. */
int mipnerf_b200_pos_enc(const float* x, int64_t num_points, int min_deg, int max_deg,
                         int append_identity, float* out, void* stream);

/* MLP.forward (models/mip_nerf.py:75-111): x [B*N, xyz_dim], view_enc [B, view_dim] or NULL ->
 * raw_rgb [B*N,3], raw_density [B*N,1]. */
int mipnerf_b200_mlp_forward(const mipnerf_b200_config* cfg, const mipnerf_b200_weights* w,
                             const float* x, const float* view_enc, int64_t num_rays,
                             int samples_per_ray, int precision, float* raw_rgb, float* raw_density,
                             void* workspace, size_t workspace_bytes, void* stream);

size_t mipnerf_b200_mlp_workspace_bytes(const mipnerf_b200_config* cfg, int64_t num_rays,
                                        int samples_per_ray, int precision);

/* volumetric_rendering (models/mip.py:366-401): rgb [B,N,3], density [B,N,1] already activated. */
int mipnerf_b200_volumetric_rendering(const float* rgb, const float* density,
                                      const float* t_samples, const float* dirs, int64_t num_rays,
                                      int num_samples, int white_bkgd, float* comp_rgb,
                                      float* distance, float* acc, float* weights, void* stream);

/* sorted_piecewise_constant_pdf (models/mip.py:168-229): bins [B,nb+1], weights [B,nb] (NOT
 * modified) -> samples [B,num_samples]; inds (nullable) are the searchsorted(right=True) results. */
int mipnerf_b200_sorted_piecewise_constant_pdf(const float* bins, const float* weights,
                                               int64_t num_rays, int num_bins, int num_samples,
                                               int randomized, const float* u_jitter,
                                               float* samples, int64_t* inds, void* stream);

/* resample_along_rays (models/mip.py:232-280): blur-pool + padding + inverse CDF + cast_rays. */
int mipnerf_b200_resample_along_rays(const mipnerf_b200_rays* rays, const float* t_samples,
                                     const float* weights, int num_samples, int randomized,
                                     const float* u_jitter, float resample_padding,
                                     float* new_t_samples, float* means, float* covs, int64_t* inds,
                                     void* stream);

/* Hardware self-test of the tcgen05 building blocks (descriptor / swizzle / TMEM conventions):
 * d[128,n] = a[128,k] . b[n,k]^T, 16-bit operands (precision BF16|FP16), fp32 accumulate in TMEM.
 * variant bit 0: B through a pre-swizzled image + cp.async.bulk (needs `scratch`); bit 1: A in TMEM. */
int mipnerf_b200_selftest_umma(const float* a, const float* b, float* d, int n, int k, int precision,
                               int variant, void* scratch, size_t scratch_bytes, void* stream);
/* Issue-rate microbenchmark of tcgen05.mma (M = 128, N = n in {128, 256}, K = 16) on resident operands: `ctas` CTAs each
 * issue iters x 16 MMAs and write their clock64 cycle count to cycles[cta] (device memory).  mode 0: SS form, A as
 * 128-byte-swizzle slabs; 1: SS form, A as dense 32-byte-swizzle K = 16 blocks; 2: TS form, A in tensor memory. */
int mipnerf_b200_selftest_umma_rate(int mode, int n, int iters, int precision, int ctas, long long* cycles, void* stream);
/* The same for CTA pairs (cta_group::2, M = 256 over two SMs, n / 2 rows of B per CTA); mode 0 (SS) or 2 (TS);
 * cycles[pair]. */
int mipnerf_b200_selftest_umma_rate_pair(int mode, int n, int iters, int precision, int pairs, long long* cycles,
                                         void* stream);

/* ---- launch accounting (bench.py: `gpu_launches`, live launch duration of the dominant kernel) ----
 * Every kernel launch of the library is counted per kernel id; with timing enabled each launch is
 * also bracketed by CUDA events on its stream.  profile_read synchronises the pending events. */
int mipnerf_b200_profile_enable(int timing_on);
int mipnerf_b200_profile_num_kernels(void);
const char* mipnerf_b200_profile_kernel_name(int kernel_id);
int mipnerf_b200_profile_read(int kernel_id, int64_t* launches, double* timed_ms,
                              int64_t* timed_launches, int reset);

#ifdef __cplusplus
}
#endif
#endif /* MIPNERF_B200_H_ */
