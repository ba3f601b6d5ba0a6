// kernels.h — internal (C++) launcher prototypes shared by the translation units of
// libmipnerf_b200.so.  The public surface is include/mipnerf_b200.h.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "draws.h"

namespace mipnerf {

// ---- ray_kernels.cu ----
cudaError_t launch_distloss(const float* weights, const float* t, float* out, int64_t num_rays, int n,
                            cudaStream_t st);
cudaError_t launch_generate_rays(const float* c2w_host, int height, int width, float focal, float near_v,
                                 float far_v, int row0, int rows, float* origins, float* directions,
                                 float* viewdirs, float* radii, float* near_o, float* far_o, cudaStream_t st);
cudaError_t launch_rays_from_pixels(const float* cam_table, const int64_t* offsets, const int32_t* widths,
                                    int num_images, const int64_t* pixel_ids, int64_t count, const float* atlas,
                                    float* origins, float* directions, float* viewdirs, float* radii,
                                    float* lossmult, float* near_o, float* far_o, float* rgb, cudaStream_t st);
cudaError_t launch_sample_pixels(const float* cam_table, const int64_t* offsets, const int32_t* widths, int num_images,
                                 int64_t num_pixels, const uint64_t* rng_state, int64_t ray_base, int64_t count,
                                 const float* atlas, int64_t* pixel_ids, float* origins, float* directions,
                                 float* viewdirs, float* radii, float* lossmult, float* near_o, float* far_o, float* rgb,
                                 cudaStream_t st);
cudaError_t launch_coarse_t(const float* near, const float* far, const Draws& t_rand, float* t_out,
                            int64_t num_rays, int n, int randomized, int disparity, cudaStream_t st);
cudaError_t launch_philox_uniform(const Draws& d, float* out, int64_t num_rays, int ncols, cudaStream_t st);
cudaError_t launch_philox_normal(const Draws& d, float* out, int64_t num_rays, int ncols, cudaStream_t st);
// raw_density [num_rays, ncols] += d.scale * normal (models/mip_nerf.py:232-233); no-op when `d` is inactive
cudaError_t launch_add_density_noise(float* raw_density, const Draws& d, int64_t num_rays, int ncols, cudaStream_t st);
cudaError_t launch_cast_rays(const float* origins, const float* directions, const float* radii,
                             const float* t, float* means, float* covs, int64_t num_rays, int n,
                             cudaStream_t st);
cudaError_t launch_ipe(const float* means, const float* covs, float* out, int64_t num_points,
                       int min_deg, int max_deg, cudaStream_t st);
cudaError_t launch_ipe_from_t(const float* origins, const float* directions, const float* radii,
                              const float* t, float* out, int64_t num_rays, int n, int min_deg,
                              int max_deg, int disable_integration, cudaStream_t st);
cudaError_t launch_pos_enc(const float* x, float* out, int64_t num_points, int min_deg, int max_deg,
                           int append_identity, cudaStream_t st);
cudaError_t launch_composite(const float* rgb, const float* dens, const float* t, const float* dirs,
                             float* comp_rgb, float* distance, float* acc, float* weights,
                             int64_t num_rays, int n, int white_bkgd, int activate,
                             float density_bias, float rgb_scale, float rgb_padding, cudaStream_t st);
cudaError_t launch_resample(const float* bins, const float* weights, const Draws& jitter, float* out,
                            int64_t* inds, int64_t num_rays, int nb, int ns, int randomized, int blur,
                            float padding, cudaStream_t st);

// ---- metrics.cu ----
size_t image_metrics_scratch_bytes(int height, int width, int channels);
cudaError_t launch_image_metrics(const float* pred, const float* target, int height, int width, int channels,
                                 int window, float sigma, float max_val, void* scratch, float* out, cudaStream_t st);

// ---- linear_f32.cu ----
// Y[M,N] = act( [X1 | X2[row / x2_row_div]] @ W[N, K1+K2]^T + bias ),  fp32 FFMA.
cudaError_t launch_linear_f32(const float* x1, int ld1, int k1, const float* x2, int ld2, int k2,
                              int x2_row_div, const float* w, const float* bias, float* y, int ldy,
                              int64_t m, int n, int relu, cudaStream_t st);

// ---- train_kernels.cu (fp32 training step: backward + Adam) ----
constexpr int kWgradMaxSlices = 160;
int wgrad_num_slices(int64_t m, int tiles);
cudaError_t launch_render_backward(const float* raw_rgb, const float* raw_dens, const float* t, const float* dirs,
                                   const float* target, const float* lossmult, const float* mask_sum,
                                   float mse_mult, float dist_mult, int white_bkgd, float density_bias,
                                   float rgb_scale, float rgb_padding, float* d_raw_rgb, float* d_raw_dens,
                                   float* sqerr_out, float* dist_out, int64_t num_rays, int n, cudaStream_t st);
cudaError_t launch_color_dgrad(const float* d_rgb, const float* wc, const float* v, float* d_v, int64_t m,
                               int k_dim, cudaStream_t st);
// dX[m,k] = (act[m,k] > 0 or act == NULL) * (dY[m,:n_dim] @ W[:n_dim, :k_dim] (row stride ldw) + r1[m] * r1w[k])
cudaError_t launch_dgrad_f32(const float* dy, int n_dim, const float* w, int ldw, const float* r1,
                             const float* r1w, const float* act, float* dx, int64_t m, int k_dim,
                             cudaStream_t st);
// dW[n_dim, k1+k2] (+)= dY^T @ [X1 | X2[row / x2_row_div]],  db[n_dim] (+)= colsum(dY); `part` holds
// up to kWgradMaxSlices * n_dim * (k1+k2+1) floats of per-slice partial sums.
cudaError_t launch_wgrad_f32(const float* dy, int n_dim, const float* x1, int ld1, int k1, const float* x2,
                             int ld2, int k2, int x2_row_div, float* part, float* dw, float* db,
                             int accumulate, int64_t m, cudaStream_t st);
cudaError_t launch_adam(float* p, const float* g, float* m, float* v, int64_t n, float beta1, float beta2,
                        float eps, float step_size, float bc2_sqrt, float grad_scale, cudaStream_t st);
constexpr int kAdamMaxTensors = 32;
struct AdamMulti {  // passed by value in the kernel parameters
  float* p[kAdamMaxTensors];
  const float* g[kAdamMaxTensors];
  float* m[kAdamMaxTensors];
  float* v[kAdamMaxTensors];
  int64_t n[kAdamMaxTensors];
  int blocks[kAdamMaxTensors];  // ceil(n / 256)
  int count;
};
cudaError_t launch_adam_multi(const AdamMulti& t, float beta1, float beta2, float eps, float step_size, float bc2_sqrt,
                              float grad_scale, cudaStream_t st);
// the same update with lr / bc1 and sqrt(bc2) read from per-step tables at the device step count *step + 1
cudaError_t launch_adam_multi_table(const AdamMulti& t, float beta1, float beta2, float eps, const float* step_size,
                                    const float* bc2_sqrt, int64_t table_len, const int64_t* step, float grad_scale,
                                    cudaStream_t st);
cudaError_t launch_train_step_advance(int64_t* step, uint64_t* rng_state, const float* loss, const float* psnr,
                                      float* ring, int ring_len, cudaStream_t st);

// ---- linear_tc.cu (tcgen05 linear layer for the training step's forward / dgrad GEMMs) ----
size_t linear_tc_image_bytes(int n, int k);
bool linear_tc_shape_ok(int n, int k);
// B image of  W[:, off:off+k]  (transposed == 0, n rows)  or of  W[off:off+k, :n]^T  (transposed == 1)
cudaError_t launch_pack_linear_image(const float* w, int ldw, int off, int transposed, void* image, int n, int k,
                                     int precision, cudaStream_t st);
// Y = [mask>0] * relu?( X[M,:k] . B^T + bias[col] + row_bias[row/row_div][col] + prev[row][col] + r1[row]*r1w[col] )
cudaError_t launch_linear_tc(const float* x, int ldx, const void* image, float* y, int ldy, int64_t m, int n, int k,
                             const float* bias, const float* row_bias, int row_div, const float* prev,
                             const float* r1, const float* r1w, const float* mask, int relu, int precision,
                             cudaStream_t st);

bool wgrad_tc_shape_ok(int n_dim);
cudaError_t launch_wgrad_tc_partials(const float* dy, int n_dim, const float* x1, int ld1, int k1, const float* x2,
                                     int ld2, int k2, int x2_row_div, float* part, int64_t m, int max_slices,
                                     int precision, int* slices_out, cudaStream_t st);
cudaError_t launch_wgrad_mn_partials(const void* dy, int dy_t16, int n_dim, const void* x1, int x1_t16, int ld1, int k1,
                                     const void* x2, int x2_t16, int ld2, int k2, int x2_row_div, float* part,
                                     int64_t m, int max_slices, int precision, int* slices_out, cudaStream_t st,
                                     void* mask_out = nullptr);
// fixed-order reduction of [slices, n_dim, k_dim + 1] partials into dW / db (train_kernels.cu)
cudaError_t launch_wgrad_reduce(const float* part, int slices, int n_dim, int k_dim, float* dw, float* db,
                                int accumulate, cudaStream_t st, float scale = 1.f);

// ---- train_t16.cu (backward pass on 16-bit tile images: [tile = 128 rows][64-column slab][128 rows x 128 B, SW128]) ----
size_t t16_image_bytes(int64_t rows, int cols);
cudaError_t launch_t16_pack(const float* src, int ld, int cols, int64_t m, void* image, int precision, cudaStream_t st);
cudaError_t launch_ipe_t16(const float* origins, const float* directions, const float* radii, const float* t, void* image,
                           int64_t num_rays, int n, int disable_integration, int precision, cudaStream_t st);
cudaError_t launch_t16_unpack(const void* image, int cols, float* dst, int ld, int64_t m, int precision,
                              cudaStream_t st);
// mask: a tile image like y (zero where mask <= 0), or mask_bits: [m][32 B] sign bits of a 256-column image
// (wgrad_mn_kernel's by-product); at most one of them
cudaError_t launch_linear_t16(const void* x, const void* image, void* y, int64_t m, int n, int k, const float* r1,
                              const float* r1w, const void* mask, int precision, cudaStream_t st,
                              const void* mask_bits = nullptr);
cudaError_t launch_color_dgrad_t16(const float* d_rgb, const float* wc, const void* v, void* d_v, int64_t m, int k_dim,
                                   int precision, cudaStream_t st);
cudaError_t launch_wgrad_small_n_t16(const float* dy, int n_dim, const void* x, int k_dim, float* part, float* dw,
                                     float* db, int accumulate, int64_t m, int precision, cudaStream_t st,
                                     float scale = 1.f);

// ---- mlp_tc.cu ----
// out[ray][n] = b[n] + W[n, in_main : in_main + view_dim] . venc[ray]   (view-direction part of the view layer)
cudaError_t launch_view_bias_from_enc(const float* venc, const float* w, const float* b, float* out,
                                      int64_t num_rays, cudaStream_t st);

}  // namespace mipnerf
