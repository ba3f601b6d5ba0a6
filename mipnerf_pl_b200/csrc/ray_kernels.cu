// ray_kernels.cu — the non-MLP stages of the path as stand-alone sm_100a kernels.
//
// These are the building blocks of the fp32 parity path and of the per-stage C-ABI entry points:
//   coarse fenceposts            models/mip.py:145-163
//   cast_rays (cone, diagonal)   models/mip.py:81-103  (+ :50-78, :22-36)
//   integrated_pos_enc / pos_enc models/mip.py:322-363
//   volumetric_rendering         models/mip.py:366-401 (+ activations models/mip_nerf.py:236-238)
//   resample_along_rays          models/mip.py:232-280 (+ sorted_piecewise_constant_pdf :168-229)
// Compositing and resampling are warp-per-ray: one ray's N samples live in one warp's registers /
// shared-memory slice, reductions are shuffles, no cross-warp traffic.
#include "kernels.h"
#include "profile.h"
#include "ray_math.cuh"
#include "ray_resample.cuh"

namespace mipnerf {

static inline unsigned blocks_for(int64_t n, int per_block) { return (unsigned)((n + per_block - 1) / per_block); }

// ---------------------------------------------------------------------------------------------
// coarse fenceposts: one thread per (ray, j)
// ---------------------------------------------------------------------------------------------
__global__ void coarse_t_kernel(const float* __restrict__ near, const float* __restrict__ far,
                                const Draws t_rand, float* __restrict__ t_out,
                                int64_t num_rays, int n, int randomized, int disparity) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  const int64_t total = num_rays * (n + 1);
  if (idx >= total) return;
  const int64_t ray = idx / (n + 1);
  const int j = (int)(idx % (n + 1));
  t_out[idx] = coarse_fencepost(__ldg(near + ray), __ldg(far + ray), j, n, disparity, randomized != 0,
                                randomized ? draw_uniform(t_rand, ray, j, n + 1) : 0.f);
}

// the uniforms the kernels draw for (seed, offset, stream): test / reproduction helper
__global__ void philox_uniform_kernel(const Draws d, float* __restrict__ out, int64_t num_rays, int ncols) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= num_rays * ncols) return;
  out[idx] = draw_uniform(d, idx / ncols, (int)(idx % ncols), ncols);
}

// the standard normals of the density noise for (seed, offset, level): test / reproduction helper
__global__ void philox_normal_kernel(const Draws d, float* __restrict__ out, int64_t num_rays, int ncols) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= num_rays * ncols) return;
  out[idx] = draw_normal(d, idx / ncols, (int)(idx % ncols), ncols);
}
// raw_density[ray, j] += density_noise * normal[ray, j]   (models/mip_nerf.py:232-233; the fp32 path keeps the raw
// heads in HBM between the MLP and the compositing, so the noise is one in-place pass; the tensor-core level kernels
// add it in their compositing epilogue instead)
__global__ void add_density_noise_kernel(float* __restrict__ raw_density, const Draws d, int64_t num_rays, int ncols) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= num_rays * ncols) return;
  raw_density[idx] = add_density_noise(raw_density[idx], d, idx / ncols, (int)(idx % ncols), ncols);
}

// ---------------------------------------------------------------------------------------------
// cast_rays: one thread per (ray, sample) -> means, covs [B,N,3]
// ---------------------------------------------------------------------------------------------
__global__ void cast_rays_kernel(const float* __restrict__ origins,
                                 const float* __restrict__ directions,
                                 const float* __restrict__ radii, const float* __restrict__ t,
                                 float* __restrict__ means, float* __restrict__ covs,
                                 int64_t num_rays, int n) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= num_rays * n) return;
  const int64_t ray = idx / n;
  const int j = (int)(idx % n);
  const RayGeom g = load_ray_geom(origins, directions, radii, ray);
  const float t0 = __ldg(t + ray * (n + 1) + j), t1 = __ldg(t + ray * (n + 1) + j + 1);
  float tm, tv, rv, mean[3], cov[3];
  frustum_moments(t0, t1, g.radius_sq, tm, tv, rv);
  lift_gaussian(g, tm, tv, rv, mean, cov);
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    means[idx * 3 + c] = mean[c];
    covs[idx * 3 + c] = cov[c];
  }
}

// ---------------------------------------------------------------------------------------------
// IPE from explicit (means, covs): one thread per (point, degree*3+coord); coalesced stores.
// ---------------------------------------------------------------------------------------------
__global__ void ipe_kernel(const float* __restrict__ means, const float* __restrict__ covs,
                           float* __restrict__ out, int64_t num_points, int min_deg, int num_deg) {
  const int half = num_deg * 3;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= num_points * half) return;
  const int64_t p = idx / half;
  const int f = (int)(idx % half);
  const int l = min_deg + f / 3, c = f % 3;
  float fs, fc;
  ipe_pair<false>(__ldg(means + p * 3 + c), __ldg(covs + p * 3 + c), l, fs, fc);
  out[p * 2 * half + f] = fs;
  out[p * 2 * half + half + f] = fc;
}

// IPE straight from fenceposts (cast_rays fused in): what forward() uses, no means/covs in HBM.
__global__ void ipe_from_t_kernel(const float* __restrict__ origins,
                                  const float* __restrict__ directions,
                                  const float* __restrict__ radii, const float* __restrict__ t,
                                  float* __restrict__ out, int64_t num_rays, int n, int min_deg,
                                  int num_deg, int disable_integration) {
  const int half = num_deg * 3;
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= num_rays * n * half) return;
  const int64_t p = idx / half;
  const int f = (int)(idx % half);
  const int64_t ray = p / n;
  const int j = (int)(p % n);
  const int l = min_deg + f / 3, c = f % 3;
  const RayGeom g = load_ray_geom(origins, directions, radii, ray);
  const float t0 = __ldg(t + ray * (n + 1) + j), t1 = __ldg(t + ray * (n + 1) + j + 1);
  float tm, tv, rv, mean[3], cov[3];
  frustum_moments(t0, t1, g.radius_sq, tm, tv, rv);
  lift_gaussian(g, tm, tv, rv, mean, cov);
  float fs, fc;
  ipe_pair<false>(mean[c], disable_integration ? 0.0f : cov[c], l, fs, fc);
  out[p * 2 * half + f] = fs;
  out[p * 2 * half + half + f] = fc;
}

// pos_enc: one thread per (point, output feature)
__global__ void pos_enc_kernel(const float* __restrict__ x, float* __restrict__ out,
                               int64_t num_points, int min_deg, int num_deg, int append_identity) {
  const int half = num_deg * 3;
  const int width = 2 * half + (append_identity ? 3 : 0);
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= num_points * width) return;
  const int64_t p = idx / width;
  int f = (int)(idx % width);
  if (append_identity) {
    if (f < 3) {
      out[idx] = __ldg(x + p * 3 + f);
      return;
    }
    f -= 3;
  }
  const int is_cos = f >= half;
  if (is_cos) f -= half;
  const int l = min_deg + f / 3, c = f % 3;
  const float y = __fmul_rn(__ldg(x + p * 3 + c), __int_as_float((127 + l) << 23));
  out[idx] = sinf(is_cos ? __fadd_rn(y, MIPNERF_HALF_PI_F32) : y);
}

// ---------------------------------------------------------------------------------------------
// volumetric_rendering: warp per ray, lane owns P = N/32 consecutive samples.
// ---------------------------------------------------------------------------------------------
template <int P, bool kActivate>
__global__ void composite_kernel(const float* __restrict__ rgb_in, const float* __restrict__ dens_in,
                                 const float* __restrict__ t, const float* __restrict__ dirs,
                                 float* __restrict__ comp_rgb, float* __restrict__ distance,
                                 float* __restrict__ acc_out, float* __restrict__ weights_out,
                                 int64_t num_rays, int white_bkgd, float density_bias,
                                 float rgb_scale, float rgb_padding) {
  constexpr int N = P * 32;
  const int lane = threadIdx.x & 31;
  const int64_t ray = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (ray >= num_rays) return;
  const float dx = __ldg(dirs + ray * 3), dy = __ldg(dirs + ray * 3 + 1), dz = __ldg(dirs + ray * 3 + 2);
  const float dnorm = sqrtf(dx * dx + dy * dy + dz * dz);  // torch.linalg.norm      (:386)
  const float* tr = t + ray * (N + 1);
  float tt[P + 1];
#pragma unroll
  for (int p = 0; p <= P; ++p) tt[p] = __ldg(tr + lane * P + p);
  float dd[P];
  double run = 0.0;
  double incl[P];
#pragma unroll
  for (int p = 0; p < P; ++p) {
    float dens = __ldg(dens_in + ray * N + lane * P + p);
    if (kActivate) dens = density_activation(dens, density_bias);
    const float delta = __fmul_rn(__fsub_rn(tt[p + 1], tt[p]), dnorm);
    dd[p] = __fmul_rn(dens, delta);
    run += (double)dd[p];
    incl[p] = run;
  }
  double total;
  const double before = warp_excl_scan_f64(run, lane, total);
  float wsum = 0.f, dsum = 0.f, r = 0.f, g = 0.f, b = 0.f;
#pragma unroll
  for (int p = 0; p < P; ++p) {
    // exclusive cumsum, fp64 running sum rounded per prefix like torch.cumsum(float32)   (:389-392)
    const double excl = before + (p == 0 ? 0.0 : incl[p - 1]);
    const float cum = (lane == 0 && p == 0) ? 0.0f : (float)excl;
    // 1 - exp(-dd) evaluated as -expm1(-dd): same expression, without the reference's fp32
    // cancellation noise (tests/test_reference_roundoff.py), so we sit next to its exact value
    const float alpha = -expm1f(-dd[p]);
    const float w = __fmul_rn(alpha, expf(-cum));
    const int64_t s = ray * N + lane * P + p;
    if (weights_out) weights_out[s] = w;
    float cr = __ldg(rgb_in + s * 3), cg = __ldg(rgb_in + s * 3 + 1), cb = __ldg(rgb_in + s * 3 + 2);
    if (kActivate) {
      cr = rgb_activation(cr, rgb_scale, rgb_padding);
      cg = rgb_activation(cg, rgb_scale, rgb_padding);
      cb = rgb_activation(cb, rgb_scale, rgb_padding);
    }
    r += w * cr;
    g += w * cg;
    b += w * cb;
    wsum += w;
    dsum += w * __fmul_rn(0.5f, __fadd_rn(tt[p], tt[p + 1]));
  }
  r = warp_sum(r), g = warp_sum(g), b = warp_sum(b), wsum = warp_sum(wsum), dsum = warp_sum(dsum);
  if (lane == 0) {
    // nan_to_num then clamp to [t_0, t_N]                                             (:398)
    const float t_first = __ldg(tr), t_last = __ldg(tr + N);
    float d = dsum;
    if (isnan(d)) d = 0.f;
    else if (isinf(d)) d = d > 0 ? 3.4028234663852886e38f : -3.4028234663852886e38f;
    d = fminf(fmaxf(d, t_first), t_last);
    const float bg = white_bkgd ? __fsub_rn(1.0f, wsum) : 0.0f;
    comp_rgb[ray * 3 + 0] = r + bg;
    comp_rgb[ray * 3 + 1] = g + bg;
    comp_rgb[ray * 3 + 2] = b + bg;
    distance[ray] = d;
    acc_out[ray] = wsum;
  }
}

template <bool kBlur>
__global__ void resample_kernel(const float* __restrict__ bins, const float* __restrict__ weights,
                                const Draws jitter, float* __restrict__ out,
                                int64_t* __restrict__ inds, int64_t num_rays, int nb, int ns,
                                int randomized, float padding) {
  extern __shared__ float smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t ray = (int64_t)blockIdx.x * (blockDim.x >> 5) + warp;
  if (ray >= num_rays) return;
  float* s_w = smem + (size_t)warp * (3 * nb + 2);
  float* s_cdf = s_w + nb;
  float* s_bins = s_cdf + nb + 1;
  resample_warp<kBlur>(bins + ray * (nb + 1), weights + ray * nb, nb, ns, randomized, jitter, ray, padding, s_w,
                       s_cdf, s_bins, out + ray * ns, inds ? inds + ray * ns : nullptr, lane);
}

// ---------------------------------------------------------------------------------------------
// distloss (models/mip.py:8-20), per ray:  (1/3) sum_i d_i w_i^2  +  sum_ij w_i w_j |m_i - m_j|.
// The reference builds two [B,N,N] tensors; midpoints are sorted (fenceposts are), so
//   sum_ij w_i w_j |m_i - m_j| = 2 sum_i w_i (m_i W_<i - M_<i),  W_<i = sum_{j<i} w_j,  M_<i = sum_{j<i} w_j m_j
// which is two warp scans.  Warp per ray, fp64 accumulation.
// ---------------------------------------------------------------------------------------------
__global__ void distloss_kernel(const float* __restrict__ weights, const float* __restrict__ t,
                                float* __restrict__ out, int64_t num_rays, int n) {
  const int lane = threadIdx.x & 31;
  const int64_t ray = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (ray >= num_rays) return;
  const float* w = weights + ray * n;
  const float* tr = t + ray * (n + 1);
  const int per = (n + 31) / 32;
  double uni = 0.0, bi = 0.0, w_run = 0.0, m_run = 0.0;
  // pass 1: lane totals over its contiguous chunk
  for (int p = 0; p < per; ++p) {
    const int i = lane * per + p;
    if (i < n) {
      const double wi = w[i], mi = 0.5 * ((double)tr[i] + (double)tr[i + 1]);
      w_run += wi;
      m_run += wi * mi;
    }
  }
  double tot;
  double w_before = warp_excl_scan_f64(w_run, lane, tot);
  double m_before = warp_excl_scan_f64(m_run, lane, tot);
  for (int p = 0; p < per; ++p) {
    const int i = lane * per + p;
    if (i < n) {
      const double wi = w[i], t0 = tr[i], t1 = tr[i + 1], mi = 0.5 * (t0 + t1);
      uni += (t1 - t0) * wi * wi;
      bi += wi * (mi * w_before - m_before);
      w_before += wi;
      m_before += wi * mi;
    }
  }
  double v = uni / 3.0 + 2.0 * bi;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  if (lane == 0) out[ray] = (float)v;
}

// ---------------------------------------------------------------------------------------------
// Blender-style pinhole rays for rows [row0, row0+rows) of an H x W frame, straight into HBM
// (datasets/datasets.py:214-263, render_video.py:29-105): one thread per pixel.
//   camera dir = ((x - W/2 + .5)/f, -(y - H/2 + .5)/f, -1);  direction = R . dir;  origin = c2w[:,3]
//   radius = |d(x,y) - d(x,y+1)| * 2/sqrt(12)  (last row repeats the previous one)
// ---------------------------------------------------------------------------------------------
struct Pose {
  float m[12];  // row-major [3,4] camera-to-world
};
__device__ __forceinline__ void pixel_dir(const Pose& c, float x, float y, float w, float h, float focal,
                                          float d[3]) {
  const float cx = __fdiv_rn(__fadd_rn(__fsub_rn(x, __fmul_rn(w, 0.5f)), 0.5f), focal);
  const float cy = -__fdiv_rn(__fadd_rn(__fsub_rn(y, __fmul_rn(h, 0.5f)), 0.5f), focal);
#pragma unroll
  for (int i = 0; i < 3; ++i) d[i] = c.m[i * 4 + 0] * cx + c.m[i * 4 + 1] * cy - c.m[i * 4 + 2];
}
__global__ void generate_rays_kernel(const Pose c, int height, int width, float focal, float near_v, float far_v,
                                     int row0, int rows, float* __restrict__ origins,
                                     float* __restrict__ directions, float* __restrict__ viewdirs,
                                     float* __restrict__ radii, float* __restrict__ near_o,
                                     float* __restrict__ far_o) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)rows * width) return;
  const int y = row0 + (int)(idx / width), x = (int)(idx % width);
  float d[3];
  pixel_dir(c, (float)x, (float)y, (float)width, (float)height, focal, d);
  // |d(x,y) - d(x,y+1)| is the rotated camera-space step (0, 1/f, 0): the same for every pixel (so
  // "the last row repeats the previous one" holds trivially) and free of the fp32 cancellation noise
  // (~3e-5 relative) the reference's finite difference carries (datasets/datasets.py:245-253)
  const float dx = c.m[1] / focal, dy = c.m[5] / focal, dz = c.m[9] / focal;
  const float inv = rsqrtf(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    origins[idx * 3 + i] = c.m[i * 4 + 3];
    directions[idx * 3 + i] = d[i];
    viewdirs[idx * 3 + i] = d[i] * inv;
  }
  radii[idx] = sqrtf(dx * dx + dy * dy + dz * dz) * 0.57735026918962576f;  // 2/sqrt(12)
  near_o[idx] = near_v;
  far_o[idx] = far_v;
}

// ---------------------------------------------------------------------------------------------
// Training rays straight from pixel ids (SURVEY.md §8f N4: datasets/datasets.py:116-168, 216-263 without the
// host-side per-pixel arrays).  The scene lives in HBM as a pixel atlas [P,3] + a camera table per image
//   cam[24] = pix2cam (3x3 row-major) | cam2world (3x4 row-major) | lossmult | near | far,
// `offsets[i]` = first atlas row of image i, `widths[i]` its width.  One thread per requested pixel:
//   image = upper_bound(offsets, id) - 1, (x, y) from the in-image index,
//   camera dir = pix2cam . (x+.5, y+.5, 1),  direction = R . dir,  origin = t,  viewdir = direction / |direction|,
//   radius = |R . pix2cam[:,1]| * 2/sqrt(12)   (the y-neighbour distance of the reference, which is the same
//   vector for every pixel of an image; see generate_rays_kernel for why it is evaluated analytically).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void ray_from_pixel(const float* __restrict__ cam_table, const int64_t* __restrict__ offsets,
                                               const int32_t* __restrict__ widths, int num_images, int64_t i,
                                               int64_t id, const float* __restrict__ atlas,
                                               float* __restrict__ origins, float* __restrict__ directions,
                                               float* __restrict__ viewdirs, float* __restrict__ radii,
                                               float* __restrict__ lossmult, float* __restrict__ near_o,
                                               float* __restrict__ far_o, float* __restrict__ rgb) {
  int lo = 0, hi = num_images;  // offsets[lo] <= id < offsets[hi]
  while (hi - lo > 1) {
    const int mid = (lo + hi) >> 1;
    if (__ldg(offsets + mid) <= id) lo = mid;
    else hi = mid;
  }
  const float* cam = cam_table + (size_t)lo * 24;
  const int64_t local = id - __ldg(offsets + lo);
  const int w = __ldg(widths + lo);
  const float px = (float)(local % w) + 0.5f, py = (float)(local / w) + 0.5f;
  float k[9], m[12];
#pragma unroll
  for (int j = 0; j < 9; ++j) k[j] = __ldg(cam + j);
#pragma unroll
  for (int j = 0; j < 12; ++j) m[j] = __ldg(cam + 9 + j);
  const float cx = k[0] * px + k[1] * py + k[2], cy = k[3] * px + k[4] * py + k[5], cz = k[6] * px + k[7] * py + k[8];
  float d[3], s[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    d[r] = m[r * 4 + 0] * cx + m[r * 4 + 1] * cy + m[r * 4 + 2] * cz;
    s[r] = m[r * 4 + 0] * k[1] + m[r * 4 + 1] * k[4] + m[r * 4 + 2] * k[7];  // d(x, y+1) - d(x, y)
  }
  const float inv_norm = 1.0f / sqrtf(d[0] * d[0] + d[1] * d[1] + d[2] * d[2]);
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    origins[i * 3 + r] = m[r * 4 + 3];
    directions[i * 3 + r] = d[r];
    viewdirs[i * 3 + r] = d[r] * inv_norm;
  }
  radii[i] = sqrtf(s[0] * s[0] + s[1] * s[1] + s[2] * s[2]) * 0.5773502691896258f;  // 2 / sqrt(12)
  lossmult[i] = __ldg(cam + 21);
  near_o[i] = __ldg(cam + 22);
  far_o[i] = __ldg(cam + 23);
  if (rgb) {
#pragma unroll
    for (int c = 0; c < 3; ++c) rgb[i * 3 + c] = __ldg(atlas + id * 3 + c);
  }
}

__global__ void rays_from_pixels_kernel(const float* __restrict__ cam_table, const int64_t* __restrict__ offsets,
                                        const int32_t* __restrict__ widths, int num_images,
                                        const int64_t* __restrict__ pixel_ids, int64_t count,
                                        const float* __restrict__ atlas, float* __restrict__ origins,
                                        float* __restrict__ directions, float* __restrict__ viewdirs,
                                        float* __restrict__ radii, float* __restrict__ lossmult,
                                        float* __restrict__ near_o, float* __restrict__ far_o,
                                        float* __restrict__ rgb) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  // ids outside the atlas are clamped to its first / last row (never read out of bounds); offsets[num_images] = P
  const int64_t total = __ldg(offsets + num_images);
  int64_t id = __ldg(pixel_ids + i);
  id = id < 0 ? 0 : (id >= total ? total - 1 : id);
  ray_from_pixel(cam_table, offsets, widths, num_images, i, id, atlas, origins, directions, viewdirs, radii, lossmult,
                 near_o, far_o, rgb);
}

// A uniformly random training batch drawn on the device: pixel id of ray i = floor(x * P / 2^32), x the first 32-bit
// Philox4x32-10 output of counter (ray_base + i, stream kPixelStream << 24, offset) under key (seed, offset) read
// from `rng_state` when the kernel runs -- the counter layout of draw_uniform, so mipnerf_b200_philox_uniform's
// generator (and its host mirror) reproduces the ids.  Each id is hit by floor or ceil of 2^32 / P of the 2^32
// draws: its probability differs from 1/P by less than 2^-32.
__global__ void sample_pixels_kernel(const float* __restrict__ cam_table, const int64_t* __restrict__ offsets,
                                     const int32_t* __restrict__ widths, int num_images, uint64_t num_pixels,
                                     const uint64_t* __restrict__ rng_state, int64_t ray_base, int64_t count,
                                     const float* __restrict__ atlas, int64_t* __restrict__ pixel_ids,
                                     float* __restrict__ origins, float* __restrict__ directions,
                                     float* __restrict__ viewdirs, float* __restrict__ radii,
                                     float* __restrict__ lossmult, float* __restrict__ near_o,
                                     float* __restrict__ far_o, float* __restrict__ rgb) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= count) return;
  const uint64_t seed = rng_state[0], offset = rng_state[1];
  const uint64_t g = (uint64_t)(ray_base + i);
  const uint32_t x = philox4x32_10_first((uint32_t)g, (uint32_t)(g >> 32), (uint32_t)kPixelStream << 24,
                                         (uint32_t)offset, (uint32_t)seed, (uint32_t)(seed >> 32) ^ (uint32_t)(offset >> 32));
  int64_t id = (int64_t)(((uint64_t)x * num_pixels) >> 32);  // num_pixels <= 2^32: id < num_pixels
  const int64_t total = __ldg(offsets + num_images);          // never past the atlas, whatever num_pixels says
  id = id < total ? id : total - 1;
  if (pixel_ids) pixel_ids[i] = id;
  ray_from_pixel(cam_table, offsets, widths, num_images, i, id, atlas, origins, directions, viewdirs, radii, lossmult,
                 near_o, far_o, rgb);
}

// ---------------------------------------------------------------------------------------------
// launchers
// ---------------------------------------------------------------------------------------------
cudaError_t launch_rays_from_pixels(const float* cam_table, const int64_t* offsets, const int32_t* widths,
                                    int num_images, const int64_t* pixel_ids, int64_t count, const float* atlas,
                                    float* origins, float* directions, float* viewdirs, float* radii,
                                    float* lossmult, float* near_o, float* far_o, float* rgb, cudaStream_t st) {
  if (count == 0) return cudaSuccess;
  LaunchScope scope(kKernRayGen, st);
  rays_from_pixels_kernel<<<blocks_for(count, 256), 256, 0, st>>>(cam_table, offsets, widths, num_images, pixel_ids,
                                                                 count, atlas, origins, directions, viewdirs, radii,
                                                                 lossmult, near_o, far_o, rgb);
  return cudaGetLastError();
}

cudaError_t launch_sample_pixels(const float* cam_table, const int64_t* offsets, const int32_t* widths, int num_images,
                                 int64_t num_pixels, const uint64_t* rng_state, int64_t ray_base, int64_t count,
                                 const float* atlas, int64_t* pixel_ids, float* origins, float* directions,
                                 float* viewdirs, float* radii, float* lossmult, float* near_o, float* far_o, float* rgb,
                                 cudaStream_t st) {
  if (count == 0) return cudaSuccess;
  LaunchScope scope(kKernRayGen, st);
  sample_pixels_kernel<<<blocks_for(count, 256), 256, 0, st>>>(cam_table, offsets, widths, num_images,
                                                              (uint64_t)num_pixels, rng_state, ray_base, count, atlas,
                                                              pixel_ids, origins, directions, viewdirs, radii, lossmult,
                                                              near_o, far_o, rgb);
  return cudaGetLastError();
}

cudaError_t launch_generate_rays(const float* c2w_host, int height, int width, float focal, float near_v,
                                 float far_v, int row0, int rows, float* origins, float* directions,
                                 float* viewdirs, float* radii, float* near_o, float* far_o, cudaStream_t st) {
  if (rows <= 0) return cudaSuccess;
  Pose c;
  for (int i = 0; i < 12; ++i) c.m[i] = c2w_host[i];
  LaunchScope scope(kKernRayGen, st);
  generate_rays_kernel<<<blocks_for((int64_t)rows * width, 256), 256, 0, st>>>(
      c, height, width, focal, near_v, far_v, row0, rows, origins, directions, viewdirs, radii, near_o, far_o);
  return cudaGetLastError();
}

cudaError_t launch_distloss(const float* weights, const float* t, float* out, int64_t num_rays, int n,
                            cudaStream_t st) {
  if (num_rays == 0) return cudaSuccess;
  LaunchScope scope(kKernDistloss, st);
  distloss_kernel<<<blocks_for(num_rays, 4), 128, 0, st>>>(weights, t, out, num_rays, n);
  return cudaGetLastError();
}

cudaError_t launch_philox_uniform(const Draws& d, float* out, int64_t num_rays, int ncols, cudaStream_t st) {
  if (num_rays == 0) return cudaSuccess;
  philox_uniform_kernel<<<blocks_for(num_rays * ncols, 256), 256, 0, st>>>(d, out, num_rays, ncols);
  return cudaGetLastError();
}

cudaError_t launch_philox_normal(const Draws& d, float* out, int64_t num_rays, int ncols, cudaStream_t st) {
  if (num_rays == 0) return cudaSuccess;
  philox_normal_kernel<<<blocks_for(num_rays * ncols, 256), 256, 0, st>>>(d, out, num_rays, ncols);
  return cudaGetLastError();
}

cudaError_t launch_add_density_noise(float* raw_density, const Draws& d, int64_t num_rays, int ncols, cudaStream_t st) {
  if (num_rays == 0 || !draws_active(d)) return cudaSuccess;
  add_density_noise_kernel<<<blocks_for(num_rays * ncols, 256), 256, 0, st>>>(raw_density, d, num_rays, ncols);
  return cudaGetLastError();
}

cudaError_t launch_coarse_t(const float* near, const float* far, const Draws& t_rand, float* t_out,
                            int64_t num_rays, int n, int randomized, int disparity, cudaStream_t st) {
  if (num_rays == 0) return cudaSuccess;
  LaunchScope scope(kKernCoarseT, st);
  coarse_t_kernel<<<blocks_for(num_rays * (n + 1), 256), 256, 0, st>>>(near, far, t_rand, t_out, num_rays,
                                                                     n, randomized, disparity);
  return cudaGetLastError();
}

cudaError_t launch_cast_rays(const float* origins, const float* directions, const float* radii,
                             const float* t, float* means, float* covs, int64_t num_rays, int n,
                             cudaStream_t st) {
  if (num_rays == 0) return cudaSuccess;
  LaunchScope scope(kKernCastRays, st);
  cast_rays_kernel<<<blocks_for(num_rays * n, 256), 256, 0, st>>>(origins, directions, radii, t, means,
                                                                 covs, num_rays, n);
  return cudaGetLastError();
}

cudaError_t launch_ipe(const float* means, const float* covs, float* out, int64_t num_points,
                       int min_deg, int max_deg, cudaStream_t st) {
  const int nd = max_deg - min_deg;
  if (num_points == 0 || nd <= 0) return cudaSuccess;
  LaunchScope scope(kKernIpe, st);
  ipe_kernel<<<blocks_for(num_points * nd * 3, 256), 256, 0, st>>>(means, covs, out, num_points, min_deg, nd);
  return cudaGetLastError();
}

cudaError_t launch_ipe_from_t(const float* origins, const float* directions, const float* radii,
                              const float* t, float* out, int64_t num_rays, int n, int min_deg,
                              int max_deg, int disable_integration, cudaStream_t st) {
  const int nd = max_deg - min_deg;
  if (num_rays == 0 || nd <= 0) return cudaSuccess;
  LaunchScope scope(kKernIpe, st);
  ipe_from_t_kernel<<<blocks_for(num_rays * n * nd * 3, 256), 256, 0, st>>>(
      origins, directions, radii, t, out, num_rays, n, min_deg, nd, disable_integration);
  return cudaGetLastError();
}

cudaError_t launch_pos_enc(const float* x, float* out, int64_t num_points, int min_deg, int max_deg,
                           int append_identity, cudaStream_t st) {
  const int nd = max_deg - min_deg;
  const int width = 6 * nd + (append_identity ? 3 : 0);
  if (num_points == 0 || width == 0) return cudaSuccess;
  LaunchScope scope(kKernPosEnc, st);
  pos_enc_kernel<<<blocks_for(num_points * width, 256), 256, 0, st>>>(x, out, num_points, min_deg, nd,
                                                                     append_identity);
  return cudaGetLastError();
}

template <bool kActivate>
static cudaError_t launch_composite_t(const float* rgb, const float* dens, const float* t,
                                      const float* dirs, float* comp_rgb, float* distance, float* acc,
                                      float* weights, int64_t num_rays, int n, int white_bkgd,
                                      float density_bias, float rgb_scale, float rgb_padding,
                                      cudaStream_t st) {
  if (num_rays == 0) return cudaSuccess;
  LaunchScope scope(kKernComposite, st);
  const unsigned grid = blocks_for(num_rays, 4);
#define MIPNERF_COMPOSITE_CASE(PP)                                                                   \
  case PP:                                                                                           \
    composite_kernel<PP, kActivate><<<grid, 128, 0, st>>>(rgb, dens, t, dirs, comp_rgb, distance,    \
                                                          acc, weights, num_rays, white_bkgd,        \
                                                          density_bias, rgb_scale, rgb_padding);     \
    break;
  switch (n / 32) {
    MIPNERF_COMPOSITE_CASE(1)
    MIPNERF_COMPOSITE_CASE(2)
    MIPNERF_COMPOSITE_CASE(3)
    MIPNERF_COMPOSITE_CASE(4)
    MIPNERF_COMPOSITE_CASE(6)
    MIPNERF_COMPOSITE_CASE(8)
    default:
      return cudaErrorInvalidValue;
  }
#undef MIPNERF_COMPOSITE_CASE
  return cudaGetLastError();
}

cudaError_t launch_composite(const float* rgb, const float* dens, const float* t, const float* dirs,
                             float* comp_rgb, float* distance, float* acc, float* weights,
                             int64_t num_rays, int n, int white_bkgd, int activate,
                             float density_bias, float rgb_scale, float rgb_padding, cudaStream_t st) {
  if (activate)
    return launch_composite_t<true>(rgb, dens, t, dirs, comp_rgb, distance, acc, weights, num_rays, n,
                                    white_bkgd, density_bias, rgb_scale, rgb_padding, st);
  return launch_composite_t<false>(rgb, dens, t, dirs, comp_rgb, distance, acc, weights, num_rays, n,
                                   white_bkgd, density_bias, rgb_scale, rgb_padding, st);
}

cudaError_t launch_resample(const float* bins, const float* weights, const Draws& jitter, float* out,
                            int64_t* inds, int64_t num_rays, int nb, int ns, int randomized, int blur,
                            float padding, cudaStream_t st) {
  if (num_rays == 0) return cudaSuccess;
  LaunchScope scope(kKernResample, st);
  const int warps = 4;
  const size_t smem = (size_t)warps * (3 * nb + 2) * sizeof(float);
  const unsigned grid = blocks_for(num_rays, warps);
  if (blur)
    resample_kernel<true><<<grid, warps * 32, smem, st>>>(bins, weights, jitter, out, inds, num_rays, nb,
                                                         ns, randomized, padding);
  else
    resample_kernel<false><<<grid, warps * 32, smem, st>>>(bins, weights, jitter, out, inds, num_rays, nb,
                                                          ns, randomized, padding);
  return cudaGetLastError();
}

}  // namespace mipnerf
