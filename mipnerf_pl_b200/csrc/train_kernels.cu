// train_kernels.cu — backward pass and optimiser kernels of the training step (SURVEY.md §8f N2:
// models/nerf_system.py:95-121 training_step, torch.optim.Adam of :70-76).  The tensor-core mode swaps the fp32
// GEMMs below for the kernels of linear_tc.cu.
//
// What is differentiated: loss = sum_l  a_l * MSE_l(comp_rgb, target; lossmult mask) + b_l * distloss_l(weights, t)
// with respect to the 24 MLP tensors.  Fenceposts carry no gradient (coarse ones are constants of near/far;
// the fine ones come out of the resampler under no_grad — stop_resample_grad=True, models/mip.py:250-264),
// and the IPE features are constants of the rays, so the backward graph is
//   loss -> comp_rgb / weights -> (rgb, density) -> raw heads -> MLP.
//
// Kernels:
//   render_backward_kernel   warp per ray: d loss / d raw_rgb, d raw_density (+ the per-ray loss terms)
//   color_dgrad_kernel       d v   = relu'(v)  * (d raw_rgb @ Wc)                     (N = 3)
//   dgrad_f32_kernel         d X   = relu'(act) * (d Y @ W[:, :k] + r[m] * rw[k])       128x128x16 FFMA tiles
//   wgrad_f32_kernel         per M-slice partials of  dY^T @ [X1 | X2 | 1]  (last column = bias grad)
//   wgrad_reduce_kernel      fixed-order sum of the partials into dW / db (deterministic, optional accumulate)
//   adam_kernel              torch.optim.Adam single-tensor update, one thread per element
#include "kernels.h"
#include "profile.h"
#include "ray_math.cuh"
#include "sgemm_tile.cuh"

namespace mipnerf {

namespace {
inline unsigned blocks_of(int64_t n, int per_block) { return (unsigned)((n + per_block - 1) / per_block); }
}  // namespace

// -------------------------------------------------------------------------------------------------
// render backward.  Forward per ray (models/mip.py:366-401, models/mip_nerf.py:236-238):
//   rgb_i = sigmoid(raw_i) * (1+2p) - p,  dens_i = softplus(rawd_i + bias),  dd_i = dens_i * (t_{i+1}-t_i) * |d|
//   T_i = exp(-sum_{j<i} dd_j),  w_i = (1 - exp(-dd_i)) * T_i,  comp = sum_i w_i rgb_i (+ 1 - sum_i w_i)
// Backward:  dw_i/ddd_i = T_i exp(-dd_i),  dw_i/ddd_k = -w_i (k < i)
//   => dL/ddd_k = gw_k T_k exp(-dd_k) - sum_{i>k} gw_i w_i              (one suffix sum)
// distloss (models/mip.py:8-20) with sorted midpoints:  d/dw_i = (2/3) len_i w_i + 2 S_i,
//   S_i = sum_j w_j |m_i - m_j| = m_i (W_<i - W_>i) - (M_<i - M_>i)      (two prefix sums)
// -------------------------------------------------------------------------------------------------
template <int P>
__global__ void render_backward_kernel(const float* __restrict__ raw_rgb, const float* __restrict__ raw_dens,
                                       const float* __restrict__ t, const float* __restrict__ dirs,
                                       const float* __restrict__ target, const float* __restrict__ lossmult,
                                       const float* __restrict__ mask_sum, float mse_mult, float dist_mult,
                                       int white_bkgd, float density_bias, float rgb_scale, float rgb_padding,
                                       float* __restrict__ d_raw_rgb, float* __restrict__ d_raw_dens,
                                       float* __restrict__ sqerr_out, float* __restrict__ dist_out,
                                       int64_t num_rays) {
  constexpr int N = P * 32;
  const int lane = threadIdx.x & 31;
  const int64_t ray = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (ray >= num_rays) return;
  const float dx = __ldg(dirs + ray * 3), dy = __ldg(dirs + ray * 3 + 1), dz = __ldg(dirs + ray * 3 + 2);
  const float dnorm = sqrtf(dx * dx + dy * dy + dz * dz);
  const float* tr = t + ray * (N + 1);
  const float t_first = __ldg(tr);
  float tt[P + 1];
#pragma unroll
  for (int p = 0; p <= P; ++p) tt[p] = __ldg(tr + lane * P + p);

  // ---- forward recompute: dd, transmittance, weights, activated colours
  float dd[P], delta[P], dsig[P], w[P], tr_after[P], rgb[P][3], srgb[P][3];
  double run = 0.0, incl[P];
#pragma unroll
  for (int p = 0; p < P; ++p) {
    const float x = __ldg(raw_dens + ray * N + lane * P + p) + density_bias;
    const float dens = x > 20.0f ? x : log1pf(expf(x));
    dsig[p] = x > 20.0f ? 1.0f : 1.0f / (1.0f + expf(-x));  // softplus'
    delta[p] = __fmul_rn(__fsub_rn(tt[p + 1], tt[p]), dnorm);
    dd[p] = __fmul_rn(dens, delta[p]);
    run += (double)dd[p];
    incl[p] = run;
  }
  double total;
  const double before = warp_excl_scan_f64(run, lane, total);
  float cr = 0.f, cg = 0.f, cb = 0.f, wsum = 0.f;
#pragma unroll
  for (int p = 0; p < P; ++p) {
    const double excl = before + (p == 0 ? 0.0 : incl[p - 1]);
    const float cum = (lane == 0 && p == 0) ? 0.0f : (float)excl;
    const float trans = expf(-cum);
    w[p] = __fmul_rn(-expm1f(-dd[p]), trans);
    tr_after[p] = trans * expf(-dd[p]);  // T_i exp(-dd_i) = dw_i / ddd_i
    const int64_t s = ray * N + lane * P + p;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float sg = 1.0f / (1.0f + expf(-__ldg(raw_rgb + s * 3 + c)));
      srgb[p][c] = sg;
      rgb[p][c] = sg * rgb_scale - rgb_padding;
    }
    cr += w[p] * rgb[p][0], cg += w[p] * rgb[p][1], cb += w[p] * rgb[p][2], wsum += w[p];
  }
  cr = warp_sum(cr), cg = warp_sum(cg), cb = warp_sum(cb), wsum = warp_sum(wsum);
  const float bg = white_bkgd ? 1.0f - wsum : 0.0f;
  const float comp[3] = {cr + bg, cg + bg, cb + bg};

  // ---- d loss / d comp_rgb                                   (models/nerf_system.py:104-105)
  const float mask = lossmult ? __ldg(lossmult + ray) : 1.0f;
  const float inv_ms = 1.0f / __ldg(mask_sum);
  float g[3], sq = 0.f;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float e = comp[c] - __ldg(target + ray * 3 + c);
    sq += e * e;
    g[c] = mse_mult * 2.0f * mask * e * inv_ms;
  }
  const float gsum_bg = white_bkgd ? (g[0] + g[1] + g[2]) : 0.0f;

  // ---- distloss prefix sums (midpoints relative to t_0: |m_i - m_j| is shift invariant)
  double w_run = 0.0, m_run = 0.0;
  float mid[P];
#pragma unroll
  for (int p = 0; p < P; ++p) {
    mid[p] = 0.5f * ((tt[p] - t_first) + (tt[p + 1] - t_first));
    w_run += (double)w[p];
    m_run += (double)w[p] * (double)mid[p];
  }
  double w_tot, m_tot;
  double w_lt = warp_excl_scan_f64(w_run, lane, w_tot);
  double m_lt = warp_excl_scan_f64(m_run, lane, m_tot);

  float gw[P];
  double gww_run = 0.0, gww_incl[P], dist_val = 0.0;
#pragma unroll
  for (int p = 0; p < P; ++p) {
    const double wi = w[p], mi = mid[p];
    const double w_gt = w_tot - w_lt - wi, m_gt = m_tot - m_lt - wi * mi;
    const double s_i = mi * (w_lt - w_gt) - (m_lt - m_gt);
    const double len = (double)tt[p + 1] - (double)tt[p];
    dist_val += len * wi * wi / 3.0 + wi * s_i;
    const float gdist = dist_mult * (float)((2.0 / 3.0) * len * wi + 2.0 * s_i);
    gw[p] = g[0] * rgb[p][0] + g[1] * rgb[p][1] + g[2] * rgb[p][2] - gsum_bg + gdist;
    gww_run += (double)gw[p] * wi;
    gww_incl[p] = gww_run;
    w_lt += wi;
    m_lt += wi * mi;
  }
  double gww_tot;
  const double gww_before = warp_excl_scan_f64(gww_run, lane, gww_tot);
#pragma unroll
  for (int p = 0; p < P; ++p) {
    const double suffix = gww_tot - (gww_before + gww_incl[p]);  // sum_{i>k} gw_i w_i
    const float d_dd = gw[p] * tr_after[p] - (float)suffix;
    const int64_t s = ray * N + lane * P + p;
    d_raw_dens[s] = d_dd * delta[p] * dsig[p];
#pragma unroll
    for (int c = 0; c < 3; ++c)
      d_raw_rgb[s * 3 + c] = g[c] * w[p] * rgb_scale * srgb[p][c] * (1.0f - srgb[p][c]);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) dist_val += __shfl_xor_sync(0xffffffffu, dist_val, o);
  if (lane == 0) {
    if (sqerr_out) sqerr_out[ray] = mask * sq;
    if (dist_out) dist_out[ray] = (float)dist_val;
  }
}

cudaError_t launch_render_backward(const float* raw_rgb, const float* raw_dens, const float* t, const float* dirs,
                                   const float* target, const float* lossmult, const float* mask_sum,
                                   float mse_mult, float dist_mult, int white_bkgd, float density_bias,
                                   float rgb_scale, float rgb_padding, float* d_raw_rgb, float* d_raw_dens,
                                   float* sqerr_out, float* dist_out, int64_t num_rays, int n, cudaStream_t st) {
  if (num_rays == 0) return cudaSuccess;
  LaunchScope scope(kKernRenderBackward, st);
  const unsigned grid = blocks_of(num_rays, 4);
#define MIPNERF_RB_CASE(PP)                                                                                    \
  case PP:                                                                                                     \
    render_backward_kernel<PP><<<grid, 128, 0, st>>>(raw_rgb, raw_dens, t, dirs, target, lossmult, mask_sum,   \
                                                     mse_mult, dist_mult, white_bkgd, density_bias, rgb_scale, \
                                                     rgb_padding, d_raw_rgb, d_raw_dens, sqerr_out, dist_out,  \
                                                     num_rays);                                                \
    break;
  switch (n / 32) {
    MIPNERF_RB_CASE(1)
    MIPNERF_RB_CASE(2)
    MIPNERF_RB_CASE(3)
    MIPNERF_RB_CASE(4)
    MIPNERF_RB_CASE(6)
    MIPNERF_RB_CASE(8)
    default:
      return cudaErrorInvalidValue;
  }
#undef MIPNERF_RB_CASE
  return cudaGetLastError();
}

// -------------------------------------------------------------------------------------------------
// colour head backward into the view layer's activation: d v[m,k] = (v[m,k] > 0) * sum_c d_rgb[m,c] Wc[c,k]
// -------------------------------------------------------------------------------------------------
__global__ void color_dgrad_kernel(const float* __restrict__ d_rgb, const float* __restrict__ wc,
                                   const float* __restrict__ v, float* __restrict__ d_v, int64_t m, int k_dim) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= m * k_dim) return;
  const int64_t row = idx / k_dim;
  const int k = (int)(idx % k_dim);
  float acc = 0.f;
#pragma unroll
  for (int c = 0; c < 3; ++c) acc = fmaf(__ldg(d_rgb + row * 3 + c), __ldg(wc + c * k_dim + k), acc);
  d_v[idx] = __ldg(v + idx) > 0.f ? acc : 0.f;
}

cudaError_t launch_color_dgrad(const float* d_rgb, const float* wc, const float* v, float* d_v, int64_t m,
                               int k_dim, cudaStream_t st) {
  if (m == 0) return cudaSuccess;
  LaunchScope scope(kKernDgrad, st);
  color_dgrad_kernel<<<blocks_of(m * k_dim, 256), 256, 0, st>>>(d_rgb, wc, v, d_v, m, k_dim);
  return cudaGetLastError();
}

// -------------------------------------------------------------------------------------------------
// dgrad:  dX[m,k] = mask * ( sum_n dY[m,n] W[n*ldw + k]  +  r1[m] * r1w[k] ),  mask = act[m,k] > 0 (or 1)
// 128 x 128 output tile, reduction over n in steps of 16, 8x8 micro-tiles (same mapping as linear_f32.cu).
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kTileThreads, 2)
dgrad_f32_kernel(const float* __restrict__ dy, int n_dim, const float* __restrict__ w, int ldw,
                 const float* __restrict__ r1, const float* __restrict__ r1w, const float* __restrict__ act,
                 float* __restrict__ dx, int64_t m, int k_dim, int vec_a, int vec_b) {
  __shared__ __align__(16) TileSmem s;
  const int tid = threadIdx.x;
  const int64_t row0 = (int64_t)blockIdx.x * kTileM;
  const int col0 = blockIdx.y * kTileN;
  const int ty = tid >> 4, tx = tid & 15;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  auto fetch_a = [&](int nn) {  // dY rows, contiguous along the reduction index n
    return fetch_frag([&](int g) {
      const int64_t row = row0 + (g >> 2);
      const int nk = nn + (g & 3) * 4;
      if (row >= m || nk >= n_dim) return make_float4(0.f, 0.f, 0.f, 0.f);
      return ld4(dy + row * n_dim + nk, n_dim - nk, vec_a);
    });
  };
  auto fetch_b = [&](int nn) {  // W rows n, contiguous along the output column k
    return fetch_frag([&](int g) {
      const int nk = nn + (g >> 5);
      const int c = col0 + (g & 31) * 4;
      if (nk >= n_dim || c >= k_dim) return make_float4(0.f, 0.f, 0.f, 0.f);
      return ld4(w + (int64_t)nk * ldw + c, k_dim - c, vec_b);
    });
  };
  Frag fa = fetch_a(0), fb = fetch_b(0);
  for (int nn = 0; nn < n_dim; nn += kTileK) {
    store_kcontig(s.a, fa);
    store_rowcontig(s.b, fb);
    __syncthreads();
    if (nn + kTileK < n_dim) {
      fa = fetch_a(nn + kTileK);
      fb = fetch_b(nn + kTileK);
    }
    tile_fma(s, acc, ty, tx);
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int64_t row = row0 + tile_row(i, ty);
    if (row >= m) continue;
    const float rv = r1 ? __ldg(r1 + row) : 0.f;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int col = col0 + tile_row(j, tx);
      if (col >= k_dim) continue;
      float v = acc[i][j];
      if (r1) v = fmaf(rv, __ldg(r1w + col), v);
      if (act && !(__ldg(act + row * k_dim + col) > 0.f)) v = 0.f;
      dx[row * k_dim + col] = v;
    }
  }
}

cudaError_t launch_dgrad_f32(const float* dy, int n_dim, const float* w, int ldw, const float* r1,
                             const float* r1w, const float* act, float* dx, int64_t m, int k_dim,
                             cudaStream_t st) {
  if (m == 0 || k_dim == 0) return cudaSuccess;
  LaunchScope scope(kKernDgrad, st);
  dim3 grid((unsigned)((m + 127) / 128), (unsigned)((k_dim + 127) / 128));
  const int vec_a = aligned16(dy) && n_dim % 4 == 0;
  const int vec_b = aligned16(w) && ldw % 4 == 0;
  dgrad_f32_kernel<<<grid, kTileThreads, 0, st>>>(dy, n_dim, w, ldw, r1, r1w, act, dx, m, k_dim, vec_a, vec_b);
  return cudaGetLastError();
}

// -------------------------------------------------------------------------------------------------
// wgrad partials:  part[s][n][kg] = sum_{m in slice s} dY[m,n] * Xc[m,kg],  Xc = [X1 (k1 cols) | X2[m / x2_row_div]
//   (k2 cols)];  column K of the partial holds the bias gradient (column sums of dY, accumulated from the staged
//   dY tile by the first column block — no extra tile for a 'ones' column).
// Both operand tiles are read along their contiguous dimension (no transposes): the reduction index is the row.
// -------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(kTileThreads, 2)
wgrad_f32_kernel(const float* __restrict__ dy, int n_dim, const float* __restrict__ x1, int ld1, int k1,
                 const float* __restrict__ x2, int ld2, int k2, int x2_row_div, float* __restrict__ part,
                 int64_t m, int64_t slice_rows, int vec_a, int vec_b) {
  __shared__ __align__(16) TileSmem s;
  const int tid = threadIdx.x;
  const int K = k1 + k2;
  const int n0 = blockIdx.y * kTileM, kg0 = blockIdx.z * kTileN;
  const int64_t m_begin = (int64_t)blockIdx.x * slice_rows;
  const int64_t m_end = (m_begin + slice_rows) < m ? (m_begin + slice_rows) : m;
  const int ty = tid >> 4, tx = tid & 15;
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  auto fetch_a = [&](int64_t m0) {  // dY rows m0..m0+15, contiguous along n
    return fetch_frag([&](int g) {
      const int64_t row = m0 + (g >> 5);
      const int nn = n0 + (g & 31) * 4;
      if (row >= m_end || nn >= n_dim) return make_float4(0.f, 0.f, 0.f, 0.f);
      return ld4(dy + row * n_dim + nn, n_dim - nn, vec_a);
    });
  };
  auto fetch_b = [&](int64_t m0) {  // [X1 | X2[row / div] | 1] rows, contiguous along the column
    return fetch_frag([&](int g) {
      const int64_t row = m0 + (g >> 5);
      const int kg = kg0 + (g & 31) * 4;
      if (row >= m_end || kg >= K) return make_float4(0.f, 0.f, 0.f, 0.f);
      if (kg + 4 <= k1) return ld4(x1 + row * ld1 + kg, 4, vec_b);
      float e[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = kg + j;
        e[j] = c < k1 ? __ldg(x1 + row * ld1 + c) : (c < K ? __ldg(x2 + (row / x2_row_div) * ld2 + (c - k1)) : 0.f);
      }
      return make_float4(e[0], e[1], e[2], e[3]);
    });
  };
  float bsum = 0.f;
  Frag fa = fetch_a(m_begin), fb = fetch_b(m_begin);
  for (int64_t m0 = m_begin; m0 < m_end; m0 += kTileK) {
    store_rowcontig(s.a, fa);
    store_rowcontig(s.b, fb);
    __syncthreads();
    if (m0 + kTileK < m_end) {
      fa = fetch_a(m0 + kTileK);
      fb = fetch_b(m0 + kTileK);
    }
    if (blockIdx.z == 0 && tid < kTileM) {  // bias gradient: column sums of the dY tile, first column block only
#pragma unroll
      for (int k = 0; k < kTileK; ++k) bsum += s.a[k][tid];
    }
    tile_fma(s, acc, ty, tx);
    __syncthreads();
  }
  float* out = part + (size_t)blockIdx.x * n_dim * (K + 1);
  if (blockIdx.z == 0 && tid < kTileM && n0 + tid < n_dim) out[(size_t)(n0 + tid) * (K + 1) + K] = bsum;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int n = n0 + tile_row(i, ty);
    if (n >= n_dim) continue;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int kg = kg0 + tile_row(j, tx);
      if (kg >= K) continue;
      out[(size_t)n * (K + 1) + kg] = acc[i][j];
    }
  }
}

// wgrad for the two narrow heads (density: n = 1, colour: n = 3), where a 128-wide output tile would be 97-99 %
// padding: thread = input column k (blockDim / k_dim row groups per block), each row's dY values are warp-uniform
// loads, X is read once, coalesced — an HBM-bound pass.  Same partial layout as wgrad_f32_kernel.
__global__ void __launch_bounds__(256)
wgrad_small_n_kernel(const float* __restrict__ dy, int n_dim, const float* __restrict__ x, int k_dim,
                     float* __restrict__ part, int64_t m, int64_t slice_rows) {
  __shared__ float red[256][5];
  const int tid = threadIdx.x;
  const int groups = 256 / k_dim;          // k_dim in {128, 256}
  const int grp = tid / k_dim, k = tid % k_dim;
  const int64_t m_begin = (int64_t)blockIdx.x * slice_rows;
  const int64_t m_end = (m_begin + slice_rows) < m ? (m_begin + slice_rows) : m;
  float acc[4] = {0.f, 0.f, 0.f, 0.f}, bsum[4] = {0.f, 0.f, 0.f, 0.f};
  if (grp < groups) {
#pragma unroll 8  // independent loads: eight rows in flight per thread (the loop is latency-bound otherwise)
    for (int64_t row = m_begin + grp; row < m_end; row += groups) {
      const float xv = __ldg(x + row * k_dim + k);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (j < n_dim) {
          const float d = __ldg(dy + row * n_dim + j);
          acc[j] = fmaf(d, xv, acc[j]);
          bsum[j] += d;
        }
      }
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) red[tid][j] = acc[j];
  __syncthreads();
  float* out = part + (size_t)blockIdx.x * n_dim * (k_dim + 1);
  if (tid < k_dim) {
    for (int j = 0; j < n_dim; ++j) {
      float v = 0.f;
      for (int g2 = 0; g2 < groups; ++g2) v += red[g2 * k_dim + tid][j];
      out[(size_t)j * (k_dim + 1) + tid] = v;
    }
  }
  __syncthreads();
  if (k == 0)
#pragma unroll
    for (int j = 0; j < 4; ++j) red[grp][j] = bsum[j];
  __syncthreads();
  if (tid < n_dim) {
    float v = 0.f;
    for (int g2 = 0; g2 < groups; ++g2) v += red[g2][tid];
    out[(size_t)tid * (k_dim + 1) + k_dim] = v;
  }
}

// Fixed-order sum of the per-slice partials.  The loads do not depend on the running sum, but one thread walking all
// 148 slices is a chain of ~19 DRAM / L2 round trips even with eight loads in flight (22 us per layer); so four
// threads share an output element — thread g sums slices [g * q, (g + 1) * q) in order, eight loads in flight — and
// the four partial sums are added in the order g = 0..3: still one fixed order, a quarter of the latency chain.
__global__ void __launch_bounds__(256)
wgrad_reduce_kernel(const float* __restrict__ part, int slices, int n_dim, int k_dim, float* __restrict__ dw,
                    float* __restrict__ db, int accumulate, float scale = 1.f) {
  __shared__ float sm[4][64];
  const int lane64 = threadIdx.x & 63, g = threadIdx.x >> 6;
  const int idx = blockIdx.x * 64 + lane64;
  const int per = k_dim + 1;
  const bool ok = idx < n_dim * per;
  const int q = (slices + 3) / 4;
  const int s_begin = g * q, s_end = (g + 1) * q < slices ? (g + 1) * q : slices;
  float acc = 0.f;
  if (ok) {
    const size_t stride = (size_t)n_dim * per;
    int s = s_begin;
    for (; s + 8 <= s_end; s += 8) {
      float v[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) v[u] = __ldg(part + (size_t)(s + u) * stride + idx);
#pragma unroll
      for (int u = 0; u < 8; ++u) acc += v[u];
    }
    for (; s < s_end; ++s) acc += __ldg(part + (size_t)s * stride + idx);
  }
  sm[g][lane64] = acc;
  __syncthreads();
  if (g == 0 && ok) {
    float t = ((sm[0][lane64] + sm[1][lane64]) + sm[2][lane64]) + sm[3][lane64];
    const int n = idx / per, kg = idx % per;
    float* dst = kg < k_dim ? dw + (size_t)n * k_dim + kg : db + n;
    t *= scale;  // 1 / (the fp16 step's gradient scale); exactly 1 otherwise
    *dst = accumulate ? *dst + t : t;
  }
}

// Number of M-slices for a wgrad with `tiles` output tiles.  Small problems: one slice per 4096 rows.  Large ones:
// fill whole waves of the grid (2 CTAs per SM resident) so the last wave is not mostly empty — 4 tiles x 74 slices
// is exactly one wave of 296 CTAs on 148 SMs, where the old fixed 128 slices left the second wave 27 % full.
int wgrad_num_slices(int64_t m, int tiles) {
  int64_t s = (m + 4095) / 4096;
  if (s < 1) s = 1;
  if (s > kWgradMaxSlices) s = kWgradMaxSlices;
  static int resident = 0;
  if (resident == 0) {
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    resident = 2 * sms;
  }
  if (tiles < 1) tiles = 1;
  if (s * tiles > resident) {  // more than one wave anyway: round the slice count to whole waves
    const int64_t waves = (s * tiles + resident - 1) / resident;
    int64_t fit = waves * resident / tiles;
    if (fit > kWgradMaxSlices) fit = (waves - 1 > 0 ? (waves - 1) * resident / tiles : kWgradMaxSlices);
    if (fit >= 1 && fit <= kWgradMaxSlices) s = fit;
  }
  return (int)s;
}

cudaError_t launch_wgrad_reduce(const float* part, int slices, int n_dim, int k_dim, float* dw, float* db,
                                int accumulate, cudaStream_t st, float scale) {
  LaunchScope scope(kKernWgrad, st);
  wgrad_reduce_kernel<<<blocks_of((int64_t)n_dim * (k_dim + 1), 64), 256, 0, st>>>(part, slices, n_dim, k_dim, dw, db,
                                                                                    accumulate, scale);
  return cudaGetLastError();
}

cudaError_t launch_wgrad_f32(const float* dy, int n_dim, const float* x1, int ld1, int k1, const float* x2,
                             int ld2, int k2, int x2_row_div, float* part, float* dw, float* db,
                             int accumulate, int64_t m, cudaStream_t st) {
  if (m == 0 || n_dim == 0) return cudaSuccess;
  if (!x2) {
    x2 = x1, ld2 = ld1, k2 = 0;
  }
  if (x2_row_div < 1) x2_row_div = 1;
  const int K = k1 + k2;
  if (n_dim <= 4 && k2 == 0 && ld1 == k1 && (k1 == 128 || k1 == 256)) {  // the density / colour heads
    // many short slices (8 blocks per SM in flight): the partial buffer is sized for 160 slices of a 256 x 353
    // layer, i.e. room for thousands of [n_dim <= 4] x [K+1 <= 257] partials
    int64_t want = m / 512;
    if (want < 1) want = 1;
    if (want > 1184) want = 1184;
    const int slices = (int)want;
    int64_t rows = (m + slices - 1) / slices;
    LaunchScope scope(kKernWgrad, st);
    wgrad_small_n_kernel<<<slices, 256, 0, st>>>(dy, n_dim, x1, k1, part, m, rows);
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
    wgrad_reduce_kernel<<<blocks_of((int64_t)n_dim * (K + 1), 64), 256, 0, st>>>(part, slices, n_dim, K, dw, db,
                                                                                 accumulate);
    return cudaGetLastError();
  }
  const int tiles = ((n_dim + 127) / 128) * ((K + 127) / 128);
  const int slices = wgrad_num_slices(m, tiles);
  int64_t slice_rows = (m + slices - 1) / slices;
  slice_rows = (slice_rows + 15) / 16 * 16;
  LaunchScope scope(kKernWgrad, st);
  dim3 grid((unsigned)slices, (unsigned)((n_dim + 127) / 128), (unsigned)((K + 127) / 128));
  const int vec_a = aligned16(dy) && n_dim % 4 == 0;
  const int vec_b = aligned16(x1) && ld1 % 4 == 0;
  wgrad_f32_kernel<<<grid, kTileThreads, 0, st>>>(dy, n_dim, x1, ld1, k1, x2, ld2, k2, x2_row_div, part, m, slice_rows,
                                                  vec_a, vec_b);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  wgrad_reduce_kernel<<<blocks_of((int64_t)n_dim * (K + 1), 64), 256, 0, st>>>(part, slices, n_dim, K, dw, db,
                                                                               accumulate);
  return cudaGetLastError();
}

// -------------------------------------------------------------------------------------------------
// torch.optim.Adam (amsgrad=False, weight_decay=0, maximize=False), single-tensor form:
//   m <- lerp(m, g, 1-b1);  v <- b2 v + (1-b2) g^2;  p <- p - (lr/bc1) * m / (sqrt(v)/sqrt(bc2) + eps)
// -------------------------------------------------------------------------------------------------
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, int64_t n, float beta1, float beta2, float eps, float step_size,
                            float bc2_sqrt, float grad_scale) {
  const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float gi = __fmul_rn(g[i], grad_scale);
  const float mi = __fadd_rn(m[i], __fmul_rn(__fsub_rn(gi, m[i]), 1.0f - beta1));
  const float vi = __fadd_rn(__fmul_rn(v[i], beta2), __fmul_rn(__fmul_rn(gi, gi), 1.0f - beta2));
  m[i] = mi;
  v[i] = vi;
  const float denom = __fadd_rn(__fdiv_rn(sqrtf(vi), bc2_sqrt), eps);
  p[i] = __fadd_rn(p[i], __fmul_rn(-step_size, __fdiv_rn(mi, denom)));
}

// All tensors of one optimiser group in ONE launch (24 launches of ~7 us otherwise): block -> tensor by a scan of the
// per-tensor block counts carried in the kernel parameters.
__global__ void adam_multi_kernel(const AdamMulti t, float beta1, float beta2, float eps, float step_size,
                                  float bc2_sqrt, float grad_scale) {
  int b = blockIdx.x, k = 0;
  while (k + 1 < t.count && b >= t.blocks[k]) b -= t.blocks[k++];
  const int64_t i = (int64_t)b * blockDim.x + threadIdx.x;
  if (i >= t.n[k]) return;
  float* __restrict__ p = t.p[k];
  float* __restrict__ m = t.m[k];
  float* __restrict__ v = t.v[k];
  const float gi = __fmul_rn(t.g[k][i], grad_scale);
  const float mi = __fadd_rn(m[i], __fmul_rn(__fsub_rn(gi, m[i]), 1.0f - beta1));
  const float vi = __fadd_rn(__fmul_rn(v[i], beta2), __fmul_rn(__fmul_rn(gi, gi), 1.0f - beta2));
  m[i] = mi;
  v[i] = vi;
  const float denom = __fadd_rn(__fdiv_rn(sqrtf(vi), bc2_sqrt), eps);
  p[i] = __fadd_rn(p[i], __fmul_rn(-step_size, __fdiv_rn(mi, denom)));
}

cudaError_t launch_adam_multi(const AdamMulti& t, float beta1, float beta2, float eps, float step_size, float bc2_sqrt,
                              float grad_scale, cudaStream_t st) {
  int total = 0;
  for (int k = 0; k < t.count; ++k) total += t.blocks[k];
  if (total == 0) return cudaSuccess;
  LaunchScope scope(kKernAdam, st);
  adam_multi_kernel<<<total, 256, 0, st>>>(t, beta1, beta2, eps, step_size, bc2_sqrt, grad_scale);
  return cudaGetLastError();
}

// adam_multi_kernel for a captured training step: the step count lives on the device, and lr / bc1, sqrt(bc2) come
// from tables the host filled with the double-precision math of mipnerf_b200_adam_step_multi (entry t = step t).
__global__ void adam_multi_table_kernel(const AdamMulti t, float beta1, float beta2, float eps,
                                        const float* __restrict__ step_size_tab, const float* __restrict__ bc2_sqrt_tab,
                                        int64_t table_len, const int64_t* __restrict__ step, float grad_scale) {
  int b = blockIdx.x, k = 0;
  while (k + 1 < t.count && b >= t.blocks[k]) b -= t.blocks[k++];
  const int64_t i = (int64_t)b * blockDim.x + threadIdx.x;
  if (i >= t.n[k]) return;
  int64_t s = *step + 1;
  s = s < 1 ? 1 : (s >= table_len ? table_len - 1 : s);  // never read outside the tables (the host sizes them)
  const float step_size = step_size_tab[s], bc2_sqrt = bc2_sqrt_tab[s];
  float* __restrict__ p = t.p[k];
  float* __restrict__ m = t.m[k];
  float* __restrict__ v = t.v[k];
  const float gi = __fmul_rn(t.g[k][i], grad_scale);
  const float mi = __fadd_rn(m[i], __fmul_rn(__fsub_rn(gi, m[i]), 1.0f - beta1));
  const float vi = __fadd_rn(__fmul_rn(v[i], beta2), __fmul_rn(__fmul_rn(gi, gi), 1.0f - beta2));
  m[i] = mi;
  v[i] = vi;
  const float denom = __fadd_rn(__fdiv_rn(sqrtf(vi), bc2_sqrt), eps);
  p[i] = __fadd_rn(p[i], __fmul_rn(-step_size, __fdiv_rn(mi, denom)));
}

// End of a captured training step: log (loss, psnr) into ring row step % ring_len, then step += 1 and the Philox
// offset += 1 (one fresh set of draws per step, like MipNerf.next_rng).  One thread; runs after every reader.
__global__ void train_step_advance_kernel(int64_t* step, uint64_t* rng_state, const float* loss, const float* psnr,
                                          float* ring, int ring_len) {
  const int64_t s = *step;
  if (ring_len > 0) {
    ring[(s % ring_len) * 2 + 0] = *loss;
    ring[(s % ring_len) * 2 + 1] = *psnr;
  }
  *step = s + 1;
  rng_state[1] += 1;
}

cudaError_t launch_adam_multi_table(const AdamMulti& t, float beta1, float beta2, float eps, const float* step_size,
                                    const float* bc2_sqrt, int64_t table_len, const int64_t* step, float grad_scale,
                                    cudaStream_t st) {
  int total = 0;
  for (int k = 0; k < t.count; ++k) total += t.blocks[k];
  if (total == 0) return cudaSuccess;
  LaunchScope scope(kKernAdam, st);
  adam_multi_table_kernel<<<total, 256, 0, st>>>(t, beta1, beta2, eps, step_size, bc2_sqrt, table_len, step, grad_scale);
  return cudaGetLastError();
}

cudaError_t launch_train_step_advance(int64_t* step, uint64_t* rng_state, const float* loss, const float* psnr,
                                      float* ring, int ring_len, cudaStream_t st) {
  train_step_advance_kernel<<<1, 1, 0, st>>>(step, rng_state, loss, psnr, ring, ring_len);
  return cudaGetLastError();
}

cudaError_t launch_adam(float* p, const float* g, float* m, float* v, int64_t n, float beta1, float beta2,
                        float eps, float step_size, float bc2_sqrt, float grad_scale, cudaStream_t st) {
  if (n == 0) return cudaSuccess;
  LaunchScope scope(kKernAdam, st);
  adam_kernel<<<blocks_of(n, 256), 256, 0, st>>>(p, g, m, v, n, beta1, beta2, eps, step_size, bc2_sqrt, grad_scale);
  return cudaGetLastError();
}

}  // namespace mipnerf
