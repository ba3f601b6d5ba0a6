// api.cu — the extern "C" surface declared in include/mipnerf_b200.h and the level loop of
// MipNerf.forward (models/mip_nerf.py:172-248) expressed as kernel launches on one stream.
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>

#include "../../include/mipnerf_b200.h"
#include "kernels.h"
#include "mlp_tc.h"

namespace {

thread_local std::string g_last_error;

int fail(int code, const char* fmt, ...) {
  char buf[512];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  g_last_error = buf;
  return code;
}

#define CUDA_TRY(expr)                                                                           \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess)                                                                       \
      return fail(MIPNERF_B200_ECUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e),    \
                  __FILE__, __LINE__);                                                           \
  } while (0)

constexpr int64_t kChunkRaysFp32 = 4096;  // bounds the fp32 path's activation scratch (~1.8 GB)

inline size_t align_up(size_t v, size_t a = 256) { return (v + a - 1) / a * a; }

struct Dims {
  int xyz_dim, view_dim, n_lin;
};

int check_config(const mipnerf_b200_config* c, Dims* d) {
  if (!c) return fail(MIPNERF_B200_EINVAL, "config is NULL");
  if (c->num_samples <= 0 || c->num_samples % 32 != 0 || c->num_samples > 256 ||
      (c->num_samples / 32 == 5) || (c->num_samples / 32 == 7))
    return fail(MIPNERF_B200_EUNSUPPORTED, "num_samples=%d: need a multiple of 32 in {32,64,96,128,192,256}",
                c->num_samples);
  if (c->num_levels < 1) return fail(MIPNERF_B200_EINVAL, "num_levels=%d", c->num_levels);
  if (c->max_deg_point <= c->min_deg_point || c->min_deg_point < -60 || c->max_deg_point > 60)
    return fail(MIPNERF_B200_EINVAL, "bad point degrees [%d,%d)", c->min_deg_point, c->max_deg_point);
  if (c->deg_view < 0 || c->deg_view > 60) return fail(MIPNERF_B200_EINVAL, "deg_view=%d", c->deg_view);
  if (c->net_depth < 1 || c->net_width < 1 || c->skip_index < 1 || c->net_depth_condition < 0 ||
      c->net_width_condition < 1)
    return fail(MIPNERF_B200_EINVAL, "bad MLP shape");
  if (c->num_rgb_channels != 3 || c->num_density_channels != 1)
    return fail(MIPNERF_B200_EUNSUPPORTED, "only 3 rgb / 1 density channels (volumetric_rendering assumes it)");
  const int last = c->net_depth - 1;
  if (last > 0 && last % c->skip_index == 0)
    return fail(MIPNERF_B200_EUNSUPPORTED,
                "skip connection after the last trunk layer: the reference's density_layer cannot take it");
  if (!c->use_viewdirs && c->net_width != c->net_width_condition)
    return fail(MIPNERF_B200_EUNSUPPORTED,
                "use_viewdirs=False needs net_width == net_width_condition (reference color_layer shape)");
  if (!(c->density_noise >= 0.f) || c->density_noise > 3.0e38f)
    return fail(MIPNERF_B200_EINVAL, "density_noise=%g: need a finite standard deviation >= 0", (double)c->density_noise);
  d->xyz_dim = (c->max_deg_point - c->min_deg_point) * 6;
  d->view_dim = c->deg_view * 6 + 3;
  d->n_lin = c->net_depth + 2 + c->net_depth_condition + 1;
  return MIPNERF_B200_OK;
}

int check_weights(const mipnerf_b200_config* c, const Dims& d, const mipnerf_b200_weights* w) {
  if (!w || !w->linears) return fail(MIPNERF_B200_EINVAL, "weights are NULL");
  if (w->num_linears != d.n_lin)
    return fail(MIPNERF_B200_EINVAL, "expected %d linears (state_dict order), got %d", d.n_lin, w->num_linears);
  auto expect = [&](int idx, int in, int out, const char* name) {
    const mipnerf_b200_linear& l = w->linears[idx];
    if (!l.weight || !l.bias) return fail(MIPNERF_B200_EINVAL, "%s has a NULL tensor", name);
    if (l.in_features != in || l.out_features != out)
      return fail(MIPNERF_B200_EINVAL, "%s is [%d,%d], expected [%d,%d]", name, l.out_features, l.in_features,
                  out, in);
    return MIPNERF_B200_OK;
  };
  int rc;
  for (int i = 0; i < c->net_depth; ++i) {
    int in = i == 0 ? d.xyz_dim : c->net_width;
    if (i > 1 && (i - 1) % c->skip_index == 0) in = c->net_width + d.xyz_dim;  // models/mip_nerf.py:40-42
    if ((rc = expect(i, in, c->net_width, "layers[i]"))) return rc;
  }
  if ((rc = expect(c->net_depth, c->net_width, 1, "density_layer"))) return rc;
  if ((rc = expect(c->net_depth + 1, c->net_width, c->net_width, "extra_layer"))) return rc;
  for (int i = 0; i < c->net_depth_condition; ++i) {
    const int in = i == 0 ? c->net_width + d.view_dim : c->net_width_condition;
    if ((rc = expect(c->net_depth + 2 + i, in, c->net_width_condition, "view_layers[i]"))) return rc;
  }
  return expect(d.n_lin - 1, c->net_width_condition, 3, "color_layer");
}

int check_rays(const mipnerf_b200_rays* r) {
  if (!r) return fail(MIPNERF_B200_EINVAL, "rays is NULL");
  if (r->num_rays < 0) return fail(MIPNERF_B200_EINVAL, "num_rays=%lld", (long long)r->num_rays);
  if (r->num_rays > 0 && (!r->origins || !r->directions || !r->radii || !r->near || !r->far))
    return fail(MIPNERF_B200_EINVAL, "a ray field is NULL");
  return MIPNERF_B200_OK;
}

mipnerf_b200_rays offset_rays(const mipnerf_b200_rays& r, int64_t off, int64_t count) {
  mipnerf_b200_rays o = r;
  o.origins = r.origins + off * 3;
  o.directions = r.directions + off * 3;
  o.viewdirs = r.viewdirs ? r.viewdirs + off * 3 : nullptr;
  o.radii = r.radii + off;
  o.near = r.near + off;
  o.far = r.far + off;
  o.num_rays = count;
  return o;
}

// Scratch layout for one chunk of R rays on the fp32 path.
struct Fp32Scratch {
  float *enc, *h0, *h1, *venc, *c0, *c1, *raw_rgb, *raw_density, *t[2], *w[2];
  size_t bytes;
};

Fp32Scratch carve_fp32(const mipnerf_b200_config* c, const Dims& d, int64_t rays, void* base,
                       bool mlp_only = false) {
  Fp32Scratch s{};
  const size_t m = (size_t)rays * c->num_samples;
  size_t off = 0;
  auto take = [&](size_t elems) {
    float* p = base ? reinterpret_cast<float*>(static_cast<char*>(base) + off) : nullptr;
    off += align_up(elems * sizeof(float));
    return p;
  };
  s.h0 = take(m * c->net_width);
  s.h1 = take(m * c->net_width);
  s.c0 = take(m * c->net_width_condition);
  s.c1 = take(m * c->net_width_condition);
  if (mlp_only) {
    s.bytes = off;
    return s;
  }
  s.enc = take(m * d.xyz_dim);
  s.venc = take((size_t)rays * d.view_dim);
  s.raw_rgb = take(m * 3);
  s.raw_density = take(m);
  for (int i = 0; i < 2; ++i) {
    s.t[i] = take((size_t)rays * (c->num_samples + 1));
    s.w[i] = take(m);
  }
  s.bytes = off;
  return s;
}

// MLP.forward on the fp32 path (models/mip_nerf.py:75-111).
int mlp_forward_fp32(const mipnerf_b200_config* c, const Dims& d, const mipnerf_b200_weights* w,
                     const float* x, const float* venc, int64_t rays, int n, const Fp32Scratch& s,
                     float* raw_rgb, float* raw_density, cudaStream_t st) {
  const int64_t m = rays * n;
  const float* cur = x;
  int cur_k = d.xyz_dim;
  bool concat = false;
  for (int i = 0; i < c->net_depth; ++i) {
    const mipnerf_b200_linear& l = w->linears[i];
    float* out = (i & 1) ? s.h1 : s.h0;
    CUDA_TRY(mipnerf::launch_linear_f32(cur, cur_k, cur_k, concat ? x : nullptr, d.xyz_dim,
                                        concat ? d.xyz_dim : 0, 1, l.weight, l.bias, out, c->net_width, m,
                                        c->net_width, 1, st));
    cur = out;
    cur_k = c->net_width;
    concat = (i % c->skip_index == 0 && i > 0);  // models/mip_nerf.py:96-97
  }
  const mipnerf_b200_linear& dl = w->linears[c->net_depth];
  CUDA_TRY(mipnerf::launch_linear_f32(cur, cur_k, cur_k, nullptr, 0, 0, 1, dl.weight, dl.bias, raw_density,
                                      1, m, 1, 0, st));
  const float* feat = cur;
  int feat_k = cur_k;
  if (c->use_viewdirs) {
    const mipnerf_b200_linear& el = w->linears[c->net_depth + 1];
    float* bott = (cur == s.h0) ? s.h1 : s.h0;
    CUDA_TRY(mipnerf::launch_linear_f32(cur, cur_k, cur_k, nullptr, 0, 0, 1, el.weight, el.bias, bott,
                                        c->net_width, m, c->net_width, 0, st));
    feat = bott;
    feat_k = c->net_width;
    for (int j = 0; j < c->net_depth_condition; ++j) {
      const mipnerf_b200_linear& vl = w->linears[c->net_depth + 2 + j];
      float* out = (j & 1) ? s.c1 : s.c0;
      CUDA_TRY(mipnerf::launch_linear_f32(feat, feat_k, feat_k, j == 0 ? venc : nullptr, d.view_dim,
                                          j == 0 ? d.view_dim : 0, n, vl.weight, vl.bias, out,
                                          c->net_width_condition, m, c->net_width_condition, 1, st));
      feat = out;
      feat_k = c->net_width_condition;
    }
    if (c->net_depth_condition == 0) {
      // view_layers is an empty Sequential: the colour head would see width+view_dim inputs, which
      // the reference's color_layer (net_width_condition inputs) cannot take.
      return fail(MIPNERF_B200_EUNSUPPORTED, "net_depth_condition=0 with use_viewdirs");
    }
  }
  const mipnerf_b200_linear& cl = w->linears[d.n_lin - 1];
  CUDA_TRY(mipnerf::launch_linear_f32(feat, feat_k, feat_k, nullptr, 0, 0, 1, cl.weight, cl.bias, raw_rgb, 3,
                                      m, 3, 0, st));
  return MIPNERF_B200_OK;
}

}  // namespace

extern "C" {

const char* mipnerf_b200_last_error(void) { return g_last_error.c_str(); }
int mipnerf_b200_abi_version(void) { return MIPNERF_B200_ABI_VERSION; }

size_t mipnerf_b200_workspace_bytes(const mipnerf_b200_config* cfg, int64_t num_rays, int precision) {
  Dims d;
  if (check_config(cfg, &d) != MIPNERF_B200_OK || num_rays < 0) return 0;
  if (precision == MIPNERF_B200_FP32) {
    const int64_t r = num_rays < kChunkRaysFp32 ? num_rays : kChunkRaysFp32;
    return carve_fp32(cfg, d, r > 0 ? r : 1, nullptr).bytes;
  }
  return mipnerf::tc_workspace_bytes(cfg, num_rays, precision);
}

size_t mipnerf_b200_packed_weights_bytes(const mipnerf_b200_config* cfg, int precision) {
  Dims d;
  if (check_config(cfg, &d) != MIPNERF_B200_OK) return 0;
  return mipnerf::tc_packed_bytes(cfg, precision);
}

int mipnerf_b200_pack_weights(const mipnerf_b200_config* cfg, const mipnerf_b200_weights* w, int precision,
                              void* packed_out, size_t packed_bytes, void* stream) {
  Dims d;
  int rc;
  if ((rc = check_config(cfg, &d))) return rc;
  if ((rc = check_weights(cfg, d, w))) return rc;
  if (!packed_out) return fail(MIPNERF_B200_EINVAL, "packed_out is NULL");
  const size_t need = mipnerf::tc_packed_bytes(cfg, precision);
  if (need == 0)
    return fail(MIPNERF_B200_EUNSUPPORTED, "no tensor-core kernel for this MLP shape / precision %d", precision);
  if (packed_bytes < need)
    return fail(MIPNERF_B200_EWORKSPACE, "packed buffer %zu < %zu bytes", packed_bytes, need);
  cudaError_t e = mipnerf::tc_pack_weights(cfg, w, precision, packed_out, (cudaStream_t)stream);
  if (e != cudaSuccess) return fail(MIPNERF_B200_ECUDA, "pack_weights: %s", cudaGetErrorString(e));
  return MIPNERF_B200_OK;
}

// randomized with density_noise > 0 (models/mip_nerf.py:232-233): the injected-noise entry points need the normals too
static int check_density_normals(const mipnerf_b200_config* cfg, int randomized, const mipnerf_b200_rng* rng,
                                 const mipnerf_b200_level_out* outs, int64_t num_rays) {
  if (!randomized || !(cfg->density_noise > 0.f) || rng || num_rays == 0) return MIPNERF_B200_OK;
  for (int l = 0; l < cfg->num_levels; ++l)
    if (!outs[l].density_normal)
      return fail(MIPNERF_B200_EINVAL,
                  "randomized=1 with density_noise > 0 needs outs[%d].density_normal (injected noise) or the _rng "
                  "entry point (in-kernel Philox)", l);
  return MIPNERF_B200_OK;
}

static int forward_impl(const mipnerf_b200_config* cfg, const mipnerf_b200_weights* w,
                        const mipnerf_b200_rays* rays, int randomized, const float* t_rand,
                        const float* u_jitter, const mipnerf_b200_rng* rng, int white_bkgd, int precision,
                        mipnerf_b200_level_out* outs, void* workspace, size_t workspace_bytes, void* stream) {
  Dims d;
  int rc;
  if ((rc = check_config(cfg, &d))) return rc;
  if ((rc = check_weights(cfg, d, w))) return rc;
  if ((rc = check_rays(rays))) return rc;
  if (!outs) return fail(MIPNERF_B200_EINVAL, "outs is NULL");
  if (cfg->use_viewdirs && rays->num_rays > 0 && !rays->viewdirs)
    return fail(MIPNERF_B200_EINVAL, "use_viewdirs but rays.viewdirs is NULL");
  if (randomized && !rng && (!t_rand || (cfg->num_levels > 1 && !u_jitter)))
    return fail(MIPNERF_B200_EINVAL,
                "randomized=1 needs t_rand and u_jitter (injected noise) or the _rng entry point (in-kernel Philox)");
  for (int l = 0; l < cfg->num_levels; ++l)
    if (rays->num_rays > 0 && (!outs[l].comp_rgb || !outs[l].distance || !outs[l].acc))
      return fail(MIPNERF_B200_EINVAL, "outs[%d] misses comp_rgb/distance/acc", l);
  if ((rc = check_density_normals(cfg, randomized, rng, outs, rays->num_rays))) return rc;
  const size_t need = mipnerf_b200_workspace_bytes(cfg, rays->num_rays, precision);
  if (rays->num_rays > 0 && (!workspace || workspace_bytes < need))
    return fail(MIPNERF_B200_EWORKSPACE, "workspace %zu < %zu bytes", workspace_bytes, need);
  cudaStream_t st = (cudaStream_t)stream;
  const int n = cfg->num_samples;
  const float rgb_scale = (float)(1.0 + 2.0 * (double)cfg->rgb_padding);

  if (precision != MIPNERF_B200_FP32) {
    if (!mipnerf::tc_supported(cfg, precision))
      return fail(MIPNERF_B200_EUNSUPPORTED,
                  "tensor-core path supports the 8x256 / 1x128 / N=128 model with min_deg_point 0, max_deg_point 1..16, "
                  "deg_view 1..4 and precision bf16|fp16|fp16x3|bf16x3; use MIPNERF_B200_FP32 for other shapes");
    if (!w->packed || w->packed_precision != precision ||
        w->packed_bytes < mipnerf::tc_packed_bytes(cfg, precision))
      return fail(MIPNERF_B200_EINVAL, "weights->packed missing or packed for another precision");
    cudaError_t e = mipnerf::tc_forward(cfg, w, rays, randomized, t_rand, u_jitter, rng, white_bkgd, precision,
                                        outs, workspace, workspace_bytes, st);
    if (e != cudaSuccess) return fail(MIPNERF_B200_ECUDA, "tc_forward: %s", cudaGetErrorString(e));
    return MIPNERF_B200_OK;
  }

  for (int64_t off = 0; off < rays->num_rays; off += kChunkRaysFp32) {
    const int64_t cnt = (rays->num_rays - off) < kChunkRaysFp32 ? (rays->num_rays - off) : kChunkRaysFp32;
    const mipnerf_b200_rays rc_ = offset_rays(*rays, off, cnt);
    const Fp32Scratch s = carve_fp32(cfg, d, cnt, workspace);
    if (cfg->use_viewdirs)
      CUDA_TRY(mipnerf::launch_pos_enc(rc_.viewdirs, s.venc, cnt, 0, cfg->deg_view, 1, st));
    const float *t_prev = nullptr, *w_prev = nullptr;
    for (int l = 0; l < cfg->num_levels; ++l) {
      float* t_cur = outs[l].t_samples ? outs[l].t_samples + off * (n + 1) : s.t[l & 1];
      float* w_cur = outs[l].weights ? outs[l].weights + off * n : s.w[l & 1];
      if (l == 0) {
        CUDA_TRY(mipnerf::launch_coarse_t(rc_.near, rc_.far, mipnerf::level_draws(randomized, t_rand, rng, off, 0, n + 1),
                                          t_cur, cnt, n, randomized, cfg->disparity, st));
      } else {
        CUDA_TRY(mipnerf::launch_resample(t_prev, w_prev, mipnerf::level_draws(randomized, u_jitter, rng, off, 1 + l, n + 1),
                                          t_cur, outs[l].inds ? outs[l].inds + off * (n + 1) : nullptr, cnt, n, n + 1,
                                          randomized, 1, cfg->resample_padding, st));
      }
      CUDA_TRY(mipnerf::launch_ipe_from_t(rc_.origins, rc_.directions, rc_.radii, t_cur, s.enc, cnt, n,
                                          cfg->min_deg_point, cfg->max_deg_point, cfg->disable_integration,
                                          st));
      if ((rc = mlp_forward_fp32(cfg, d, w, s.enc, cfg->use_viewdirs ? s.venc : nullptr, cnt, n, s, s.raw_rgb,
                                 s.raw_density, st)))
        return rc;
      CUDA_TRY(mipnerf::launch_add_density_noise(                                   // models/mip_nerf.py:232-233
          s.raw_density, mipnerf::density_noise_draws(cfg, randomized, outs[l].density_normal, rng, off, l, n), cnt, n, st));
      CUDA_TRY(mipnerf::launch_composite(s.raw_rgb, s.raw_density, t_cur, rc_.directions,
                                         outs[l].comp_rgb + off * 3, outs[l].distance + off, outs[l].acc + off,
                                         w_cur, cnt, n, white_bkgd, 1, cfg->density_bias, rgb_scale,
                                         cfg->rgb_padding, st));
      t_prev = t_cur;
      w_prev = w_cur;
    }
  }
  return MIPNERF_B200_OK;
}

int mipnerf_b200_forward(const mipnerf_b200_config* cfg, const mipnerf_b200_weights* w,
                         const mipnerf_b200_rays* rays, int randomized, const float* t_rand,
                         const float* u_jitter, int white_bkgd, int precision, mipnerf_b200_level_out* outs,
                         void* workspace, size_t workspace_bytes, void* stream) {
  return forward_impl(cfg, w, rays, randomized, t_rand, u_jitter, nullptr, white_bkgd, precision, outs, workspace,
                      workspace_bytes, stream);
}

int mipnerf_b200_forward_rng(const mipnerf_b200_config* cfg, const mipnerf_b200_weights* w,
                             const mipnerf_b200_rays* rays, const mipnerf_b200_rng* rng, int white_bkgd,
                             int precision, mipnerf_b200_level_out* outs, void* workspace,
                             size_t workspace_bytes, void* stream) {
  if (!rng) return fail(MIPNERF_B200_EINVAL, "rng is NULL");
  return forward_impl(cfg, w, rays, 1, nullptr, nullptr, rng, white_bkgd, precision, outs, workspace,
                      workspace_bytes, stream);
}

int mipnerf_b200_philox_normal(const mipnerf_b200_rng* rng, int level, int64_t num_rays, int num_samples, float* out,
                               void* stream) {
  if (!rng || level < 0 || level >= 64 || num_rays < 0 || num_samples < 1 || (num_rays > 0 && !out))
    return fail(MIPNERF_B200_EINVAL, "bad argument");
  const mipnerf::Draws d = mipnerf::draws_philox(rng->seed, rng->offset, 0, mipnerf::kDensityNoiseStream + level, 1.f);
  CUDA_TRY(mipnerf::launch_philox_normal(d, out, num_rays, num_samples, (cudaStream_t)stream));
  return MIPNERF_B200_OK;
}

int mipnerf_b200_philox_uniform(const mipnerf_b200_rng* rng, int stream_id, int64_t num_rays, int ncols, float* out,
                                void* stream) {
  if (!rng || stream_id < 0 || num_rays < 0 || ncols < 1 || (num_rays > 0 && !out))
    return fail(MIPNERF_B200_EINVAL, "bad argument");
  const mipnerf::Draws d = mipnerf::level_draws(1, nullptr, rng, 0, stream_id, ncols);
  CUDA_TRY(mipnerf::launch_philox_uniform(d, out, num_rays, ncols, (cudaStream_t)stream));
  return MIPNERF_B200_OK;
}

// ---- training step -------------------------------------------------------------------------------
namespace {
constexpr int kMaxTrainDepth = 16;
struct TrainScratch {
  float *enc, *venc, *h[kMaxTrainDepth], *bott, *v, *raw_rgb, *raw_density;
  float *d_a, *d_b, *d_v, *d_raw_rgb, *d_raw_density, *part, *t[2], *w[2];
  float* vrow;      // tensor-core mode: per-ray view-direction bias [rays, net_width_condition]
  uint8_t* images;  // tensor-core mode: packed B operands (kTrainImages x kTrainImageBytes)
  size_t bytes;
};
constexpr int kTrainImages = 2 * kMaxTrainDepth + 8;
constexpr size_t kTrainImageBytes = 131072;  // 256 x 256 x 16 bit

TrainScratch carve_train(const mipnerf_b200_config* c, const Dims& d, int64_t rays, void* base) {
  TrainScratch s{};
  const size_t m = (size_t)rays * c->num_samples;
  size_t off = 0;
  auto take = [&](size_t elems) {
    float* p = base ? reinterpret_cast<float*>(static_cast<char*>(base) + off) : nullptr;
    off += align_up(elems * sizeof(float));
    return p;
  };
  s.enc = take(m * d.xyz_dim);
  s.venc = take((size_t)rays * d.view_dim);
  for (int i = 0; i < c->net_depth; ++i) s.h[i] = take(m * c->net_width);
  s.bott = take(m * c->net_width);
  s.v = take(m * c->net_width_condition);
  s.raw_rgb = take(m * 3);
  s.raw_density = take(m);
  s.d_a = take(m * c->net_width);
  s.d_b = take(m * c->net_width);
  s.d_v = take(m * c->net_width_condition);
  s.d_raw_rgb = take(m * 3);
  s.d_raw_density = take(m);
  const size_t max_n = c->net_width > c->net_width_condition ? c->net_width : c->net_width_condition;
  const size_t max_k = (size_t)c->net_width + (d.xyz_dim > d.view_dim ? d.xyz_dim : d.view_dim) + 1;
  s.part = take((size_t)mipnerf::kWgradMaxSlices * max_n * max_k);
  for (int i = 0; i < 2; ++i) {
    s.t[i] = take((size_t)rays * (c->num_samples + 1));
    s.w[i] = take(m);
  }
  s.vrow = take((size_t)rays * c->net_width_condition);
  s.images = reinterpret_cast<uint8_t*>(take(kTrainImages * kTrainImageBytes / sizeof(float)));
  s.bytes = off;
  return s;
}

// Scratch of the fused tensor-core training step (forward = the level kernels with the activation dump, backward on
// 16-bit tile images, train_t16.cu).  Overlays the same workspace as TrainScratch.
struct FusedScratch {
  uint8_t *act[2], *v[2];                // forward dump per level: [9][rays][64 KB], [rays][32 KB]
  float *raw_rgb[2], *raw_density[2];    // raw heads per level
  float *enc, *venc, *d_raw_rgb, *d_raw_density, *part, *t[2], *w[2];
  uint8_t *enc16;                        // the IPE features as a tile image [rays][2 slabs] (96 columns + zero padding)
  uint8_t *relu_bits;                    // [m][32 B]: sign mask of the layer input the current wgrad streams
  uint8_t *d_v, *d_a, *d_b;              // gradient tile images: [rays][32 KB], [rays][64 KB] x 2
  uint8_t *images, *packed, *tcws;
  size_t tcws_bytes, bytes;
};

FusedScratch carve_fused(const mipnerf_b200_config* c, const Dims& d, int64_t rays, int precision, void* base) {
  FusedScratch s{};
  const size_t m = (size_t)rays * c->num_samples;
  size_t off = 0;
  auto take_bytes = [&](size_t bytes) {
    uint8_t* p = base ? static_cast<uint8_t*>(base) + off : nullptr;
    off += align_up(bytes);
    return p;
  };
  auto take = [&](size_t elems) { return reinterpret_cast<float*>(take_bytes(elems * sizeof(float))); };
  for (int l = 0; l < 2; ++l) {
    s.act[l] = take_bytes((size_t)9 * rays * 65536);
    s.v[l] = take_bytes((size_t)rays * 32768);
    s.raw_rgb[l] = take(m * 3);
    s.raw_density[l] = take(m);
    s.t[l] = take((size_t)rays * (c->num_samples + 1));
    s.w[l] = take(m);
  }
  s.enc = take(m * d.xyz_dim);
  s.venc = take((size_t)rays * d.view_dim);
  s.d_raw_rgb = take(m * 3);
  s.d_raw_density = take(m);
  s.enc16 = take_bytes((size_t)rays * 32768);
  s.relu_bits = take_bytes(m * 32);
  s.d_v = take_bytes((size_t)rays * 32768);
  s.d_a = take_bytes((size_t)rays * 65536);
  s.d_b = take_bytes((size_t)rays * 65536);
  const size_t max_n = c->net_width > c->net_width_condition ? c->net_width : c->net_width_condition;
  const size_t max_k = (size_t)c->net_width + (d.xyz_dim > d.view_dim ? d.xyz_dim : d.view_dim) + 1;
  s.part = take((size_t)mipnerf::kWgradMaxSlices * max_n * max_k);
  s.images = take_bytes((size_t)kTrainImages * kTrainImageBytes);
  s.packed = take_bytes(mipnerf::tc_packed_bytes(c, precision));
  s.tcws_bytes = mipnerf::tc_workspace_bytes(c, rays, precision);
  s.tcws = take_bytes(s.tcws_bytes);
  s.bytes = off;
  return s;
}

// The fused step needs the level kernels' architecture (8 x 256 trunk, 128 samples, ...) and at most two levels.
// MIPNERF_B200_TRAIN_FUSED=0 keeps the per-layer tensor-core path (A/B runs).
bool train_fused_supported(const mipnerf_b200_config* c, int precision) {
  return (precision == MIPNERF_B200_BF16 || precision == MIPNERF_B200_FP16) && mipnerf::tc_supported(c, precision) &&
         mipnerf::tc_default_degrees(c) &&  // the backward's tile images carry the full 96 / 27 encodings
         c->num_levels <= 2 && c->net_depth == 8;
}

// Tensor-core GEMMs of the training step exist for the default widths only (linear_tc.cu).
bool train_tc_supported(const mipnerf_b200_config* c, const Dims& d) {
  if (!(c->net_width == 256 && c->net_width_condition == 128 && d.xyz_dim == 96 && d.view_dim == 27 &&
        c->net_depth <= kMaxTrainDepth))
    return false;
  // packed-operand slots the step needs (forward + skip + transposed dgrad images + bottleneck / view layer x 2):
  // must fit the kTrainImages slots carved from the workspace
  int slots = 4;
  for (int i = 0; i < c->net_depth; ++i) slots += 1 + (i > 1 && (i - 1) % c->skip_index == 0 ? 1 : 0) + (i > 0 ? 1 : 0);
  return slots <= kTrainImages;
}

int check_train_config(const mipnerf_b200_config* c) {
  if (!c->use_viewdirs || c->net_depth_condition != 1)
    return fail(MIPNERF_B200_EUNSUPPORTED, "training: use_viewdirs=True with one view layer only");
  if (c->net_depth > kMaxTrainDepth)
    return fail(MIPNERF_B200_EUNSUPPORTED, "training: net_depth <= %d", kMaxTrainDepth);
  return MIPNERF_B200_OK;
}

inline bool takes_skip(const mipnerf_b200_config* c, int layer) {  // models/mip_nerf.py:40-42
  return layer > 1 && (layer - 1) % c->skip_index == 0;
}
}  // namespace

size_t mipnerf_b200_train_workspace_bytes(const mipnerf_b200_config* cfg, int64_t num_rays) {
  Dims d;
  if (check_config(cfg, &d) != MIPNERF_B200_OK || check_train_config(cfg) != MIPNERF_B200_OK || num_rays < 0)
    return 0;
  const int64_t r = num_rays < kChunkRaysFp32 ? num_rays : kChunkRaysFp32;
  size_t bytes = carve_train(cfg, d, r > 0 ? r : 1, nullptr).bytes;
  for (int precision : {MIPNERF_B200_BF16, MIPNERF_B200_FP16})  // the fused tensor-core step overlays the same buffer
    if (train_fused_supported(cfg, precision)) {
      const size_t f = carve_fused(cfg, d, r > 0 ? r : 1, precision, nullptr).bytes;
      if (f > bytes) bytes = f;
    }
  return bytes;
}

static int forward_backward_fused(const mipnerf_b200_config* cfg, const Dims& d, const mipnerf_b200_weights* w,
                                  const mipnerf_b200_rays* rays, int randomized, const float* t_rand,
                                  const float* u_jitter, const mipnerf_b200_rng* rng, int white_bkgd, int precision,
                                  const mipnerf_b200_loss* loss, mipnerf_b200_level_out* outs,
                                  const mipnerf_b200_linear_grad* grads, bool* touched, void* workspace,
                                  cudaStream_t st, const uint64_t* rng_state) {
  const int n = cfg->num_samples, depth = cfg->net_depth, W = cfg->net_width, Wc = cfg->net_width_condition;
  const float rgb_scale = (float)(1.0 + 2.0 * (double)cfg->rgb_padding);
  const int64_t B = rays->num_rays;
  const FusedScratch s0 = carve_fused(cfg, d, B < kChunkRaysFp32 ? B : kChunkRaysFp32, precision, workspace);
  // ---- once per call (the weights change every optimiser step): the level kernels' packed image, and the
  //      transposed B operands of the dgrad chain  bwd[i] = W_i[:, :256]^T  (slots depth / depth+1: bottleneck, view)
  mipnerf_b200_weights wl = *w;
  wl.packed = s0.packed;
  CUDA_TRY(mipnerf::tc_pack_weights(cfg, w, precision, s0.packed, st, /*with_v3=*/false));
  const uint8_t* img_bwd[kMaxTrainDepth + 2] = {nullptr};
  {
    int slot = 0;
    auto pack = [&](const mipnerf_b200_linear& l, int nn, int kk, const uint8_t** out) {
      uint8_t* dst = s0.images + (size_t)(slot++) * kTrainImageBytes;
      *out = dst;
      return mipnerf::launch_pack_linear_image(l.weight, l.in_features, 0, 1, dst, nn, kk, precision, st);
    };
    for (int i = 1; i < depth; ++i) CUDA_TRY(pack(w->linears[i], W, W, &img_bwd[i]));
    CUDA_TRY(pack(w->linears[depth + 1], W, W, &img_bwd[depth]));
    CUDA_TRY(pack(w->linears[depth + 2], W, Wc, &img_bwd[depth + 1]));
  }
  const mipnerf_b200_linear& dl = w->linears[depth];
  const mipnerf_b200_linear& cl = w->linears[d.n_lin - 1];
  // fp16 gradients underflow: d loss / d activation is ~1e-7 .. 1e-4 per sample (the loss is a mean over the batch),
  // below fp16's 6e-5 normal range.  The backward pass is linear in d loss / d raw, so render_backward emits it
  // scaled by 2^10 (it is bounded by 2/3 per sample: no overflow), every gradient tile image carries that factor, and
  // the fixed-order reduction of the wgrad partials takes it out again.  bf16 has fp32's range: scale 1.
  const float gscale = precision == MIPNERF_B200_FP16 ? 1024.f : 1.f, inv_gscale = 1.f / gscale;
  for (int64_t off = 0; off < B; off += kChunkRaysFp32) {
    const int64_t cnt = (B - off) < kChunkRaysFp32 ? (B - off) : kChunkRaysFp32;
    const int64_t m = cnt * n;
    const mipnerf_b200_rays rc_ = offset_rays(*rays, off, cnt);
    const FusedScratch s = carve_fused(cfg, d, cnt, precision, workspace);
    CUDA_TRY(mipnerf::launch_pos_enc(rc_.viewdirs, s.venc, cnt, 0, cfg->deg_view, 1, st));
    // ---- forward of all levels: two launches, everything the backward needs is left behind as tile images
    mipnerf_b200_level_out lo[2];
    mipnerf::TcTrainDump dump{};
    for (int l = 0; l < cfg->num_levels; ++l) {
      lo[l] = outs[l];
      lo[l].comp_rgb = outs[l].comp_rgb + off * 3, lo[l].distance = outs[l].distance + off, lo[l].acc = outs[l].acc + off;
      lo[l].t_samples = outs[l].t_samples ? outs[l].t_samples + off * (n + 1) : s.t[l];
      lo[l].weights = outs[l].weights ? outs[l].weights + off * n : s.w[l];
      lo[l].inds = outs[l].inds ? outs[l].inds + off * (n + 1) : nullptr;
      lo[l].density_normal = outs[l].density_normal ? outs[l].density_normal + off * n : nullptr;
      dump.act[l] = s.act[l], dump.v[l] = s.v[l], dump.raw_rgb[l] = s.raw_rgb[l], dump.raw_density[l] = s.raw_density[l];
    }
    dump.rng_state = rng_state;
    CUDA_TRY(mipnerf::tc_forward(cfg, &wl, &rc_, randomized, t_rand ? t_rand + off * (n + 1) : nullptr,
                                 u_jitter ? u_jitter + off * (n + 1) : nullptr, rng, white_bkgd, precision, lo, s.tcws,
                                 s.tcws_bytes, st, &dump, off));
    // MIPNERF_B200_TRAIN_MASKBITS=0: the dgrad GEMMs read the ReLU mask from the activation tile images again (A/B)
    const char* bits_env = getenv("MIPNERF_B200_TRAIN_MASKBITS");
    const bool use_bits = !(bits_env && bits_env[0] == '0');
    auto wgrad = [&](int idx, const void* dy16, const void* x1, int k1, const void* x2, int x2_t16, int k2, int div,
                     bool emit_mask = false) {
      const mipnerf_b200_linear& l = w->linears[idx];
      int slices = 0;
      cudaError_t e2 = mipnerf::launch_wgrad_mn_partials(dy16, 1, l.out_features, x1, 1, k1, k1, x2, x2_t16, k2, k2, div,
                                                         s.part, m, mipnerf::kWgradMaxSlices, precision, &slices, st,
                                                         emit_mask && use_bits ? s.relu_bits : nullptr);
      if (e2 != cudaSuccess) return e2;
      e2 = mipnerf::launch_wgrad_reduce(s.part, slices, l.out_features, k1 + k2, grads[idx].weight_grad,
                                        grads[idx].bias_grad, touched[idx] ? 1 : 0, st, inv_gscale);
      touched[idx] = true;
      return e2;
    };
    for (int l = 0; l < cfg->num_levels; ++l) {
      const float* t_cur = lo[l].t_samples;
      const uint8_t* act = s.act[l];
      auto h16 = [&](int i) { return act + (size_t)i * cnt * 65536; };  // h_0..h_7, 8 = bottleneck
      // the IPE features again (operand of two wgrads; the level kernel keeps its own 16-bit copy on chip), written
      // straight into a tile image so that those wgrads stage them by bulk copy like every other operand
      CUDA_TRY(mipnerf::launch_ipe_t16(rc_.origins, rc_.directions, rc_.radii, t_cur, s.enc16, cnt, n,
                                       cfg->disable_integration, precision, st));
      CUDA_TRY(mipnerf::launch_render_backward(
          s.raw_rgb[l], s.raw_density[l], t_cur, rc_.directions, loss->target_rgb + off * 3,
          loss->lossmult ? loss->lossmult + off : nullptr, loss->mask_sum, loss->level_mse_mult[l] * gscale,
          loss->level_dist_mult[l] * loss->dist_scale * gscale, white_bkgd, cfg->density_bias, rgb_scale,
          cfg->rgb_padding, s.d_raw_rgb, s.d_raw_density,
          loss->per_ray_sqerr ? loss->per_ray_sqerr + (int64_t)l * B + off : nullptr,
          loss->per_ray_distloss ? loss->per_ray_distloss + (int64_t)l * B + off : nullptr, cnt, n, st));
      // colour head, view layer                                          (models/mip_nerf.py:106-110)
      CUDA_TRY(mipnerf::launch_wgrad_small_n_t16(s.d_raw_rgb, 3, s.v[l], Wc, s.part, grads[d.n_lin - 1].weight_grad,
                                                 grads[d.n_lin - 1].bias_grad, touched[d.n_lin - 1] ? 1 : 0, m,
                                                 precision, st, inv_gscale));
      touched[d.n_lin - 1] = true;
      CUDA_TRY(mipnerf::launch_color_dgrad_t16(s.d_raw_rgb, cl.weight, s.v[l], s.d_v, m, Wc, precision, st));
      CUDA_TRY(wgrad(depth + 2, s.d_v, h16(8), W, s.venc, 0, d.view_dim, n));
      CUDA_TRY(mipnerf::launch_linear_t16(s.d_v, img_bwd[depth + 1], s.d_a, m, W, Wc, nullptr, nullptr, nullptr,
                                          precision, st));
      // bottleneck + density head share h_7                              (models/mip_nerf.py:98-101)
      CUDA_TRY(wgrad(depth + 1, s.d_a, h16(depth - 1), W, nullptr, 0, 0, 1, /*emit_mask=*/true));  // sign mask of h_7
      CUDA_TRY(mipnerf::launch_wgrad_small_n_t16(s.d_raw_density, 1, h16(depth - 1), W, s.part,
                                                 grads[depth].weight_grad, grads[depth].bias_grad,
                                                 touched[depth] ? 1 : 0, m, precision, st, inv_gscale));
      touched[depth] = true;
      CUDA_TRY(mipnerf::launch_linear_t16(s.d_a, img_bwd[depth], s.d_b, m, W, W, s.d_raw_density, dl.weight,
                                          use_bits ? nullptr : h16(depth - 1), precision, st,
                                          use_bits ? s.relu_bits : nullptr));
      // trunk                                                            (models/mip_nerf.py:93-97)
      uint8_t *cur = s.d_b, *other = s.d_a;
      for (int i = depth - 1; i >= 0; --i) {
        const bool skip = takes_skip(cfg, i);
        if (i == 0) CUDA_TRY(wgrad(0, cur, s.enc16, d.xyz_dim, nullptr, 0, 0, 1));
        else CUDA_TRY(wgrad(i, cur, h16(i - 1), W, skip ? s.enc16 : nullptr, 1, skip ? d.xyz_dim : 0, 1, true));
        if (i > 0) {  // the wgrad just streamed h_{i-1} and left its sign mask behind: 32 B per row instead of 512
          CUDA_TRY(mipnerf::launch_linear_t16(cur, img_bwd[i], other, m, W, W, nullptr, nullptr,
                                              use_bits ? nullptr : h16(i - 1), precision, st,
                                              use_bits ? s.relu_bits : nullptr));
          uint8_t* tmp = cur;
          cur = other;
          other = tmp;
        }
      }
    }
  }
  return MIPNERF_B200_OK;
}

static int forward_backward_impl(const mipnerf_b200_config* cfg, const mipnerf_b200_weights* w,
                                 const mipnerf_b200_rays* rays, int randomized, const float* t_rand,
                                 const float* u_jitter, const mipnerf_b200_rng* rng, int white_bkgd, int precision,
                                 const mipnerf_b200_loss* loss, mipnerf_b200_level_out* outs,
                                 const mipnerf_b200_linear_grad* grads, int num_grads, int accumulate,
                                 void* workspace, size_t workspace_bytes, void* stream,
                                 const uint64_t* rng_state = nullptr) {
  Dims d;
  int rc;
  if ((rc = check_config(cfg, &d))) return rc;
  if ((rc = check_train_config(cfg))) return rc;
  if ((rc = check_weights(cfg, d, w))) return rc;
  if ((rc = check_rays(rays))) return rc;
  const bool tc = precision == MIPNERF_B200_BF16 || precision == MIPNERF_B200_FP16;
  if (precision == MIPNERF_B200_FP16X3 || precision == MIPNERF_B200_BF16X3)
    return fail(MIPNERF_B200_EUNSUPPORTED,
                "training: the split-operand precisions are forward-only; use FP32 (parity) or BF16 / FP16");
  if (precision != MIPNERF_B200_FP32 && !tc) return fail(MIPNERF_B200_EINVAL, "precision %d", precision);
  if (tc && !train_tc_supported(cfg, d))
    return fail(MIPNERF_B200_EUNSUPPORTED,
                "tensor-core training GEMMs: 8x256 trunk / 128 view layer / 96-d IPE only; use MIPNERF_B200_FP32");
  if (!outs || !loss || !grads) return fail(MIPNERF_B200_EINVAL, "outs / loss / grads is NULL");
  if (num_grads != d.n_lin) return fail(MIPNERF_B200_EINVAL, "expected %d gradient pairs, got %d", d.n_lin, num_grads);
  for (int i = 0; i < d.n_lin; ++i)
    if (!grads[i].weight_grad || !grads[i].bias_grad) return fail(MIPNERF_B200_EINVAL, "grads[%d] has a NULL tensor", i);
  if (!loss->level_mse_mult || !loss->level_dist_mult)
    return fail(MIPNERF_B200_EINVAL, "loss multipliers are NULL");
  if (rays->num_rays > 0 && (!loss->target_rgb || !loss->mask_sum || !rays->viewdirs))
    return fail(MIPNERF_B200_EINVAL, "target_rgb / mask_sum / viewdirs is NULL");
  if (randomized && !rng && (!t_rand || (cfg->num_levels > 1 && !u_jitter)))
    return fail(MIPNERF_B200_EINVAL,
                "randomized=1 needs t_rand and u_jitter (injected noise) or the _rng entry point (in-kernel Philox)");
  for (int l = 0; l < cfg->num_levels; ++l)
    if (rays->num_rays > 0 && (!outs[l].comp_rgb || !outs[l].distance || !outs[l].acc))
      return fail(MIPNERF_B200_EINVAL, "outs[%d] misses comp_rgb/distance/acc", l);
  {
    const int rcn = check_density_normals(cfg, randomized, rng, outs, rays->num_rays);
    if (rcn) return rcn;
  }
  const size_t need = mipnerf_b200_train_workspace_bytes(cfg, rays->num_rays);
  if (rays->num_rays > 0 && (!workspace || workspace_bytes < need))
    return fail(MIPNERF_B200_EWORKSPACE, "workspace %zu < %zu bytes", workspace_bytes, need);
  cudaStream_t st = (cudaStream_t)stream;
  const int n = cfg->num_samples, depth = cfg->net_depth, W = cfg->net_width, Wc = cfg->net_width_condition;
  const float rgb_scale = (float)(1.0 + 2.0 * (double)cfg->rgb_padding);
  const int64_t B = rays->num_rays;
  bool touched[kMaxTrainDepth + 8];
  for (int i = 0; i < d.n_lin; ++i) touched[i] = accumulate != 0;
  if (B == 0 && !accumulate)
    for (int i = 0; i < d.n_lin; ++i) {
      const mipnerf_b200_linear& l = w->linears[i];
      CUDA_TRY(cudaMemsetAsync(grads[i].weight_grad, 0, sizeof(float) * l.in_features * l.out_features, st));
      CUDA_TRY(cudaMemsetAsync(grads[i].bias_grad, 0, sizeof(float) * l.out_features, st));
    }

  {
    const char* fused_env = getenv("MIPNERF_B200_TRAIN_FUSED");
    const bool fused = tc && train_fused_supported(cfg, precision) && !(fused_env && fused_env[0] == '0');
    if (rng_state && !fused)
      return fail(MIPNERF_B200_EUNSUPPORTED,
                  "rng_state: the fused BF16 / FP16 training step only (default architecture, "
                  "MIPNERF_B200_TRAIN_FUSED unset)");
    if (fused && B > 0)
      return forward_backward_fused(cfg, d, w, rays, randomized, t_rand, u_jitter, rng, white_bkgd, precision, loss, outs,
                                    grads, touched, workspace, st, rng_state);
  }
  // ---- tensor-core mode: B operands of every forward / dgrad GEMM, packed once per call (the weights change every
  //      optimiser step).  fwd[i] = W_i[:, :k_main], fwd_skip[i] = W_i[:, 256:352], bwd[i] = W_i[:, :256]^T;
  //      slots depth / depth+1 hold the bottleneck and the view layer.
  const uint8_t *img_fwd[kMaxTrainDepth + 2] = {nullptr}, *img_skip[kMaxTrainDepth] = {nullptr},
                *img_bwd[kMaxTrainDepth + 2] = {nullptr};
  if (tc && B > 0) {
    uint8_t* base = carve_train(cfg, d, B < kChunkRaysFp32 ? B : kChunkRaysFp32, workspace).images;
    int slot = 0;
    auto pack = [&](const mipnerf_b200_linear& l, int off, int transposed, int nn, int kk, const uint8_t** out) {
      uint8_t* dst = base + (size_t)(slot++) * kTrainImageBytes;
      *out = dst;
      return mipnerf::launch_pack_linear_image(l.weight, l.in_features, off, transposed, dst, nn, kk, precision, st);
    };
    for (int i = 0; i < depth; ++i) {
      const mipnerf_b200_linear& l = w->linears[i];
      CUDA_TRY(pack(l, 0, 0, W, i == 0 ? d.xyz_dim : W, &img_fwd[i]));
      if (takes_skip(cfg, i)) CUDA_TRY(pack(l, W, 0, W, d.xyz_dim, &img_skip[i]));
      if (i > 0) CUDA_TRY(pack(l, 0, 1, W, W, &img_bwd[i]));          // B[k_out][n] = W_i[n][k_out]
    }
    CUDA_TRY(pack(w->linears[depth + 1], 0, 0, W, W, &img_fwd[depth]));      // bottleneck
    CUDA_TRY(pack(w->linears[depth + 1], 0, 1, W, W, &img_bwd[depth]));
    CUDA_TRY(pack(w->linears[depth + 2], 0, 0, Wc, W, &img_fwd[depth + 1]));  // view layer, bottleneck columns
    CUDA_TRY(pack(w->linears[depth + 2], 0, 1, W, Wc, &img_bwd[depth + 1]));
  }

  for (int64_t off = 0; off < B; off += kChunkRaysFp32) {
    const int64_t cnt = (B - off) < kChunkRaysFp32 ? (B - off) : kChunkRaysFp32;
    const int64_t m = cnt * n;
    const mipnerf_b200_rays rc_ = offset_rays(*rays, off, cnt);
    const TrainScratch s = carve_train(cfg, d, cnt, workspace);
    CUDA_TRY(mipnerf::launch_pos_enc(rc_.viewdirs, s.venc, cnt, 0, cfg->deg_view, 1, st));
    if (tc) {
      const mipnerf_b200_linear& vl0 = w->linears[depth + 2];
      CUDA_TRY(mipnerf::launch_view_bias_from_enc(s.venc, vl0.weight, vl0.bias, s.vrow, cnt, st));
    }
    // tensor-core mode: wgrad partials on tcgen05 as well (transposing staging: 1.21 vs 1.33 ms per 256x256 layer, the
    // staging is latency-bound).  MIPNERF_B200_WGRAD_TC=0 keeps wgrad on the fp32 FFMA tiles (A/B runs).
    const char* wgrad_env = getenv("MIPNERF_B200_WGRAD_TC");
    const bool wgrad_on_tc = !(wgrad_env && wgrad_env[0] == '0');
    auto wgrad = [&](int idx, const float* dy, const float* x1, int k1, const float* x2, int k2, int div) {
      const mipnerf_b200_linear& l = w->linears[idx];
      if (tc && wgrad_on_tc && mipnerf::wgrad_tc_shape_ok(l.out_features)) {  // tensor-core partials + same reduction
        int slices = 0;
        cudaError_t e2 = mipnerf::launch_wgrad_tc_partials(dy, l.out_features, x1, k1, k1, x2, k2, k2, div, s.part, m,
                                                           mipnerf::kWgradMaxSlices, precision, &slices, st);
        if (e2 != cudaSuccess) return e2;
        e2 = mipnerf::launch_wgrad_reduce(s.part, slices, l.out_features, k1 + k2, grads[idx].weight_grad,
                                          grads[idx].bias_grad, touched[idx] ? 1 : 0, st);
        touched[idx] = true;
        return e2;
      }
      cudaError_t e = mipnerf::launch_wgrad_f32(dy, l.out_features, x1, k1, k1, x2, k2, k2, div, s.part,
                                                grads[idx].weight_grad, grads[idx].bias_grad, touched[idx] ? 1 : 0,
                                                m, st);
      touched[idx] = true;
      return e;
    };
    const float *t_prev = nullptr, *w_prev = nullptr;
    for (int l = 0; l < cfg->num_levels; ++l) {
      float* t_cur = outs[l].t_samples ? outs[l].t_samples + off * (n + 1) : s.t[l & 1];
      float* w_cur = outs[l].weights ? outs[l].weights + off * n : s.w[l & 1];
      // ---- forward of this level, every activation kept (models/mip_nerf.py:203-240)
      if (l == 0) {
        CUDA_TRY(mipnerf::launch_coarse_t(rc_.near, rc_.far, mipnerf::level_draws(randomized, t_rand, rng, off, 0, n + 1),
                                          t_cur, cnt, n, randomized, cfg->disparity, st));
      } else {
        CUDA_TRY(mipnerf::launch_resample(t_prev, w_prev, mipnerf::level_draws(randomized, u_jitter, rng, off, 1 + l, n + 1),
                                          t_cur, outs[l].inds ? outs[l].inds + off * (n + 1) : nullptr, cnt, n, n + 1,
                                          randomized, 1, cfg->resample_padding, st));
      }
      CUDA_TRY(mipnerf::launch_ipe_from_t(rc_.origins, rc_.directions, rc_.radii, t_cur, s.enc, cnt, n,
                                          cfg->min_deg_point, cfg->max_deg_point, cfg->disable_integration, st));
      for (int i = 0; i < depth; ++i) {
        const mipnerf_b200_linear& li = w->linears[i];
        const bool skip = takes_skip(cfg, i);
        const float* in = i == 0 ? s.enc : s.h[i - 1];
        const int k1 = i == 0 ? d.xyz_dim : W;
        if (!tc) {
          CUDA_TRY(mipnerf::launch_linear_f32(in, k1, k1, skip ? s.enc : nullptr, d.xyz_dim, skip ? d.xyz_dim : 0, 1,
                                              li.weight, li.bias, s.h[i], W, m, W, 1, st));
        } else if (!skip) {
          CUDA_TRY(mipnerf::launch_linear_tc(in, k1, img_fwd[i], s.h[i], W, m, W, k1, li.bias, nullptr, 1, nullptr,
                                             nullptr, nullptr, nullptr, 1, precision, st));
        } else {  // cat([h, enc]) as two K passes: the second adds the first's partial sums, the bias and the ReLU
          CUDA_TRY(mipnerf::launch_linear_tc(in, k1, img_fwd[i], s.h[i], W, m, W, k1, nullptr, nullptr, 1, nullptr,
                                             nullptr, nullptr, nullptr, 0, precision, st));
          CUDA_TRY(mipnerf::launch_linear_tc(s.enc, d.xyz_dim, img_skip[i], s.h[i], W, m, W, d.xyz_dim, li.bias, nullptr,
                                             1, s.h[i], nullptr, nullptr, nullptr, 1, precision, st));
        }
      }
      const float* h_last = s.h[depth - 1];
      const mipnerf_b200_linear& dl = w->linears[depth];
      const mipnerf_b200_linear& el = w->linears[depth + 1];
      const mipnerf_b200_linear& vl = w->linears[depth + 2];
      const mipnerf_b200_linear& cl = w->linears[d.n_lin - 1];
      CUDA_TRY(mipnerf::launch_linear_f32(h_last, W, W, nullptr, 0, 0, 1, dl.weight, dl.bias, s.raw_density, 1, m, 1,
                                          0, st));
      // density noise (models/mip_nerf.py:232-233), in place: render_backward then takes softplus' at the noisy point
      CUDA_TRY(mipnerf::launch_add_density_noise(
          s.raw_density, mipnerf::density_noise_draws(cfg, randomized, outs[l].density_normal, rng, off, l, n), cnt, n, st));
      if (!tc) {
        CUDA_TRY(mipnerf::launch_linear_f32(h_last, W, W, nullptr, 0, 0, 1, el.weight, el.bias, s.bott, W, m, W, 0, st));
        CUDA_TRY(mipnerf::launch_linear_f32(s.bott, W, W, s.venc, d.view_dim, d.view_dim, n, vl.weight, vl.bias, s.v,
                                            Wc, m, Wc, 1, st));
      } else {
        CUDA_TRY(mipnerf::launch_linear_tc(h_last, W, img_fwd[depth], s.bott, W, m, W, W, el.bias, nullptr, 1, nullptr,
                                           nullptr, nullptr, nullptr, 0, precision, st));
        CUDA_TRY(mipnerf::launch_linear_tc(s.bott, W, img_fwd[depth + 1], s.v, Wc, m, Wc, W, nullptr, s.vrow, n, nullptr,
                                           nullptr, nullptr, nullptr, 1, precision, st));
      }
      CUDA_TRY(mipnerf::launch_linear_f32(s.v, Wc, Wc, nullptr, 0, 0, 1, cl.weight, cl.bias, s.raw_rgb, 3, m, 3, 0,
                                          st));
      CUDA_TRY(mipnerf::launch_composite(s.raw_rgb, s.raw_density, t_cur, rc_.directions, outs[l].comp_rgb + off * 3,
                                         outs[l].distance + off, outs[l].acc + off, w_cur, cnt, n, white_bkgd, 1,
                                         cfg->density_bias, rgb_scale, cfg->rgb_padding, st));

      // ---- backward of this level (its fenceposts are constants, so levels are independent here)
      CUDA_TRY(mipnerf::launch_render_backward(
          s.raw_rgb, s.raw_density, t_cur, rc_.directions, loss->target_rgb + off * 3,
          loss->lossmult ? loss->lossmult + off : nullptr, loss->mask_sum, loss->level_mse_mult[l],
          loss->level_dist_mult[l] * loss->dist_scale, white_bkgd, cfg->density_bias, rgb_scale, cfg->rgb_padding,
          s.d_raw_rgb, s.d_raw_density, loss->per_ray_sqerr ? loss->per_ray_sqerr + (int64_t)l * B + off : nullptr,
          loss->per_ray_distloss ? loss->per_ray_distloss + (int64_t)l * B + off : nullptr, cnt, n, st));
      // colour head, view layer                                          (models/mip_nerf.py:106-110)
      CUDA_TRY(wgrad(d.n_lin - 1, s.d_raw_rgb, s.v, Wc, nullptr, 0, 1));
      CUDA_TRY(mipnerf::launch_color_dgrad(s.d_raw_rgb, cl.weight, s.v, s.d_v, m, Wc, st));
      CUDA_TRY(wgrad(depth + 2, s.d_v, s.bott, W, s.venc, d.view_dim, n));
      if (!tc)
        CUDA_TRY(mipnerf::launch_dgrad_f32(s.d_v, Wc, vl.weight, W + d.view_dim, nullptr, nullptr, nullptr, s.d_a, m, W,
                                           st));
      else
        CUDA_TRY(mipnerf::launch_linear_tc(s.d_v, Wc, img_bwd[depth + 1], s.d_a, W, m, W, Wc, nullptr, nullptr, 1,
                                           nullptr, nullptr, nullptr, nullptr, 0, precision, st));
      // bottleneck + density head share h_last                           (models/mip_nerf.py:98-101)
      CUDA_TRY(wgrad(depth + 1, s.d_a, h_last, W, nullptr, 0, 1));
      CUDA_TRY(wgrad(depth, s.d_raw_density, h_last, W, nullptr, 0, 1));
      if (!tc)
        CUDA_TRY(mipnerf::launch_dgrad_f32(s.d_a, W, el.weight, W, s.d_raw_density, dl.weight, h_last, s.d_b, m, W, st));
      else
        CUDA_TRY(mipnerf::launch_linear_tc(s.d_a, W, img_bwd[depth], s.d_b, W, m, W, W, nullptr, nullptr, 1, nullptr,
                                           s.d_raw_density, dl.weight, h_last, 0, precision, st));
      // trunk                                                            (models/mip_nerf.py:93-97)
      float *cur = s.d_b, *other = s.d_a;
      for (int i = depth - 1; i >= 0; --i) {
        const bool skip = takes_skip(cfg, i);
        const float* in = i == 0 ? s.enc : s.h[i - 1];
        const int k1 = i == 0 ? d.xyz_dim : W;
        CUDA_TRY(wgrad(i, cur, in, k1, skip ? s.enc : nullptr, skip ? d.xyz_dim : 0, 1));
        if (i > 0) {
          if (!tc)
            CUDA_TRY(mipnerf::launch_dgrad_f32(cur, W, w->linears[i].weight, k1 + (skip ? d.xyz_dim : 0), nullptr,
                                               nullptr, s.h[i - 1], other, m, W, st));
          else
            CUDA_TRY(mipnerf::launch_linear_tc(cur, W, img_bwd[i], other, W, m, W, W, nullptr, nullptr, 1, nullptr,
                                               nullptr, nullptr, s.h[i - 1], 0, precision, st));
          float* tmp = cur;
          cur = other;
          other = tmp;
        }
      }
      t_prev = t_cur;
      w_prev = w_cur;
    }
  }
  return MIPNERF_B200_OK;
}

int mipnerf_b200_forward_backward(const mipnerf_b200_config* cfg, const mipnerf_b200_weights* w,
                                  const mipnerf_b200_rays* rays, int randomized, const float* t_rand,
                                  const float* u_jitter, int white_bkgd, int precision,
                                  const mipnerf_b200_loss* loss, mipnerf_b200_level_out* outs,
                                  const mipnerf_b200_linear_grad* grads, int num_grads, int accumulate,
                                  void* workspace, size_t workspace_bytes, void* stream) {
  return forward_backward_impl(cfg, w, rays, randomized, t_rand, u_jitter, nullptr, white_bkgd, precision, loss, outs,
                               grads, num_grads, accumulate, workspace, workspace_bytes, stream);
}

int mipnerf_b200_forward_backward_rng(const mipnerf_b200_config* cfg, const mipnerf_b200_weights* w,
                                      const mipnerf_b200_rays* rays, const mipnerf_b200_rng* rng, int white_bkgd,
                                      int precision, const mipnerf_b200_loss* loss, mipnerf_b200_level_out* outs,
                                      const mipnerf_b200_linear_grad* grads, int num_grads, int accumulate,
                                      void* workspace, size_t workspace_bytes, void* stream) {
  if (!rng) return fail(MIPNERF_B200_EINVAL, "rng is NULL");
  return forward_backward_impl(cfg, w, rays, 1, nullptr, nullptr, rng, white_bkgd, precision, loss, outs, grads, num_grads,
                               accumulate, workspace, workspace_bytes, stream);
}

int mipnerf_b200_forward_backward_rng_state(const mipnerf_b200_config* cfg, const mipnerf_b200_weights* w,
                                            const mipnerf_b200_rays* rays, const uint64_t* rng_state, int white_bkgd,
                                            int precision, const mipnerf_b200_loss* loss, mipnerf_b200_level_out* outs,
                                            const mipnerf_b200_linear_grad* grads, int num_grads, int accumulate,
                                            void* workspace, size_t workspace_bytes, void* stream) {
  if (!rng_state) return fail(MIPNERF_B200_EINVAL, "rng_state is NULL");
  const mipnerf_b200_rng placeholder = {0, 0};  // selects the in-kernel draws; the kernel reads rng_state instead
  return forward_backward_impl(cfg, w, rays, 1, nullptr, nullptr, &placeholder, white_bkgd, precision, loss, outs, grads,
                               num_grads, accumulate, workspace, workspace_bytes, stream, rng_state);
}

int mipnerf_b200_linear_tc(const float* x, const float* weight, const float* bias, float* y, int64_t m, int n,
                           int k, int relu, int precision, void* scratch, size_t scratch_bytes, void* stream) {
  if (m < 0 || !mipnerf::linear_tc_shape_ok(n, k))
    return fail(MIPNERF_B200_EUNSUPPORTED, "linear_tc: n in {128,256}, k in {96,128,256} (got n=%d k=%d)", n, k);
  if (precision != MIPNERF_B200_BF16 && precision != MIPNERF_B200_FP16)
    return fail(MIPNERF_B200_EINVAL, "linear_tc: precision must be BF16 or FP16");
  if (m > 0 && (!x || !weight || !y)) return fail(MIPNERF_B200_EINVAL, "NULL tensor");
  const size_t need = mipnerf::linear_tc_image_bytes(n, k);
  if (!scratch || scratch_bytes < need) return fail(MIPNERF_B200_EWORKSPACE, "scratch %zu < %zu bytes", scratch_bytes, need);
  cudaStream_t st = (cudaStream_t)stream;
  CUDA_TRY(mipnerf::launch_pack_linear_image(weight, k, 0, 0, scratch, n, k, precision, st));
  CUDA_TRY(mipnerf::launch_linear_tc(x, k, scratch, y, n, m, n, k, bias, nullptr, 1, nullptr, nullptr, nullptr, nullptr,
                                     relu, precision, st));
  return MIPNERF_B200_OK;
}

size_t mipnerf_b200_wgrad_tc_scratch_bytes(int n, int k) {
  if (n < 1 || k < 1) return 0;
  return sizeof(float) * (size_t)mipnerf::kWgradMaxSlices * n * (k + 1);
}

int mipnerf_b200_wgrad_tc(const float* dy, int n, const float* x1, int k1, const float* x2, int k2, int x2_row_div,
                          int64_t m, float* dw, float* db, int precision, void* scratch, size_t scratch_bytes,
                          void* stream) {
  if (m < 0 || k1 < 1 || k2 < 0 || !mipnerf::wgrad_tc_shape_ok(n))
    return fail(MIPNERF_B200_EUNSUPPORTED, "wgrad_tc: n in {128,256} (got n=%d)", n);
  if (precision != MIPNERF_B200_BF16 && precision != MIPNERF_B200_FP16)
    return fail(MIPNERF_B200_EINVAL, "wgrad_tc: precision must be BF16 or FP16");
  if (!dw || !db || (m > 0 && (!dy || !x1 || (k2 > 0 && !x2)))) return fail(MIPNERF_B200_EINVAL, "NULL tensor");
  const size_t need = mipnerf_b200_wgrad_tc_scratch_bytes(n, k1 + k2);
  if (!scratch || scratch_bytes < need) return fail(MIPNERF_B200_EWORKSPACE, "scratch %zu < %zu bytes", scratch_bytes, need);
  cudaStream_t st = (cudaStream_t)stream;
  int slices = 0;
  CUDA_TRY(mipnerf::launch_wgrad_tc_partials(dy, n, x1, k1, k1, k2 > 0 ? x2 : nullptr, k2, k2, x2_row_div,
                                             static_cast<float*>(scratch), m, mipnerf::kWgradMaxSlices, precision,
                                             &slices, st));
  CUDA_TRY(mipnerf::launch_wgrad_reduce(static_cast<float*>(scratch), slices, n, k1 + k2, dw, db, 0, st));
  return MIPNERF_B200_OK;
}

int mipnerf_b200_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, int64_t n,
                           double lr, double beta1, double beta2, double eps, int64_t step, double grad_scale,
                           void* stream) {
  if (n < 0 || step < 1) return fail(MIPNERF_B200_EINVAL, "bad n / step");
  if (n > 0 && (!param || !grad || !exp_avg || !exp_avg_sq)) return fail(MIPNERF_B200_EINVAL, "NULL tensor");
  const double bc1 = 1.0 - pow(beta1, (double)step), bc2 = 1.0 - pow(beta2, (double)step);
  CUDA_TRY(mipnerf::launch_adam(param, grad, exp_avg, exp_avg_sq, n, (float)beta1, (float)beta2, (float)eps,
                                (float)(lr / bc1), (float)sqrt(bc2), (float)grad_scale, (cudaStream_t)stream));
  return MIPNERF_B200_OK;
}

int mipnerf_b200_adam_step_multi(int count, float* const* params, const float* const* grads, float* const* exp_avg,
                                 float* const* exp_avg_sq, const int64_t* sizes, double lr, double beta1, double beta2,
                                 double eps, int64_t step, double grad_scale, void* stream) {
  if (count < 0 || step < 1) return fail(MIPNERF_B200_EINVAL, "bad count / step");
  if (count > 0 && (!params || !grads || !exp_avg || !exp_avg_sq || !sizes)) return fail(MIPNERF_B200_EINVAL, "NULL array");
  const double bc1 = 1.0 - pow(beta1, (double)step), bc2 = 1.0 - pow(beta2, (double)step);
  for (int base = 0; base < count; base += mipnerf::kAdamMaxTensors) {
    mipnerf::AdamMulti t{};
    t.count = (count - base) < mipnerf::kAdamMaxTensors ? (count - base) : mipnerf::kAdamMaxTensors;
    for (int k = 0; k < t.count; ++k) {
      const int i = base + k;
      if (sizes[i] < 0 || (sizes[i] > 0 && (!params[i] || !grads[i] || !exp_avg[i] || !exp_avg_sq[i])))
        return fail(MIPNERF_B200_EINVAL, "tensor %d: NULL pointer or negative size", i);
      t.p[k] = params[i], t.g[k] = grads[i], t.m[k] = exp_avg[i], t.v[k] = exp_avg_sq[i], t.n[k] = sizes[i];
      t.blocks[k] = (int)((sizes[i] + 255) / 256);
    }
    CUDA_TRY(mipnerf::launch_adam_multi(t, (float)beta1, (float)beta2, (float)eps, (float)(lr / bc1), (float)sqrt(bc2),
                                        (float)grad_scale, (cudaStream_t)stream));
  }
  return MIPNERF_B200_OK;
}

int mipnerf_b200_adam_step_multi_table(int count, float* const* params, const float* const* grads,
                                       float* const* exp_avg, float* const* exp_avg_sq, const int64_t* sizes,
                                       const float* step_size, const float* bc2_sqrt, int64_t table_len,
                                       const int64_t* step, double beta1, double beta2, double eps, double grad_scale,
                                       void* stream) {
  if (count < 0 || table_len < 2) return fail(MIPNERF_B200_EINVAL, "bad count / table_len");
  if (count > 0 && (!params || !grads || !exp_avg || !exp_avg_sq || !sizes || !step_size || !bc2_sqrt || !step))
    return fail(MIPNERF_B200_EINVAL, "NULL array");
  for (int base = 0; base < count; base += mipnerf::kAdamMaxTensors) {
    mipnerf::AdamMulti t{};
    t.count = (count - base) < mipnerf::kAdamMaxTensors ? (count - base) : mipnerf::kAdamMaxTensors;
    for (int k = 0; k < t.count; ++k) {
      const int i = base + k;
      if (sizes[i] < 0 || (sizes[i] > 0 && (!params[i] || !grads[i] || !exp_avg[i] || !exp_avg_sq[i])))
        return fail(MIPNERF_B200_EINVAL, "tensor %d: NULL pointer or negative size", i);
      t.p[k] = params[i], t.g[k] = grads[i], t.m[k] = exp_avg[i], t.v[k] = exp_avg_sq[i], t.n[k] = sizes[i];
      t.blocks[k] = (int)((sizes[i] + 255) / 256);
    }
    CUDA_TRY(mipnerf::launch_adam_multi_table(t, (float)beta1, (float)beta2, (float)eps, step_size, bc2_sqrt, table_len,
                                              step, (float)grad_scale, (cudaStream_t)stream));
  }
  return MIPNERF_B200_OK;
}

int mipnerf_b200_train_step_advance(int64_t* step, uint64_t* rng_state, const float* loss, const float* psnr,
                                    float* ring, int ring_len, void* stream) {
  if (!step || !rng_state) return fail(MIPNERF_B200_EINVAL, "step / rng_state is NULL");
  if (ring_len < 0 || (ring_len > 0 && (!ring || !loss || !psnr))) return fail(MIPNERF_B200_EINVAL, "bad ring");
  CUDA_TRY(mipnerf::launch_train_step_advance(step, rng_state, loss, psnr, ring, ring_len, (cudaStream_t)stream));
  return MIPNERF_B200_OK;
}

int mipnerf_b200_sample_pixels(const float* cam_table, const int64_t* offsets, const int32_t* widths, int num_images,
                               int64_t num_pixels, const uint64_t* rng_state, int64_t ray_base, int64_t count,
                               const float* atlas, int64_t* pixel_ids, float* origins, float* directions,
                               float* viewdirs, float* radii, float* lossmult, float* near_out, float* far_out,
                               float* rgb, void* stream) {
  if (num_images < 1 || num_pixels < 1 || num_pixels > ((int64_t)1 << 32) || count < 0 || ray_base < 0)
    return fail(MIPNERF_B200_EINVAL, "bad num_images / num_pixels (1 .. 2^32) / count / ray_base");
  if (count > 0 && (!cam_table || !offsets || !widths || !atlas || !rng_state || !origins || !directions || !viewdirs ||
                    !radii || !lossmult || !near_out || !far_out))
    return fail(MIPNERF_B200_EINVAL, "NULL tensor");
  CUDA_TRY(mipnerf::launch_sample_pixels(cam_table, offsets, widths, num_images, num_pixels, rng_state, ray_base, count,
                                         atlas, pixel_ids, origins, directions, viewdirs, radii, lossmult, near_out,
                                         far_out, rgb, (cudaStream_t)stream));
  return MIPNERF_B200_OK;
}

int mipnerf_b200_distloss(const float* weights, const float* samples, int64_t num_rays, int num_samples,
                          float* per_ray_loss, void* stream) {
  if (num_rays < 0 || num_samples < 1) return fail(MIPNERF_B200_EINVAL, "bad sizes");
  if (num_rays > 0 && (!weights || !samples || !per_ray_loss)) return fail(MIPNERF_B200_EINVAL, "NULL tensor");
  CUDA_TRY(mipnerf::launch_distloss(weights, samples, per_ray_loss, num_rays, num_samples, (cudaStream_t)stream));
  return MIPNERF_B200_OK;
}

size_t mipnerf_b200_image_metrics_scratch_bytes(int height, int width, int channels) {
  if (height < 1 || width < 1 || channels < 1) return 0;
  return mipnerf::image_metrics_scratch_bytes(height, width, channels);
}

int mipnerf_b200_image_metrics(const float* pred, const float* target, int height, int width, int channels,
                               void* scratch, size_t scratch_bytes, float* out, void* stream) {
  if (height < 1 || width < 1 || channels < 1) return fail(MIPNERF_B200_EINVAL, "bad image shape");
  if (!pred || !target || !out) return fail(MIPNERF_B200_EINVAL, "NULL tensor");
  const size_t need = mipnerf::image_metrics_scratch_bytes(height, width, channels);
  if (!scratch || scratch_bytes < need) return fail(MIPNERF_B200_EWORKSPACE, "scratch %zu < %zu bytes", scratch_bytes, need);
  CUDA_TRY(mipnerf::launch_image_metrics(pred, target, height, width, channels, 11, 1.5f, 1.0f, scratch, out,
                                         (cudaStream_t)stream));
  return MIPNERF_B200_OK;
}

int mipnerf_b200_generate_rays(const float* c2w_host, int height, int width, float focal, float near, float far,
                               int row0, int rows, float* origins, float* directions, float* viewdirs,
                               float* radii, float* near_out, float* far_out, void* stream) {
  if (!c2w_host || height < 2 || width < 1 || !(focal > 0.f) || row0 < 0 || rows < 0 || row0 + rows > height)
    return fail(MIPNERF_B200_EINVAL, "bad frame geometry");
  if (rows > 0 && (!origins || !directions || !viewdirs || !radii || !near_out || !far_out))
    return fail(MIPNERF_B200_EINVAL, "NULL output");
  CUDA_TRY(mipnerf::launch_generate_rays(c2w_host, height, width, focal, near, far, row0, rows, origins, directions,
                                         viewdirs, radii, near_out, far_out, (cudaStream_t)stream));
  return MIPNERF_B200_OK;
}

int mipnerf_b200_rays_from_pixels(const float* cam_table, const int64_t* offsets, const int32_t* widths,
                                  int num_images, const int64_t* pixel_ids, int64_t count, const float* atlas,
                                  float* origins, float* directions, float* viewdirs, float* radii,
                                  float* lossmult, float* near_out, float* far_out, float* rgb, void* stream) {
  if (num_images < 1 || count < 0) return fail(MIPNERF_B200_EINVAL, "bad sizes");
  if (!cam_table || !offsets || !widths) return fail(MIPNERF_B200_EINVAL, "NULL scene table");
  if (count > 0 && (!pixel_ids || !origins || !directions || !viewdirs || !radii || !lossmult || !near_out || !far_out))
    return fail(MIPNERF_B200_EINVAL, "NULL ray tensor");
  if (rgb && !atlas) return fail(MIPNERF_B200_EINVAL, "rgb requested without a pixel atlas");
  CUDA_TRY(mipnerf::launch_rays_from_pixels(cam_table, offsets, widths, num_images, pixel_ids, count, atlas, origins,
                                            directions, viewdirs, radii, lossmult, near_out, far_out, rgb,
                                            (cudaStream_t)stream));
  return MIPNERF_B200_OK;
}

int mipnerf_b200_sample_along_rays(const mipnerf_b200_rays* rays, int num_samples, int randomized,
                                   int disparity, const float* t_rand, float* t_samples, float* means,
                                   float* covs, void* stream) {
  int rc;
  if ((rc = check_rays(rays))) return rc;
  if (num_samples < 1 || !t_samples) return fail(MIPNERF_B200_EINVAL, "bad num_samples / t_samples");
  if (randomized && !t_rand) return fail(MIPNERF_B200_EINVAL, "randomized=1 needs t_rand");
  cudaStream_t st = (cudaStream_t)stream;
  CUDA_TRY(mipnerf::launch_coarse_t(rays->near, rays->far, mipnerf::draws_from_array(randomized ? t_rand : nullptr),
                                    t_samples, rays->num_rays, num_samples, randomized, disparity, st));
  if (means && covs)
    CUDA_TRY(mipnerf::launch_cast_rays(rays->origins, rays->directions, rays->radii, t_samples, means, covs,
                                       rays->num_rays, num_samples, st));
  return MIPNERF_B200_OK;
}

int mipnerf_b200_cast_rays(const mipnerf_b200_rays* rays, const float* t_samples, int num_samples,
                           float* means, float* covs, void* stream) {
  int rc;
  if ((rc = check_rays(rays))) return rc;
  if (num_samples < 1 || !t_samples || !means || !covs) return fail(MIPNERF_B200_EINVAL, "NULL argument");
  CUDA_TRY(mipnerf::launch_cast_rays(rays->origins, rays->directions, rays->radii, t_samples, means, covs,
                                     rays->num_rays, num_samples, (cudaStream_t)stream));
  return MIPNERF_B200_OK;
}

int mipnerf_b200_integrated_pos_enc(const float* means, const float* covs, int64_t num_points, int min_deg,
                                    int max_deg, float* out, void* stream) {
  if (num_points < 0 || (num_points > 0 && (!means || !covs || !out)) || max_deg <= min_deg ||
      min_deg < -60 || max_deg > 60)
    return fail(MIPNERF_B200_EINVAL, "bad argument");
  CUDA_TRY(mipnerf::launch_ipe(means, covs, out, num_points, min_deg, max_deg, (cudaStream_t)stream));
  return MIPNERF_B200_OK;
}

int mipnerf_b200_pos_enc(const float* x, int64_t num_points, int min_deg, int max_deg, int append_identity,
                         float* out, void* stream) {
  if (num_points < 0 || (num_points > 0 && (!x || !out)) || max_deg < min_deg || min_deg < -60 || max_deg > 60)
    return fail(MIPNERF_B200_EINVAL, "bad argument");
  CUDA_TRY(mipnerf::launch_pos_enc(x, out, num_points, min_deg, max_deg, append_identity, (cudaStream_t)stream));
  return MIPNERF_B200_OK;
}

int mipnerf_b200_mlp_forward(const mipnerf_b200_config* cfg, const mipnerf_b200_weights* w, const float* x,
                             const float* view_enc, int64_t num_rays, int samples_per_ray, int precision,
                             float* raw_rgb, float* raw_density, void* workspace, size_t workspace_bytes,
                             void* stream) {
  Dims d;
  int rc;
  mipnerf_b200_config c2;
  if (!cfg) return fail(MIPNERF_B200_EINVAL, "config is NULL");
  c2 = *cfg;
  c2.num_samples = 32;  // the MLP itself does not care; validate the rest
  if ((rc = check_config(&c2, &d))) return rc;
  if ((rc = check_weights(cfg, d, w))) return rc;
  if (num_rays < 0 || samples_per_ray < 1) return fail(MIPNERF_B200_EINVAL, "bad sizes");
  if (num_rays == 0) return MIPNERF_B200_OK;
  if (!x || !raw_rgb || !raw_density || (cfg->use_viewdirs && !view_enc))
    return fail(MIPNERF_B200_EINVAL, "NULL tensor");
  cudaStream_t st = (cudaStream_t)stream;
  if (precision != MIPNERF_B200_FP32) {
    if (!mipnerf::tc_mlp_supported(cfg, samples_per_ray, precision))
      return fail(MIPNERF_B200_EUNSUPPORTED, "tensor-core MLP: default 8x256 model, 128 samples/ray only");
    if (!w->packed || w->packed_precision != precision)
      return fail(MIPNERF_B200_EINVAL, "weights->packed missing or packed for another precision");
    if (!workspace || workspace_bytes < mipnerf::tc_mlp_workspace_bytes(num_rays))
      return fail(MIPNERF_B200_EWORKSPACE, "workspace %zu < %zu bytes", workspace_bytes,
                  mipnerf::tc_mlp_workspace_bytes(num_rays));
    cudaError_t e = mipnerf::tc_mlp_forward(cfg, w, x, view_enc, num_rays, precision, raw_rgb, raw_density, workspace,
                                            st);
    if (e != cudaSuccess) return fail(MIPNERF_B200_ECUDA, "tc_mlp_forward: %s", cudaGetErrorString(e));
    return MIPNERF_B200_OK;
  }
  c2.num_samples = samples_per_ray;
  const int64_t max_rows = kChunkRaysFp32 * 128;
  int64_t per = max_rows / samples_per_ray;
  if (per < 1) per = 1;
  const size_t need = mipnerf_b200_mlp_workspace_bytes(cfg, num_rays, samples_per_ray, precision);
  if (!workspace || workspace_bytes < need)
    return fail(MIPNERF_B200_EWORKSPACE, "workspace %zu < %zu bytes", workspace_bytes, need);
  for (int64_t off = 0; off < num_rays; off += per) {
    const int64_t cnt = (num_rays - off) < per ? (num_rays - off) : per;
    const Fp32Scratch s = carve_fp32(&c2, d, cnt, workspace, /*mlp_only=*/true);
    const int64_t row = off * samples_per_ray;
    if ((rc = mlp_forward_fp32(cfg, d, w, x + row * d.xyz_dim, view_enc ? view_enc + off * d.view_dim : nullptr,
                               cnt, samples_per_ray, s, raw_rgb + row * 3, raw_density + row, st)))
      return rc;
  }
  return MIPNERF_B200_OK;
}

size_t mipnerf_b200_mlp_workspace_bytes(const mipnerf_b200_config* cfg, int64_t num_rays, int samples_per_ray,
                                        int precision) {
  Dims d;
  if (!cfg || num_rays < 0 || samples_per_ray < 1) return 0;
  mipnerf_b200_config c2 = *cfg;
  c2.num_samples = 32;
  if (check_config(&c2, &d) != MIPNERF_B200_OK) return 0;
  if (precision != MIPNERF_B200_FP32) return mipnerf::tc_mlp_workspace_bytes(num_rays);
  c2.num_samples = samples_per_ray;
  int64_t per = (kChunkRaysFp32 * 128) / samples_per_ray;
  if (per < 1) per = 1;
  if (per > num_rays) per = num_rays > 0 ? num_rays : 1;
  return carve_fp32(&c2, d, per, nullptr, true).bytes;
}

int mipnerf_b200_volumetric_rendering(const float* rgb, const float* density, const float* t_samples,
                                      const float* dirs, int64_t num_rays, int num_samples, int white_bkgd,
                                      float* comp_rgb, float* distance, float* acc, float* weights,
                                      void* stream) {
  if (num_rays < 0 || num_samples < 1) return fail(MIPNERF_B200_EINVAL, "bad sizes");
  if (num_rays == 0) return MIPNERF_B200_OK;
  if (!rgb || !density || !t_samples || !dirs || !comp_rgb || !distance || !acc)
    return fail(MIPNERF_B200_EINVAL, "NULL tensor");
  cudaError_t e = mipnerf::launch_composite(rgb, density, t_samples, dirs, comp_rgb, distance, acc, weights,
                                            num_rays, num_samples, white_bkgd, 0, 0.f, 1.f, 0.f,
                                            (cudaStream_t)stream);
  if (e == cudaErrorInvalidValue)
    return fail(MIPNERF_B200_EUNSUPPORTED, "num_samples=%d: need a multiple of 32 in {32..256}", num_samples);
  CUDA_TRY(e);
  return MIPNERF_B200_OK;
}

int mipnerf_b200_sorted_piecewise_constant_pdf(const float* bins, const float* weights, int64_t num_rays,
                                               int num_bins, int num_samples, int randomized,
                                               const float* u_jitter, float* samples, int64_t* inds,
                                               void* stream) {
  if (num_rays < 0 || num_bins < 1 || num_samples < 2) return fail(MIPNERF_B200_EINVAL, "bad sizes");
  if (num_bins % 32 != 0 || num_bins > 1024)
    return fail(MIPNERF_B200_EUNSUPPORTED, "num_bins=%d: need a multiple of 32, <= 1024", num_bins);
  if (num_rays == 0) return MIPNERF_B200_OK;
  if (!bins || !weights || !samples || (randomized && !u_jitter)) return fail(MIPNERF_B200_EINVAL, "NULL tensor");
  CUDA_TRY(mipnerf::launch_resample(bins, weights, mipnerf::draws_from_array(randomized ? u_jitter : nullptr), samples,
                                    inds, num_rays, num_bins, num_samples, randomized, 0, 0.f, (cudaStream_t)stream));
  return MIPNERF_B200_OK;
}

int mipnerf_b200_resample_along_rays(const mipnerf_b200_rays* rays, const float* t_samples, const float* weights,
                                     int num_samples, int randomized, const float* u_jitter,
                                     float resample_padding, float* new_t_samples, float* means, float* covs,
                                     int64_t* inds, void* stream) {
  int rc;
  if ((rc = check_rays(rays))) return rc;
  if (num_samples < 32 || num_samples % 32 != 0 || num_samples > 1024)
    return fail(MIPNERF_B200_EUNSUPPORTED, "num_samples=%d: need a multiple of 32, <= 1024", num_samples);
  if (rays->num_rays == 0) return MIPNERF_B200_OK;
  if (!t_samples || !weights || !new_t_samples || (randomized && !u_jitter))
    return fail(MIPNERF_B200_EINVAL, "NULL tensor");
  cudaStream_t st = (cudaStream_t)stream;
  CUDA_TRY(mipnerf::launch_resample(t_samples, weights, mipnerf::draws_from_array(randomized ? u_jitter : nullptr),
                                    new_t_samples, inds, rays->num_rays, num_samples, num_samples + 1, randomized, 1,
                                    resample_padding, st));
  if (means && covs)
    CUDA_TRY(mipnerf::launch_cast_rays(rays->origins, rays->directions, rays->radii, new_t_samples, means,
                                       covs, rays->num_rays, num_samples, st));
  return MIPNERF_B200_OK;
}

}  // extern "C"
