// mlp_tc.h — internal interface of the tcgen05 (tensor-core) path, implemented in mlp_tc.cu.
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/mipnerf_b200.h"
#include "draws.h"

namespace mipnerf {

// true iff (cfg, precision) is the shape the fused tensor-core kernels are specialised for.
bool tc_supported(const mipnerf_b200_config* cfg, int precision);
bool tc_default_degrees(const mipnerf_b200_config* cfg);  // max_deg_point == 16 && deg_view == 4 (no weight padding)
bool tc_mlp_supported(const mipnerf_b200_config* cfg, int samples_per_ray, int precision);
size_t tc_packed_bytes(const mipnerf_b200_config* cfg, int precision);
size_t tc_workspace_bytes(const mipnerf_b200_config* cfg, int64_t num_rays, int precision);
cudaError_t tc_pack_weights(const mipnerf_b200_config* cfg, const mipnerf_b200_weights* w, int precision,
                            void* packed_out, cudaStream_t st, bool with_v3 = true);
// Training forward: where the level kernels leave what the backward pass needs (per level l < 2; at most
// kTcTrainChunk rays per call).  Activations are 16-bit "tile images": per 128-row tile (= ray) and 64-column slab a
// [128 x 128 B] block in the 128-byte-swizzle layout the tensor core reads (sw128_offset), slabs of a tile contiguous.
struct TcTrainDump {
  uint8_t* act[2];        // [9][rays][64 KB]: h_0..h_7 (post-ReLU), bottleneck
  uint8_t* v[2];          // [rays][32 KB]: view-layer output (post-ReLU)
  float* raw_rgb[2];      // [rays,128,3]
  float* raw_density[2];  // [rays,128]
  const uint64_t* rng_state;  // nullable: device (seed, offset) of the in-kernel draws, read when the kernel runs
};
cudaError_t tc_forward(const mipnerf_b200_config* cfg, const mipnerf_b200_weights* w,
                       const mipnerf_b200_rays* rays, int randomized, const float* t_rand,
                       const float* u_jitter, const mipnerf_b200_rng* rng, int white_bkgd, int precision,
                       mipnerf_b200_level_out* outs, void* workspace, size_t workspace_bytes, cudaStream_t st,
                       const TcTrainDump* dump = nullptr, int64_t ray_base = 0);
// the uniforms of one launch (see mlp_tc.cu)
Draws level_draws(int randomized, const float* array, const mipnerf_b200_rng* rng, int64_t off, int stream, int ncols);
// the density-noise normals of one launch of `level` (inactive unless randomized and cfg->density_noise > 0)
Draws density_noise_draws(const mipnerf_b200_config* cfg, int randomized, const float* normal,
                          const mipnerf_b200_rng* rng, int64_t off, int level, int n);
cudaError_t tc_mlp_forward(const mipnerf_b200_config* cfg, const mipnerf_b200_weights* w, const float* x,
                           const float* view_enc, int64_t num_rays, int precision, float* raw_rgb,
                           float* raw_density, void* workspace, cudaStream_t st);
size_t tc_mlp_workspace_bytes(int64_t num_rays);

}  // namespace mipnerf
