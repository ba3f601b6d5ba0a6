// draws.h — where the uniforms of randomized=True come from (plain struct, usable from host code and kernels).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace mipnerf {

struct Draws {
  const float* ptr;    // explicit [rays, ncols] array (row 0 = this launch's ray 0), or nullptr
  uint64_t seed, offset;
  int64_t ray_base;    // global index of this launch's ray 0
  int stream;          // 0: t_rand (models/mip.py:159), 1 + level: u_jitter (:201-202), 32 + level: density normals
  int philox;          // draw in-kernel when ptr == nullptr
  float scale;         // u_jitter: 1/num_samples - eps (uniform_(to=...)); t_rand: 1; density normals: density_noise
};
constexpr int kDensityNoiseStream = 32;  // + level (models/mip_nerf.py:232-233)
constexpr int kPixelStream = 64;         // training batch: the pixel ids of mipnerf_b200_sample_pixels
__host__ __device__ __forceinline__ Draws draws_from_array(const float* ptr) {
  Draws d{};
  d.ptr = ptr;
  d.scale = 1.f;
  return d;
}
__host__ __device__ __forceinline__ bool draws_active(const Draws& d) { return d.ptr != nullptr || d.philox != 0; }

// in-kernel Philox draws of `stream` (0: t_rand, 1: u_jitter), scaled by `scale`
__host__ __device__ __forceinline__ Draws draws_philox(uint64_t seed, uint64_t offset, int64_t ray_base, int stream,
                                                       float scale) {
  Draws d{};
  d.seed = seed, d.offset = offset, d.ray_base = ray_base, d.stream = stream, d.philox = 1, d.scale = scale;
  return d;
}

// `d` with (seed, offset) read from the device array `state` when the kernel runs (a captured training step replays
// the same kernel parameters and still draws fresh numbers), if d draws in-kernel and state is set; kDevice = false
// compiles to `d` itself.  The pointer travels next to the Draws (LevelParams::rng_state), not inside them: a larger
// Draws would move the parameter offsets of every inference kernel and with them their code.
template <bool kDevice>
__device__ __forceinline__ Draws draws_at_state(const Draws& d, const uint64_t* state) {
  if constexpr (kDevice) {
    if (state && d.philox && !d.ptr) {
      Draws r = d;
      r.seed = state[0], r.offset = state[1];
      return r;
    }
  }
  return d;
}

}  // namespace mipnerf
