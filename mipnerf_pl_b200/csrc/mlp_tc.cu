// mlp_tc.cu — the tensor-core path: one fused kernel per sampling level that does, per ray,
//   fenceposts (coarse, or resampled from the previous level)      (models/mip.py:127-165, 168-280)
//   -> conical-frustum Gaussians -> IPE features                   (models/mip.py:81-103, 322-350)
//   -> 8x256 trunk + density / bottleneck / view / colour heads    (models/mip_nerf.py:75-111)
//   -> activations + front-to-back alpha compositing               (models/mip_nerf.py:236-238, mip.py:366-401)
// without any intermediate tensor touching HBM.  Per level the kernel reads 52 B of ray data (+ the previous
// level's fenceposts / weights for the resampler) and writes t_samples/comp_rgb/distance/acc/weights; the
// weights stream from L2.  A forward is two launches of this kernel and nothing else.
//
// Mapping (sm_100a, 1 persistent CTA per SM, 384 threads = 12 warps):
//   * tile = one ray = 128 samples = UMMA M.  Each CTA keeps TWO rays in flight ("slots") so that
//     while slot 0's epilogue warps turn an accumulator into the next layer's A operand, the tensor
//     core runs slot 1's layer.  TMEM: 2 x 256 fp32 columns (the whole 512).
//   * warp 0    : weight producer — cp.async.bulk of pre-swizzled [128 x 32] (SW64, 8 KB) operand stages
//   * warp 1    : MMA issuer (one elected lane around the whole issue loop) / relay in the peer CTA
//   * warps 2-5 : slot 0 workers, warps 6-9: slot 1 workers — thread = sample row = TMEM lane:
//                 epilogues (tcgen05.ld, packed FADD2 bias, cvt.relu 16-bit pack -> st.shared SW128 A operand),
//                 density/colour heads on CUDA cores (FFMA2), 128-thread compositing scan.
//   * warps 10-11: IPE warps (one per slot) — for the slot's NEXT ray: the ray prologue (coarse fenceposts or the
//                 bit-exact inverse-CDF resampler, per-ray view-layer bias) while the current ray's layers 0..5
//                 still read the feature tile, then Gaussians + 96 features into that tile once it is released.
//   * layer-5 skip connection = extra K slabs read from the feature tile (no concat), the
//     per-ray view-direction term of the view layer is a per-ray bias vector.
// CTA-pair mode (kPair, default): the grid is launched as 2-CTA clusters and the MMA is
// tcgen05.mma.cta_group::2 (M=256: rays of both CTAs, N=256): each CTA stages only ITS half of every
// weight tile (N rows rank*128..), so L2->SMEM weight traffic and SMEM operand reads per SM halve.
// The leader CTA's warp 1 issues for the pair; the other CTA's warp 1 relays "my half has landed";
// epilogue warps of both CTAs arrive on the leader's a_ready barrier (remote mbarrier arrive);
// tcgen05.commit multicasts stage-free / accumulator-full to both CTAs.
// A operand: 4 SW128 slabs (64 KB) per slot, overwritten in place layer after layer; features:
// SW128 slab (K 0..63) + SW64 slab (K 64..95) per slot; weight ring: 6 x 8 KB.
// Other modes of the same kernel: MLP-only (features from the caller, raw heads out: mipnerf_b200_mlp_forward),
// separate prologue (MIPNERF_B200_TC_PROLOGUE=separate); mlp_level_kernel_v2 is the "shared weight stream" variant.
#include "mlp_tc.h"

#include <cstdlib>
#include <mutex>

#include "kernels.h"
#include "profile.h"
#include "ray_math.cuh"
#include "ray_resample.cuh"
#include "tc_common.cuh"

namespace mipnerf {
namespace {

using namespace tc;

constexpr int kN = 128;         // samples per ray (UMMA M)
constexpr int kWidth = 256;     // trunk width
constexpr int kCond = 128;      // view layer width
constexpr int kFeat = 96;       // IPE width
constexpr int kViewDim = 27;
constexpr int kNumLayers = 10;  // 8 trunk + extra_layer + view layer
#ifndef MIPNERF_TC_DEFAULT_VARIANT
#define MIPNERF_TC_DEFAULT_VARIANT 1
#endif
constexpr int kThreads = 384;   // 12 warps: producer, MMA, 2x4 epilogue workers, 2 IPE warps
#ifndef MIPNERF_TC_STAGES
#define MIPNERF_TC_STAGES 6
#endif
constexpr int kStages = MIPNERF_TC_STAGES;
constexpr uint32_t kStageBytes = 16384;  // A-operand slab: [128 x 64] 16-bit, SW128
constexpr uint32_t kTailBytes = 8192;    // feature tail slab: [128 x 32] 16-bit, SW64
constexpr uint32_t kWStage = 8192;       // weight stage: [128 x 32] 16-bit, SW64 (K = 32 = two MMA steps)
constexpr uint32_t kABytes = 65536;      // 4 slabs
constexpr uint32_t kFBytes = kStageBytes + kTailBytes;  // feature tile: SW128 slab (K 0..63) + SW64 slab (K 64..95)
constexpr uint32_t kSmemA = 0;
constexpr uint32_t kSmemF = kSmemA + 2 * kABytes;
constexpr uint32_t kSmemW = kSmemF + 2 * kFBytes;
constexpr uint32_t kSmemMisc = kSmemW + kStages * kWStage;
constexpr uint32_t kMiscBytes = 256 + 16 + 2 * 128 * 4 + 8 * 4 + 2 * 4 * 8 * 4;
constexpr uint32_t kSmemTotal = kSmemMisc + kMiscBytes + 1024 + 64;  // + slack for 1024-B alignment (when the base
                                                                       // is aligned, the slack holds the resampler scratch)
static_assert(kSmemTotal <= 232448, "exceeds 227 KB of shared memory per CTA");

// Biases and the two CUDA-core heads, broadcast-read by every thread: constant bank.
struct SmallParams {
  float bias[9][kWidth];      // layers.0..7, extra_layer
  float w_density[kWidth];    // density_layer.weight
  float w_color[3][kCond];    // color_layer.weight
  float b_density;
  float b_color[3];
};
__constant__ SmallParams c_small;

// Packed weight image: per layer, per N-half (rows h*128..), K-slabs of 32 as [128 x 64 B] SW64 stages.
// number of 32-wide K slabs of layer l (96, 256, .., 352 = [h | x], .., view layer uses the first 256)
__host__ __device__ constexpr int num_k32(int l) { return l == 0 ? 3 : (l == 5 ? 11 : 8); }
__host__ __device__ constexpr int num_halves(int l) { return l == 9 ? 1 : 2; }
__host__ __device__ constexpr uint32_t layer_bytes(int l) { return (uint32_t)num_halves(l) * num_k32(l) * kWStage; }
__host__ __device__ constexpr uint32_t layer_offset(int l) {
  uint32_t o = 0;
  for (int i = 0; i < l; ++i) o += layer_bytes(i);
  return o;
}
constexpr uint32_t kImageStageBytes = layer_offset(kNumLayers);
// pair mode splits the 128-wide view layer into two 64-row halves: 2 x 8 stages of [64 x 32] (4 KB)
constexpr uint32_t kViewPairOffset = kImageStageBytes;
constexpr uint32_t kViewPairStage = 4096;
constexpr size_t kSmallOffset = ((size_t)kViewPairOffset + 2 * 8 * kViewPairStage + 255) / 256 * 256;
// view-direction part of the view layer, transposed for coalesced per-ray reads by the IPE warps:
// fp32 [27][128] weights W_view[n, 256 + k] as [k][n], then the 128 biases
constexpr size_t kViewDirOffset = kSmallOffset + ((sizeof(SmallParams) + 255) / 256 * 256);
constexpr size_t kViewDirBytes = (size_t)(kViewDim + 1) * kCond * sizeof(float);
constexpr size_t kImageBytes = kViewDirOffset + ((kViewDirBytes + 255) / 256 * 256);
// Split-operand ("x3") modes: a second stage image with the LOW halves of the weights (w - fl16(w), rounded to the
// same 16-bit format), same internal layout as the stage part of the first image, appended after it.
constexpr size_t kLoOffset = kImageBytes;
constexpr size_t kLoBytes = ((size_t)kViewPairOffset + 2 * 8 * kViewPairStage + 255) / 256 * 256;
// third region: the "v3" kernel's weight blocks (mlp_tc_v3.cuh), [32 rows x 64 K] per CTA in issue order
constexpr size_t kV3Offset = kLoOffset + kLoBytes;

#ifdef MIPNERF_TC_TRACE
// debug build only: (clock64, event) pairs of CTA 0.  Each traced thread (one per role) owns a
// private region with a register cursor, so an event costs one clock read + one fire-and-forget store.
__device__ unsigned long long* g_trace = nullptr;
constexpr int kTraceRegion = 15000;
struct Tracer {
  unsigned long long* base = nullptr;
  int n = 0;
  __device__ void init(int region) {
    base = (blockIdx.x == 0 && g_trace) ? g_trace + 8 + 2ull * region * kTraceRegion : nullptr;
  }
  __device__ __forceinline__ void ev(uint32_t code) {
    if (base && n < kTraceRegion) {
      base[2 * n] = clock64();
      base[2 * n + 1] = code;
      ++n;
    }
  }
  __device__ void finish(int region) {
    if (base) g_trace[region] = n;
  }
};
#define TRACER_DECL(region) Tracer tracer; tracer.init(region)
#define TRACE(code) tracer.ev(code)
#define TRACER_DONE(region) tracer.finish(region)
// cumulative clock64 counters of CTA 0 (v4 paths): g_trace[16 + base + i], read by tools/v4_counters.py
#define V4_DECL() long long v4c[8] = {0, 0, 0, 0, 0, 0, 0, 0}
#define V4_CLK() clock64()
#define V4_ADD(i, t0) v4c[i] += clock64() - (t0)
#define V4_FLUSH(base)                                                                      \
  if (blockIdx.x == 0 && g_trace) {                                                         \
    for (int i_ = 0; i_ < 8; ++i_) g_trace[16 + (base) + i_] = (unsigned long long)v4c[i_]; \
  }
#else
#define V4_DECL()
#define V4_CLK() 0
#define V4_ADD(i, t0) ((void)(t0))
#define V4_FLUSH(base)
#define TRACER_DECL(region) ((void)0)
#define TRACE(code) ((void)0)
#define TRACER_DONE(region) ((void)0)
#endif
// event codes: role<<24 | kind<<16 | g<<8 | slot/stage
#define EV(role, kind, g, x) (((uint32_t)(role) << 24) | ((uint32_t)(kind) << 16) | ((uint32_t)(g) << 8) | (uint32_t)(x))

struct LevelParams {
  const uint8_t* wimage;
  const float* origins;
  const float* directions;
  const float* radii;
  float* t;                // [B,129] fenceposts of this level (read; written first when t_mode != 0)
  float* view_bias;        // [B,128]  b_view + W_view[:,256:] . pos_enc(viewdir) (written first when vb_mode != 0)
  // Fused ray prologue (v1 kernels): the IPE warps produce the fenceposts / view bias of the slot's next ray
  // themselves instead of reading what a separate launch left in HBM.
  int t_mode;              // 0: read p.t; 1: coarse fenceposts from near/far (models/mip.py:143-160);
                           // 2: resample t_prev / w_prev (models/mip.py:232-280)
  int vb_mode;             // 0: read p.view_bias; 1: compute it from viewdirs and the fp32 view-layer weights
  const float* near;       // t_mode 1
  const float* far;
  Draws t_rand;            // t_mode 1, randomized: the [B,129] stratified uniforms (array or in-kernel Philox)
  int disparity;
  const float* t_prev;     // t_mode 2: previous level's fenceposts [B,129] and weights [B,128]
  const float* w_prev;
  Draws u_jitter;          // t_mode 2, randomized: the [B,129] inverse-CDF jitter (array or in-kernel Philox)
  int64_t* inds;           // t_mode 2: optional searchsorted indices [B,129]
  int randomized;
  float resample_padding;
  const float* viewdirs;   // vb_mode 1: [B,3]; the weights come from the packed image (kViewDirOffset)
  const float* feat_in;    // MLP-only mode (mipnerf_b200_mlp_forward): [B,128,96] features supplied by the caller
  float* raw_rgb_out;      // MLP-only mode: [B,128,3] / [B,128] raw heads instead of compositing
  float* raw_density_out;
  uint8_t* feat_scratch;   // v2 kernel: per-CTA pre-swizzled feature slabs in global memory (L2 resident)
  // Training forward (v1 kernels): every activation the backward pass needs leaves the SM exactly as the tensor core
  // saw it — the 16-bit SW128 activation tile of each trunk layer / the bottleneck is copied out by ONE bulk store
  // (64 KB, shared -> global) after its epilogue; the view layer's output and the raw heads go out from registers.
  uint8_t* act_dump;       // [9][dump_tiles][64 KB]: h_0..h_7 (post-ReLU), bottleneck; tile = ray
  uint8_t* v_dump;         // [dump_tiles][32 KB]: view-layer output (post-ReLU), two SW128 slabs
  float* raw_rgb_keep;     // [B,128,3] / [B,128]: raw heads (before the activations) for render_backward
  float* raw_density_keep;
  int64_t dump_tiles;
  float* comp_rgb;
  float* distance;
  float* acc;
  float* weights;  // [B,128]
  int64_t num_rays;
  int rounds;
  int white_bkgd;
  int disable_integration;
  float density_bias, rgb_scale, rgb_padding;
  Draws dnoise;  // density noise of randomized mode (models/mip_nerf.py:232-233): normals [B,128] or in-kernel; scale = std
  const uint64_t* rng_state;  // training forward, nullable: device (seed, offset) of the in-kernel draws (last member:
                              // the inference kernels' parameter offsets stay where they were)
};

// raw density of (ray, row) with the density noise added; kept out of line so that the (default) noise-free
// instantiations of the level kernel carry none of the generator's registers or code
__device__ __noinline__ float noisy_raw_density(float raw, const Draws d, int64_t ray, int row) {
  return add_density_noise(raw, d, ray, row, kN);
}

__device__ __forceinline__ void named_bar_sync(int id, int count) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(count) : "memory");
}

template <int kFmt>
__device__ __forceinline__ void store8(uint8_t* dst, const float (&x)[8]) {
  *reinterpret_cast<uint4*>(dst) = make_uint4(pack2<kFmt>(x[0], x[1]), pack2<kFmt>(x[2], x[3]),
                                              pack2<kFmt>(x[4], x[5]), pack2<kFmt>(x[6], x[7]));
}

template <int kFmt>
__device__ __forceinline__ float2 unpack2(uint32_t v) {
  if (kFmt == 1) return __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&v));
  return __half22float2(*reinterpret_cast<__half2*>(&v));
}
// x = hi + lo with hi = fl16(x), lo = fl16(x - hi): the two 16-bit operands of the split ("x3") modes
template <int kFmt>
__device__ __forceinline__ void store8_split(uint8_t* dst_hi, uint8_t* dst_lo, const float (&x)[8]) {
  uint32_t h[4], l[4];
#pragma unroll
  for (int e = 0; e < 4; ++e) {
    h[e] = pack2<kFmt>(x[2 * e], x[2 * e + 1]);
    const float2 f = unpack2<kFmt>(h[e]);
    l[e] = pack2<kFmt>(x[2 * e] - f.x, x[2 * e + 1] - f.y);
  }
  *reinterpret_cast<uint4*>(dst_hi) = make_uint4(h[0], h[1], h[2], h[3]);
  *reinterpret_cast<uint4*>(dst_lo) = make_uint4(l[0], l[1], l[2], l[3]);
}

// Byte offset of the 16-byte chunk holding columns [col, col + 8) of `row` in a slot's activation tile.
//   kA32 == false: four 64-column SW128 slabs ([128 x 128 B] each) — the layout the training dump / the backward
//                  pass use (tile images), and the v2 kernel;
//   kA32 == true:  sixteen K = 16 blocks ([128 x 32 B] each, 32-byte swizzle): the block one MMA reads is DENSE in
//                  shared memory (32 lines of 128 B instead of 32 B out of each of 128 lines), which takes the A
//                  operand's shared-memory port time per MMA from 128 to 32 cycles.
template <bool kA32>
__device__ __forceinline__ uint32_t a_chunk_offset(int row, int col) {
  if (kA32) return (uint32_t)(col >> 4) * 4096u + sw32_offset(row, col & 15);
  return (uint32_t)(col >> 6) * kStageBytes + sw128_offset(row, col & 63);
}

// Epilogue of trunk layer / bottleneck L (compile-time so that every bias is an immediate
// constant-bank operand): TMEM accumulator row -> +bias -> ReLU (L < 8) -> 16-bit -> A operand
// slabs, software-pipelined over 32-column TMEM loads.  L == 7 also accumulates the density head.
template <int kFmt, int L, bool kX3, bool kA32 = false>
__device__ __forceinline__ void epilogue_trunk(uint32_t t_acc, uint8_t* myA, int row, float& dens) {
  float dpart[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};  // independent chains for the density head
  uint32_t v[2][32];
  tmem_ld32(t_acc, v[0]);
#pragma unroll
  for (int k = 0; k < 8; ++k) {
    tmem_ld_wait();  // chunk k has landed
    if (k < 7) tmem_ld32(t_acc + 32 * (k + 1), v[(k + 1) & 1]);  // next chunk in flight while we work
    const int c0 = 32 * k;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      uint32_t w[4], wl[4];
#pragma unroll
      for (int e = 0; e < 4; ++e) {
        const int c = c0 + j * 8 + 2 * e;
        float a = __uint_as_float(v[k & 1][j * 8 + 2 * e]), b = __uint_as_float(v[k & 1][j * 8 + 2 * e + 1]);
        fadd2(a, b, c_small.bias[L][c], c_small.bias[L][c + 1]);  // one FADD2 for the pair
        if (L == 7)  // density_layer on the fp32 (un-rounded) h7        (models/mip_nerf.py:98)
          ffma2(dpart[2 * e], dpart[2 * e + 1], fmaxf(a, 0.f), fmaxf(b, 0.f), c_small.w_density[c],
                c_small.w_density[c + 1]);
        if (kX3) {  // hi = fl16(x), lo = fl16(x - hi): 22 (fp16) / 16 (bf16) significant bits reach the next layer
          if (L < 8) a = fmaxf(a, 0.f), b = fmaxf(b, 0.f);
          w[e] = pack2<kFmt>(a, b);
          const float2 h = unpack2<kFmt>(w[e]);
          wl[e] = pack2<kFmt>(a - h.x, b - h.y);
        } else {
          w[e] = L < 8 ? pack2_relu<kFmt>(a, b) : pack2<kFmt>(a, b);
        }
      }
      const uint32_t off = a_chunk_offset<kA32>(row, c0 + j * 8);
      *reinterpret_cast<uint4*>(myA + off) = make_uint4(w[0], w[1], w[2], w[3]);
      if (kX3) *reinterpret_cast<uint4*>(myA + kABytes + off) = make_uint4(wl[0], wl[1], wl[2], wl[3]);
    }
  }
  if (L == 7)
    dens = ((dpart[0] + dpart[1]) + (dpart[2] + dpart[3])) + ((dpart[4] + dpart[5]) + (dpart[6] + dpart[7]));
}

// "v4" (kTS): activations live in TENSOR memory and the MMAs take them from there (TS form: 128.6 cycles per
// M128 x N256 x K16 MMA against 171 for the SS form, tools/umma_rate.py).  A slot owns 256 TMEM columns — 128 for its
// fp32 accumulator, 128 for its 16-bit activation row (two elements per column) — so a 256-wide layer runs as two
// N = 128 halves through the same accumulator.  Epilogue of half kHalf of trunk layer / bottleneck L:
//   kHalf == 0: accumulator -> +bias -> ReLU -> 64 packed words kept in REGISTERS (the activation buffer is still the
//               A operand of the other half's MMAs); `drained()` runs as soon as the accumulator has been read, so the
//               second half's MMAs may overwrite it while the arithmetic is still going on;
//   kHalf == 1: words 64..127 go to the activation buffer as they are produced (every MMA that read it has
//               completed: that is what this half's acc_full says), then the 64 held words.
template <int kFmt, int L, int kHalf, class Drained>
__device__ __forceinline__ void epilogue_half_ts(uint32_t t_acc, uint32_t t_a, uint32_t (&held)[64], float& dens,
                                                 Drained drained) {
  float dpart[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  // half 0: all 128 columns are read before any arithmetic (nothing is held yet, the registers are there), so that the
  // accumulator is handed back to the tensor core at once; half 1: two-chunk pipeline next to the 64 held words
  constexpr int kBuf = kHalf == 0 ? 4 : 2;
  uint32_t v[kBuf][32];
  tmem_ld32(t_acc, v[0]);
  if (kHalf == 0) {
    tmem_ld32(t_acc + 32, v[1 % kBuf]);
    tmem_ld32(t_acc + 64, v[2 % kBuf]);
    tmem_ld32(t_acc + 96, v[3 % kBuf]);
    tmem_ld_wait();
    drained();
  }
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (kHalf == 1) {
      tmem_ld_wait();
      if (k < 3) tmem_ld32(t_acc + 32 * (k + 1), v[(k + 1) % kBuf]);
    }
    uint32_t w[16];
#pragma unroll
    for (int j = 0; j < 16; ++j) {
      const int c = 128 * kHalf + 32 * k + 2 * j;
      float a = __uint_as_float(v[k % kBuf][2 * j]), b = __uint_as_float(v[k % kBuf][2 * j + 1]);
      fadd2(a, b, c_small.bias[L][c], c_small.bias[L][c + 1]);
      if (L == 7)  // density_layer on the fp32 (un-rounded) h7        (models/mip_nerf.py:98)
        ffma2(dpart[(2 * j) & 7], dpart[(2 * j + 1) & 7], fmaxf(a, 0.f), fmaxf(b, 0.f), c_small.w_density[c],
              c_small.w_density[c + 1]);
      w[j] = L < 8 ? pack2_relu<kFmt>(a, b) : pack2<kFmt>(a, b);
    }
    if (kHalf == 0) {
#pragma unroll
      for (int j = 0; j < 16; ++j) held[16 * k + j] = w[j];
    } else {
      tmem_st16(t_a + 64 + 16 * k, w);
    }
  }
  if (kHalf == 1) {
#pragma unroll
    for (int k = 0; k < 4; ++k) tmem_st16(t_a + 16 * k, *reinterpret_cast<const uint32_t(*)[16]>(&held[16 * k]));
  }
  if (L == 7) {
    const float d = ((dpart[0] + dpart[1]) + (dpart[2] + dpart[3])) + ((dpart[4] + dpart[5]) + (dpart[6] + dpart[7]));
    dens = kHalf == 0 ? d : dens + d;
  }
}

// Rolled form of the same epilogue with the layer index at RUN time: one copy of the code for all nine layers, a loop
// over 64-column steps (two pipelined 32-column TMEM loads each).  The ncu source page of the unrolled, per-layer
// instantiated version shows its arithmetic stalled on instruction fetch (stall_no_inst: ~45 % of the epilogue samples
// of the bf16 kernel, ~80 % in the split modes, whose nine instantiations are 190 KB of straight-line code that every
// worker warp streams through once per ray): the rolled body is ~2-5 KB and stays in the instruction caches.
#ifndef MIPNERF_TC_ROLLED_EPILOGUE
#define MIPNERF_TC_ROLLED_EPILOGUE 0
#endif
template <int kFmt, bool kX3, bool kRelu, bool kDens, bool kA32>
__device__ __forceinline__ void epilogue_chunk(const uint32_t (&v)[32], int layer, int c0, uint8_t* myA, uint32_t rowoff,
                                               uint32_t rx, float (&dpart)[8], const SmallParams* __restrict__ gsp) {
  // A runtime layer index turns c_small.bias[layer][c] into indexed constant-bank loads (LDC c[3][R+imm], ~30 cycles
  // each and not pipelined); the same words read from the packed image in global memory are warp-uniform LDG.128s
  // that pipeline, so the rolled epilogue takes its biases from there.
  float bias[32], wden[kDens ? 32 : 1];
#pragma unroll
  for (int q = 0; q < 8; ++q) {
    const float4 t = __ldg(reinterpret_cast<const float4*>(gsp->bias[layer] + c0) + q);
    bias[4 * q] = t.x, bias[4 * q + 1] = t.y, bias[4 * q + 2] = t.z, bias[4 * q + 3] = t.w;
    if (kDens) {
      const float4 u = __ldg(reinterpret_cast<const float4*>(gsp->w_density + c0) + q);
      wden[4 * q] = u.x, wden[4 * q + 1] = u.y, wden[4 * q + 2] = u.z, wden[4 * q + 3] = u.w;
    }
  }
  uint8_t* slab = myA + (c0 >> 6) * kStageBytes + rowoff;
  const uint32_t ci0 = (uint32_t)(c0 & 63) >> 3;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    uint32_t w[4], wl[4];
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int c = j * 8 + 2 * e;
      float a = __uint_as_float(v[c]), b = __uint_as_float(v[c + 1]);
      fadd2(a, b, bias[c], bias[c + 1]);
      if (kDens)  // density_layer on the fp32 (un-rounded) h7        (models/mip_nerf.py:98)
        ffma2(dpart[2 * e], dpart[2 * e + 1], fmaxf(a, 0.f), fmaxf(b, 0.f), wden[kDens ? c : 0],
              wden[kDens ? c + 1 : 0]);
      if (kX3) {
        if (kRelu) a = fmaxf(a, 0.f), b = fmaxf(b, 0.f);
        w[e] = pack2<kFmt>(a, b);
        const float2 h = unpack2<kFmt>(w[e]);
        wl[e] = pack2<kFmt>(a - h.x, b - h.y);
      } else {
        w[e] = kRelu ? pack2_relu<kFmt>(a, b) : pack2<kFmt>(a, b);
      }
    }
    if (kA32) {
      const uint32_t off = a_chunk_offset<true>((int)(rowoff >> 7), c0 + j * 8);
      *reinterpret_cast<uint4*>(myA + off) = make_uint4(w[0], w[1], w[2], w[3]);
      if (kX3) *reinterpret_cast<uint4*>(myA + kABytes + off) = make_uint4(wl[0], wl[1], wl[2], wl[3]);
    } else {
      const uint32_t off = ((ci0 + j) ^ rx) << 4;  // sw128_offset(row, .) with the row part hoisted
      *reinterpret_cast<uint4*>(slab + off) = make_uint4(w[0], w[1], w[2], w[3]);
      if (kX3) *reinterpret_cast<uint4*>(slab + kABytes + off) = make_uint4(wl[0], wl[1], wl[2], wl[3]);
    }
  }
}

template <int kFmt, bool kX3, bool kA32 = false>
__device__ __forceinline__ void epilogue_trunk_rolled(uint32_t t_acc, uint8_t* myA, int row, float& dens, int layer,
                                                      const SmallParams* __restrict__ gsp, int kk_begin = 0,
                                                      int kk_end = 4) {
  // columns [64 kk_begin, 64 kk_end): the split modes share one ray's epilogue between both worker groups
  float dpart[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  const uint32_t rowoff = (uint32_t)row * 128u, rx = (uint32_t)row & 7u;
  uint32_t v0[32], v1[32];
  tmem_ld32(t_acc + 64 * kk_begin, v0);
#pragma unroll 1
  for (int kk = kk_begin; kk < kk_end; ++kk) {
    tmem_ld_wait();
    tmem_ld32(t_acc + 64 * kk + 32, v1);
    if (layer == 7) epilogue_chunk<kFmt, kX3, true, true, kA32>(v0, layer, 64 * kk, myA, rowoff, rx, dpart, gsp);
    else if (layer < 8) epilogue_chunk<kFmt, kX3, true, false, kA32>(v0, layer, 64 * kk, myA, rowoff, rx, dpart, gsp);
    else epilogue_chunk<kFmt, kX3, false, false, kA32>(v0, layer, 64 * kk, myA, rowoff, rx, dpart, gsp);
    tmem_ld_wait();
    if (kk + 1 < kk_end) tmem_ld32(t_acc + 64 * kk + 64, v0);
    if (layer == 7) epilogue_chunk<kFmt, kX3, true, true, kA32>(v1, layer, 64 * kk + 32, myA, rowoff, rx, dpart, gsp);
    else if (layer < 8) epilogue_chunk<kFmt, kX3, true, false, kA32>(v1, layer, 64 * kk + 32, myA, rowoff, rx, dpart, gsp);
    else epilogue_chunk<kFmt, kX3, false, false, kA32>(v1, layer, 64 * kk + 32, myA, rowoff, rx, dpart, gsp);
  }
  if (layer == 7)
    dens = ((dpart[0] + dpart[1]) + (dpart[2] + dpart[3])) + ((dpart[4] + dpart[5]) + (dpart[6] + dpart[7]));
}

// view layer epilogue + colour head (models/mip_nerf.py:108-110); vb = per-ray view-direction bias
template <int kFmt>
__device__ __forceinline__ void epilogue_view(uint32_t t_acc, const float* __restrict__ vb, float& rgb0,
                                              float& rgb1, float& rgb2, uint8_t* __restrict__ vdump = nullptr,
                                              int row = 0, int k_begin = 0, int k_end = 4) {
  // columns [32 k_begin, 32 k_end) (split modes: half of the 128 per worker group, partial colour dots)
  float acc[3][4] = {{0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}, {0.f, 0.f, 0.f, 0.f}};  // independent chains
  uint32_t v[2][32];
  tmem_ld32(t_acc + 32 * k_begin, v[0]);  // k_begin is even (0 or 2)
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    if (k < k_begin || k >= k_end) continue;
    tmem_ld_wait();
    if (k + 1 < k_end) tmem_ld32(t_acc + 32 * (k + 1), v[(k + 1) & 1]);
#pragma unroll
    for (int e = 0; e < 32; e += 4) {
      const float4 b4 = *reinterpret_cast<const float4*>(vb + 32 * k + e);
      const float bb[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; i += 2) {
        const int c = 32 * k + e + i;
        float y0 = __uint_as_float(v[k & 1][e + i]), y1 = __uint_as_float(v[k & 1][e + i + 1]);
        fadd2(y0, y1, bb[i], bb[i + 1]);
        y0 = fmaxf(y0, 0.f), y1 = fmaxf(y1, 0.f);
        v[k & 1][e + i] = __float_as_uint(y0), v[k & 1][e + i + 1] = __float_as_uint(y1);  // kept for the dump
#pragma unroll
        for (int ch = 0; ch < 3; ++ch)
          ffma2(acc[ch][i], acc[ch][i + 1], y0, y1, c_small.w_color[ch][c], c_small.w_color[ch][c + 1]);
      }
    }
    if (vdump) {  // training: the 16-bit view-layer output, same tile layout as the trunk's activation slabs
      uint8_t* slab = vdump + (k >> 1) * kStageBytes + (uint32_t)row * 128u;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const uint32_t* y = v[k & 1] + 8 * j;
        const uint32_t ci = (uint32_t)((k & 1) * 4 + j);
        *reinterpret_cast<uint4*>(slab + ((ci ^ ((uint32_t)row & 7u)) << 4)) =
            make_uint4(pack2<kFmt>(__uint_as_float(y[0]), __uint_as_float(y[1])),
                       pack2<kFmt>(__uint_as_float(y[2]), __uint_as_float(y[3])),
                       pack2<kFmt>(__uint_as_float(y[4]), __uint_as_float(y[5])),
                       pack2<kFmt>(__uint_as_float(y[6]), __uint_as_float(y[7])));
      }
    }
  }
  rgb0 = (acc[0][0] + acc[0][1]) + (acc[0][2] + acc[0][3]);
  rgb1 = (acc[1][0] + acc[1][1]) + (acc[1][2] + acc[1][3]);
  rgb2 = (acc[2][0] + acc[2][1]) + (acc[2][2] + acc[2][3]);
}

// Gaussian + 96 IPE features of one sample row of a ray (or, in MLP-only mode, the caller's features) into the
// slot's feature tile: SW128 slab (K 0..63) + SW64 tail (K 64..95).
template <int kFmt, bool kX3>
__device__ __forceinline__ void ipe_row_group(const LevelParams& p, const RayGeom& g, int64_t ray, int row, float t0,
                                              float t1, uint8_t* myF) {
  float mean[3] = {0.f, 0.f, 0.f}, cov[3] = {0.f, 0.f, 0.f};
  const float* fin = nullptr;
  if (p.feat_in) {
    fin = p.feat_in + (ray * kN + row) * kFeat;  // MLP-only mode: the caller's encoding
  } else {
    float tm, tv, rv;
    frustum_moments(t0, t1, g.radius_sq, tm, tv, rv);
    lift_gaussian(g, tm, tv, rv, mean, cov);
    if (p.disable_integration) cov[0] = cov[1] = cov[2] = 0.f;
  }
#pragma unroll
  for (int gi = 0; gi < 6; ++gi) {
    float fsin[8], fcos[8];
    if (fin) {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        fsin[e] = __ldg(fin + gi * 8 + e);
        fcos[e] = __ldg(fin + 48 + gi * 8 + e);
      }
    } else {
#pragma unroll
      for (int e = 0; e < 8; ++e) {
        const int f = gi * 8 + e;  // feature index = degree*3 + coord   (models/mip.py:335-341)
        // (measured: the accurate sinf / expf in place of the MUFU pair changes the split modes' error against the
        //  reference goldens by < 3 % — 1.06e-4 vs 1.08e-4 on the worst one — and costs 7x the IPE time: not used)
        ipe_pair<true>(mean[f % 3], cov[f % 3], f / 3, fsin[e], fcos[e]);
      }
    }
    const uint32_t o_sin = sw128_offset(row, gi * 8);                                     // K = f
    const uint32_t o_cos = gi < 2 ? sw128_offset(row, 48 + gi * 8)                        // K = 48 + f < 64
                                  : kStageBytes + sw64_offset(row, (gi - 2) * 8);         // K = 64.. -> SW64 tail
    if (kX3) {  // low halves go to the second feature tile (the other slot's, unused in the split modes)
      store8_split<kFmt>(myF + o_sin, myF + kFBytes + o_sin, fsin);
      store8_split<kFmt>(myF + o_cos, myF + kFBytes + o_cos, fcos);
    } else {
      store8<kFmt>(myF + o_sin, fsin);
      store8<kFmt>(myF + o_cos, fcos);
    }
  }
}

// kX3 (split-operand parity modes, CTA pair only): ONE ray per CTA (slot 0); every activation / feature / weight is
// carried as hi + lo 16-bit halves (A_lo and F_lo live where slot 1's tiles would be, W_lo stages alternate with W_hi
// in the ring) and every K step issues  A_hi.W_hi + A_lo.W_hi + A_hi.W_lo  into the same fp32 accumulator: 3x the MMAs,
// ~2^-22 (fp16 halves) / 2^-16 (bf16 halves) relative operand error instead of 2^-11 / 2^-8.
// v4 (kTS) issue path of one (layer, N half, slot): every K-slab index is a compile-time constant (fully unrolled), so an
// MMA costs the one issuing thread a handful of uniform-register moves — with run-time slab indices and feature /
// activation branches it was ~100 cycles per 64-cycle MMA.  kType 0: layer 0 (three feature slabs, SS form);
// 1: eight activation slabs (TS form); 2: layer 5 = eight activation slabs + three feature slabs.
constexpr int kTsSlabsPerStage = 4;
template <int kType>
__device__ __forceinline__ void ts_issue_half(uint32_t d_tmem, uint32_t a_tmem, uint32_t f_base, uint32_t sW_u,
                                              uint32_t bars_u, int& st, uint32_t& wph, uint32_t idesc) {
  constexpr int ns = kType == 0 ? 3 : (kType == 1 ? 8 : 11);
#pragma unroll
  for (int s0 = 0; s0 < ns; s0 += kTsSlabsPerStage) {
    mbar_wait_fast(bars_u + st * 8, wph);  // w_full[st]: both CTAs' rows of up to four slabs landed
    tc_fence_after();
    const uint32_t b0 = desc_lo(sW_u + st * (kTsSlabsPerStage * 4096u));
#pragma unroll
    for (int i = 0; i < kTsSlabsPerStage; ++i) {
      const int s2 = s0 + i;
      if (s2 < ns) {
        const uint32_t b_lo = b0 + i * (4096u >> 4);
        const int fs = kType == 0 ? s2 : (kType == 2 ? s2 - 8 : -1);  // >= 0: K-slab fs of the feature tile
        const uint32_t first = s2 > 0 ? 1u : 0u;
        if (fs < 0) {  // K-slab s2 of the activations: TMEM columns 16 s2 .. 16 s2 + 15
          umma_ts_pair_lohi(d_tmem, a_tmem + 16 * s2, b_lo, kDescHiSw64, idesc, first);
          umma_ts_pair_lohi(d_tmem, a_tmem + 16 * s2 + 8, b_lo + 2, kDescHiSw64, idesc, 1u);
        } else {  // features: SS form from the slot's feature tile
          const uint32_t a_lo = desc_lo(fs < 2 ? f_base + fs * 64 : f_base + kStageBytes);
          const uint32_t a_hi = fs == 2 ? kDescHiSw64 : kDescHiSw128;
          umma_ss_pair_lohi(d_tmem, a_lo, a_hi, b_lo, kDescHiSw64, idesc, first);
          umma_ss_pair_lohi(d_tmem, a_lo + 2, a_hi, b_lo + 2, kDescHiSw64, idesc, 1u);
        }
      }
    }
    umma_commit_pair_addr(bars_u + (kStages + st) * 8);  // w_empty[st]
    if (++st == kStages) {
      st = 0;
      wph ^= 1;
    }
  }
}

template <int kFmt, bool kPair, bool kX3, bool kTrain = false, bool kTS = false, bool kNoise = false>
__global__ void __launch_bounds__(kThreads, 1) mlp_level_kernel(const LevelParams p) {
  static_assert(!kNoise || (kPair && !kTS && !kTrain), "density noise: the v1 CTA-pair kernels (kTrain checks p.dnoise itself)");
  static_assert(!kX3 || kPair, "split-operand modes exist for the CTA-pair kernel only");
  static_assert(!kTS || (kPair && !kX3 && !kTrain), "the TS variant is the plain CTA-pair inference kernel");
  static_assert(!kTrain || (kPair && !kX3), "the training forward (activation dump) is the plain CTA-pair kernel");
  // Activation-tile layout (a_chunk_offset).  -DMIPNERF_TC_A_SW32 builds the dense K = 16 block layout (never in the
  // training forward, whose tiles leave the SM as tile images).  Measured: all parity tests pass with it and the level
  // kernel takes 0.542 ms against 0.541 ms — the A operand's access pattern is not what holds a weight stage at 331
  // instead of 256 cycles — so the proven SW128 layout stays the default.
#ifdef MIPNERF_TC_A_SW32
  constexpr bool kA32 = !kTrain;
#else
  constexpr bool kA32 = false;
#endif
  constexpr int kSlots = kX3 ? 1 : 2;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  uint8_t* sA = smem + kSmemA;
  uint8_t* sF = smem + kSmemF;
  // kTS: no activation tiles in shared memory; their 128 KB hold the weight ring — 6 stages of 16 KB = up to FOUR K = 32
  // slabs of this CTA's 64 rows of one N = 128 half (a TS MMA of that shape is 64 cycles: one wait / commit per two
  // MMAs made the issuing thread the bottleneck, 250 cycles per 128 cycles of tensor work) — and the barrier block
  constexpr int kNS = kStages;
  constexpr int kTsSlabs = kTsSlabsPerStage;                   // K slabs per stage
  constexpr uint32_t kRingStride = kTS ? kTsSlabs * 4096u : kWStage;
  uint8_t* sW = kTS ? sA : smem + kSmemW;
  uint64_t* bars = reinterpret_cast<uint64_t*>(kTS ? sA + kStages * kTsSlabs * 4096 : smem + kSmemMisc);
  uint64_t* w_full = bars;                  // [kNS] producer (+ peer relay) -> MMA   (tx bytes)
  uint64_t* w_empty = bars + kNS;           // [kNS] MMA -> producer                  (tcgen05.commit)
  uint64_t* a_ready = bars + 2 * kNS;       // [2] worker warps -> MMA: A operand written, accumulator drained
  uint64_t* acc_full = bars + 2 * kNS + 2;  // [2] MMA -> workers                          (tcgen05.commit)
  uint64_t* f_ready = bars + 2 * kNS + 4;   // [2] IPE warp -> MMA: feature tile of the next ray written
  uint64_t* f_free = bars + 2 * kNS + 6;    // [2] MMA -> IPE warp: layer 5 has read the feature tile
  uint64_t* acc_drained = bars + 2 * kNS + 8;  // [2] kTS: worker warps -> MMA: half 0 of the accumulator has been read
  static_assert(kTS || (2 * kStages + 8) * 8 <= 256, "barrier block");
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + kSmemMisc + 256);
  float* vb_s = reinterpret_cast<float*>(smem + kSmemMisc + 272);  // [2][128] per-ray view-layer bias
  float* cs = vb_s + 256;                                          // [2][4]   scan carries
  float* ps = cs + 8;                                              // [2][4][8] partial sums

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = kPair ? cluster_ctarank() : 0u;
  const bool leader = !kPair || rank == 0;
  if (tid == 0) {
    for (int i = 0; i < kNS; ++i) {
      mbar_init(&w_full[i], (kPair && leader) ? 2 : 1);  // leader: own producer + the peer's relay
      mbar_init(&w_empty[i], 1);
    }
    for (int s = 0; s < 2; ++s) {
      if (kTS) mbar_init(&acc_drained[s], 8);
      mbar_init(&a_ready[s], kX3 ? 16 : (kPair ? 8 : 4));  // one arrive per worker warp (of both CTAs in pair mode;
                                                             // split modes: both worker groups work on the one slot)
      mbar_init(&acc_full[s], 1);
      mbar_init(&f_ready[s], kPair ? 2 : 1);  // one arrive per IPE warp (of both CTAs)
      mbar_init(&f_free[s], 1);
    }
    fence_mbar_init();
  }
  if (warp == 0) {
    if (kPair) tmem_alloc_pair(tmem_slot, 512);
    else tmem_alloc(tmem_slot, 512);
  }
  tc_fence_before();
  __syncthreads();
  if (kPair) cluster_sync_all();  // peer barriers initialised before any remote arrive / multicast
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int rounds = p.rounds;
  auto tile_of = [&](int round, int slot) -> int64_t {
    return kPair ? ((((int64_t)round * (gridDim.x >> 1) + (blockIdx.x >> 1)) * kSlots + slot) * 2 + rank)
                 : (((int64_t)round * gridDim.x + blockIdx.x) * 2 + slot);
  };

  if (warp == 0) {
    // ============================ weight producer ============================
    if (lane == 0) {
      TRACER_DECL(0);
      int st = 0;
      uint32_t ph = 0;
      const uint64_t w_policy = kTrain ? l2_policy_evict_last() : 0ull;
      if (kTS) {  // per layer: (half 0: slot 0, slot 1), (half 1: slot 0, slot 1) — the MMA issue order
        for (int round = 0; round < rounds; ++round)
          for (int l = 0; l < kNumLayers; ++l) {
            const int ns = num_k32(l), nh = l == 9 ? 1 : 2;
            for (int h = 0; h < nh; ++h)
              for (int slot = 0; slot < 2; ++slot) {
                // rows [64 rank, +64) of the packed image's [128 x 64 B] SW64 stage (layer l, N-half h, K-slab s)
                const uint8_t* src = p.wimage + layer_offset(l) + (uint32_t)h * (layer_bytes(l) / num_halves(l)) + rank * 4096u;
                for (int s2 = 0; s2 < ns; s2 += kTsSlabs) {
                  const int cnt = ns - s2 < kTsSlabs ? ns - s2 : kTsSlabs;
                  mbar_wait(&w_empty[st], ph ^ 1);
                  mbar_arrive_expect_tx(&w_full[st], (uint32_t)cnt * 4096u);
                  for (int i = 0; i < cnt; ++i)
                    bulk_g2s(sW + st * kRingStride + i * 4096u, src + (size_t)(s2 + i) * kWStage, 4096u, &w_full[st]);
                  if (++st == kNS) {
                    st = 0;
                    ph ^= 1;
                  }
                }
              }
          }
      } else
      for (int round = 0; round < rounds; ++round)
        for (int l = 0; l < kNumLayers; ++l) {
          const int ns = num_k32(l);
          const int nh = kPair ? 1 : num_halves(l);
          const uint32_t bytes = (kPair && l == 9) ? kViewPairStage : kWStage;
          for (int slot = 0; slot < kSlots; ++slot)
            for (int h = 0; h < nh; ++h) {
              // pair mode: this CTA streams only half `rank` of the layer (64 rows for the view layer)
              const uint8_t* src =
                  (kPair && l == 9) ? p.wimage + kViewPairOffset + rank * 8 * kViewPairStage
                                    : p.wimage + layer_offset(l) + (kPair ? rank : (uint32_t)h) * (layer_bytes(l) / num_halves(l));
              for (int s = 0; s < ns; ++s) {
#pragma unroll
                for (int part = 0; part < (kX3 ? 2 : 1); ++part) {  // x3: W_hi stage, then the W_lo stage of the slab
                  mbar_wait(&w_empty[st], ph ^ 1);
                  mbar_arrive_expect_tx(&w_full[st], bytes);
                  if (kTrain) bulk_g2s_hint(sW + st * kWStage, src, bytes, &w_full[st], w_policy);  // keep the image in L2
                  else bulk_g2s(sW + st * kWStage, src + (part ? kLoOffset : 0), bytes, &w_full[st]);
                  TRACE(EV(0, 0, l, st));
                  if (++st == kStages) {
                    st = 0;
                    ph ^= 1;
                  }
                }
                src += bytes;
              }
            }
        }
      TRACER_DONE(0);
    }
  } else if (warp == 1) {
    // ============================ MMA issuer ============================
    // One elected lane runs the whole role; every operand is derived from warp-uniform values
    // (shuffled bases, loop counters) so the tcgen05 operands stay in uniform registers.
    const uint32_t tm_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t sA_u = __shfl_sync(0xffffffffu, smem_u32(sA), 0);
    const uint32_t sF_u = __shfl_sync(0xffffffffu, smem_u32(sF), 0);
    const uint32_t sW_u = __shfl_sync(0xffffffffu, smem_u32(sW), 0);
    const uint32_t bars_u = __shfl_sync(0xffffffffu, smem_u32(bars), 0);
    const uint32_t rank_u = __shfl_sync(0xffffffffu, rank, 0);
    if (elect_one_sync()) {
      if (!kPair || rank_u == 0) {
        TRACER_DECL(1);
        constexpr int kM = kPair ? 256 : 128;
        constexpr int kNn = kPair ? 256 : 128;
        const uint32_t idesc = make_idesc_f16(kM, kNn, kFmt);
        const uint32_t idesc_view = make_idesc_f16(kM, 128, kFmt);
        int st = 0;
        uint32_t wph = 0, ph_ready0 = 0, ph_ready1 = 0, ph_f0 = 0, ph_f1 = 0;
        if (kTS) {
          const uint32_t idesc_t = make_idesc_f16(256, 128, kFmt);
          uint32_t ph_dr[2] = {0u, 0u}, ph_rd[2] = {0u, 0u}, ph_ff[2] = {0u, 0u};
          V4_DECL();
          const long long t_all_ = V4_CLK();
          for (int round = 0; round < rounds; ++round)
            for (int l = 0; l < kNumLayers; ++l) {
              const int ns = num_k32(l), nh = l == 9 ? 1 : 2;
              for (int h = 0; h < nh; ++h)
                for (int slot = 0; slot < 2; ++slot) {
                  if (h == 0) {
                    if (l == 0) {  // the ray's feature tile (written ahead of time by the IPE warp)
                      const long long t_ = V4_CLK();
                      mbar_wait_fast(bars_u + (2 * kNS + 4 + slot) * 8, ph_ff[slot]);
                      ph_ff[slot] ^= 1;
                      V4_ADD(0, t_);
                    }
                    const long long t_ = V4_CLK();
                    mbar_wait_fast(bars_u + (2 * kNS + slot) * 8, ph_rd[slot]);  // a_ready: activations written
                    ph_rd[slot] ^= 1;
                    V4_ADD(1, t_);
                  } else {
                    const long long t_ = V4_CLK();
                    mbar_wait_fast(bars_u + (2 * kNS + 8 + slot) * 8, ph_dr[slot]);  // acc_drained: half 0 read out
                    ph_dr[slot] ^= 1;
                    V4_ADD(2, t_);
                  }
                  tc_fence_after();
                  const uint32_t d_tmem = tm_u + slot * 256, a_tmem = d_tmem + 128;
                  const uint32_t f_base = sF_u + slot * kFBytes;
                  {
                    const long long tw_ = V4_CLK();
                    if (l == 0) ts_issue_half<0>(d_tmem, a_tmem, f_base, sW_u, bars_u, st, wph, idesc_t);
                    else if (l == 5) ts_issue_half<2>(d_tmem, a_tmem, f_base, sW_u, bars_u, st, wph, idesc_t);
                    else ts_issue_half<1>(d_tmem, a_tmem, f_base, sW_u, bars_u, st, wph, idesc_t);
                    V4_ADD(3, tw_);  // issue + weight waits + tensor back-pressure of this (layer, half, slot)
                  }
                  umma_commit_pair(&acc_full[slot]);
                  if (l == 5 && h == 1) umma_commit_pair(&f_free[slot]);
                }
            }
          V4_ADD(4, t_all_);
          V4_FLUSH(0);
        } else
        for (int round = 0; round < rounds; ++round)
          for (int l = 0; l < kNumLayers; ++l) {
            const int ns = num_k32(l);
            const int nh = kPair ? 1 : num_halves(l);
            const uint32_t id = l == 9 ? idesc_view : idesc;
            for (int slot = 0; slot < kSlots; ++slot) {
              if (l == 0) {  // the ray's feature tile (written ahead of time by the IPE warp)
                if (slot == 0) {
                  mbar_wait_fast(bars_u + (2 * kStages + 4) * 8, ph_f0);
                  ph_f0 ^= 1;
                } else {
                  mbar_wait_fast(bars_u + (2 * kStages + 5) * 8, ph_f1);
                  ph_f1 ^= 1;
                }
              }
              if (slot == 0) {
                mbar_wait_fast(bars_u + (2 * kStages) * 8, ph_ready0);
                ph_ready0 ^= 1;
              } else {
                mbar_wait_fast(bars_u + (2 * kStages + 1) * 8, ph_ready1);
                ph_ready1 ^= 1;
              }
              tc_fence_after();
              TRACE(EV(1, 0, l, slot));
              const uint32_t a_base = sA_u + slot * kABytes;
              const uint32_t f_base = sF_u + slot * kFBytes;
              for (int h = 0; h < nh; ++h) {
                const uint32_t d_tmem = tm_u + slot * 256 + h * 128;
                for (int s = 0; s < ns; ++s) {
                  mbar_wait_fast(bars_u + st * 8, wph);  // w_full[st] (pair: both halves landed)
                  tc_fence_after();
                  TRACE(EV(1, 1, l, slot * 16 + s));
                  // A side of K-slab s (32 wide): activations live in 64-wide SW128 slabs, the features in
                  // one SW128 slab (K 0..63) + one SW64 slab (K 64..95)
                  const int fs = (l == 0) ? s : (l == 5 ? s - 8 : -1);  // >= 0: K-slab fs of the feature tile
                  const bool a_sw64 = fs == 2;
                  const bool a_blk = kA32 && fs < 0;  // activation tile as dense K = 16 blocks (2 per K-slab)
                  const uint32_t a_addr = fs < 0 ? (kA32 ? a_base + s * 8192u : a_base + (s >> 1) * kStageBytes + (s & 1) * 64)
                                                 : (fs < 2 ? f_base + fs * 64 : f_base + kStageBytes);
                  const uint32_t a_lo_addr = a_addr + (fs < 0 ? kABytes : kFBytes);  // x3: low halves of the A operand
                  const uint32_t a_step = a_blk ? 4096u : 32u;  // second K = 16 half of the slab
                  auto a_desc = [&](uint32_t addr) {
                    return a_blk ? make_sw32_desc(addr) : (a_sw64 ? make_sw64_desc(addr) : make_sw128_desc(addr));
                  };
                  uint32_t b_addr = sW_u + st * kWStage;
#pragma unroll
                  for (int j = 0; j < 2; ++j) {
                    const uint64_t ad = a_desc(a_addr + j * a_step);
                    const uint64_t bd = make_sw64_desc(b_addr + j * 32);
                    if (kPair) umma_ss_pair(d_tmem, ad, bd, id, (s > 0 || j > 0) ? 1u : 0u);
                    else umma_ss(d_tmem, ad, bd, id, (s > 0 || j > 0) ? 1u : 0u);
                  }
                  if (kX3) {
#pragma unroll
                    for (int j = 0; j < 2; ++j) {  // A_lo . W_hi
                      const uint64_t ad = a_desc(a_lo_addr + j * a_step);
                      umma_ss_pair(d_tmem, ad, make_sw64_desc(b_addr + j * 32), id, 1u);
                    }
                    umma_commit_pair(&w_empty[st]);
                    if (++st == kStages) {
                      st = 0;
                      wph ^= 1;
                    }
                    mbar_wait_fast(bars_u + st * 8, wph);  // the slab's W_lo stage
                    tc_fence_after();
                    b_addr = sW_u + st * kWStage;
#pragma unroll
                    for (int j = 0; j < 2; ++j) {  // A_hi . W_lo
                      const uint64_t ad = a_desc(a_addr + j * a_step);
                      umma_ss_pair(d_tmem, ad, make_sw64_desc(b_addr + j * 32), id, 1u);
                    }
                  }
                  // stage reusable (in both CTAs) once these MMAs have read it
                  if (kPair) umma_commit_pair(&w_empty[st]);
                  else umma_commit(&w_empty[st]);
                  if (++st == kStages) {
                    st = 0;
                    wph ^= 1;
                  }
                }
              }
              if (kPair) umma_commit_pair(&acc_full[slot]);  // accumulator of (l, slot) complete
              else umma_commit(&acc_full[slot]);
              if (l == 5) {  // last reader of this ray's feature tile: hand it back to the IPE warp(s)
                if (kPair) umma_commit_pair(&f_free[slot]);
                else umma_commit(&f_free[slot]);
              }
              TRACE(EV(1, 2, l, slot));
            }
          }
        TRACER_DONE(1);
      } else {
        // pair mode, non-leader CTA: relay "my half of stage st has landed" to the leader's w_full[st]
        int st = 0;
        uint32_t wph = 0;
        const uint32_t leader_w_full = mapa_u32(bars_u, 0);
        for (int round = 0; round < rounds; ++round)
          for (int l = 0; l < kNumLayers; ++l) {
            const int ns = num_k32(l);
            // kTS: two N halves per slot, up to four K slabs per stage
            const int per_layer = kTS ? (l != 9 ? 4 : 2) * ((ns + kTsSlabs - 1) / kTsSlabs) : 2 * ns;
            for (int k = 0; k < per_layer; ++k) {
              mbar_wait_fast(bars_u + st * 8, wph);
              mbar_arrive_remote(leader_w_full + st * 8);
              if (++st == kNS) {
                st = 0;
                wph ^= 1;
              }
            }
          }
      }
    }
    __syncwarp();
  } else if (warp >= 10) {
    // ============================ IPE warps (one per slot) ============================
    // Conical-frustum Gaussians + 96 IPE features of the slot's NEXT ray, written into the feature
    // tile as soon as layer 5 of the current ray has read it: off the per-ray critical path.
    const int slot = warp - 10;
    uint8_t* myF = sF + slot * kFBytes;
    const int my_rounds = slot < kSlots ? rounds : 0;  // x3: only slot 0 exists
    // One (kN+1)-float array per slot for the in-kernel resampler, carved out of the alignment slack at the end of
    // the dynamic allocation when the runtime placed the buffer favourably (it does: 1024-aligned base).
    float* early_scratch = nullptr;
    {
      const uint32_t used = (uint32_t)(smem - smem_raw) + kSmemMisc + kMiscBytes;
      const uint32_t need = 2u * (kN + 1) * (uint32_t)sizeof(float);
      if (used + need <= kSmemTotal)
        early_scratch = reinterpret_cast<float*>(smem + kSmemMisc + kMiscBytes) + slot * (kN + 1);
    }
    const uint32_t f_ready_leader = kPair ? mapa_u32(smem_u32(&f_ready[slot]), 0) : 0u;
    uint32_t ph_free = 0;
#ifdef MIPNERF_TC_TRACE
    Tracer tracer;
    if (slot == 0 && lane == 0) tracer.init(4);
#endif
    for (int round = 0; round < my_rounds; ++round) {
      const int64_t tile = tile_of(round, slot);
      const int64_t ray = tile < p.num_rays ? tile : p.num_rays - 1;
      TRACE(EV(3, 2, 0, slot));
      // ---- ray prologue of the NEXT ray of this slot.  None of it touches the feature tile, so it runs while
      //      layers 0..5 of the current ray are still reading that tile (this warp would be idle otherwise).
      RayGeom g{};
      if (!p.feat_in) g = load_ray_geom(p.origins, p.directions, p.radii, ray);
      float* t_ray = p.t + ray * (kN + 1);
      if (p.t_mode == 1) {
        // coarse fenceposts (bit-identical to coarse_t_kernel)
        const float nr = __ldg(p.near + ray), fr = __ldg(p.far + ray);
        const bool jit = draws_active(p.t_rand);
        const Draws t_rand = draws_at_state<kTrain>(p.t_rand, p.rng_state);
        for (int j = lane; j <= kN; j += 32)
          __stcg(t_ray + j, coarse_fencepost(nr, fr, j, kN, p.disparity, jit,
                                             jit ? draw_uniform(t_rand, ray, j, kN + 1) : 0.f));
      } else if (p.t_mode == 2 && early_scratch) {
        resample_warp_lean<true>(p.t_prev + ray * (kN + 1), p.w_prev + ray * kN, kN, kN + 1, p.randomized,
                                 draws_at_state<kTrain>(p.u_jitter, p.rng_state),
                                 ray, p.resample_padding, early_scratch, t_ray,
                                 p.inds ? p.inds + ray * (kN + 1) : nullptr, lane);
      }
      if (p.vb_mode == 1) {
        // per-ray view-layer bias  b[n] + W[n, 256:283] . pos_enc(viewdir)   (models/mip.py:353-363,
        // models/mip_nerf.py:106-108): lane f < 27 owns encoding element f, lane owns outputs n = lane + 32 j
        float enc = 0.f;
        if (lane < kViewDim) {
          if (lane < 3) {
            enc = __ldg(p.viewdirs + ray * 3 + lane);  // append_identity
          } else {
            const int gidx = lane - 3, is_cos = gidx >= 12, h = is_cos ? gidx - 12 : gidx;  // scale-major, then xyz
            const float y = __fmul_rn(__ldg(p.viewdirs + ray * 3 + h % 3), __int_as_float((127 + h / 3) << 23));
            enc = sinf(is_cos ? __fadd_rn(y, MIPNERF_HALF_PI_F32) : y);
          }
        }
        const float* wt = reinterpret_cast<const float*>(p.wimage + kViewDirOffset);  // [27][128] | bias[128]
        float acc[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[j] = __ldg(wt + kViewDim * kCond + lane + 32 * j);
#pragma unroll
        for (int k = 0; k < kViewDim; ++k) {
          const float e = __shfl_sync(0xffffffffu, enc, k);
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[j] = fmaf(__ldg(wt + k * kCond + lane + 32 * j), e, acc[j]);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) __stcg(p.view_bias + ray * kCond + lane + 32 * j, acc[j]);
      }
      // Stores above are consumed by this CTA's own warps only (this warp below, the slot's workers later):
      // order them at CTA scope here, off the critical path, and fetch this lane's fenceposts now.
      __threadfence_block();
      __syncwarp();
      const bool t_known = !p.feat_in && !(p.t_mode == 2 && !early_scratch);
      float tq[4][2];  // [i][0|1] = t[i*32+lane], t[i*32+lane+1]
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        tq[i][0] = t_known ? __ldcg(t_ray + i * 32 + lane) : 0.f;  // L2: may be our own stores
        tq[i][1] = t_known ? __ldcg(t_ray + i * 32 + lane + 1) : 0.f;
      }
      TRACE(EV(3, 3, 0, slot));
      mbar_wait(&f_free[slot], ph_free ^ 1);  // first pass falls through (fresh barrier)
      ph_free ^= 1;
      TRACE(EV(3, 0, 0, slot));
      if (p.t_mode == 2 && !early_scratch) {
        // no spare shared memory: the feature tile this warp is about to fill doubles as the scratch
        resample_warp_lean<true>(p.t_prev + ray * (kN + 1), p.w_prev + ray * kN, kN, kN + 1, p.randomized,
                                 draws_at_state<kTrain>(p.u_jitter, p.rng_state), ray, p.resample_padding,
                                 reinterpret_cast<float*>(myF), t_ray,
                                 p.inds ? p.inds + ray * (kN + 1) : nullptr, lane);
        __threadfence_block();
        __syncwarp();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          tq[i][0] = __ldcg(t_ray + i * 32 + lane);
          tq[i][1] = __ldcg(t_ray + i * 32 + lane + 1);
        }
      }
#pragma unroll 1
      for (int i = 0; i < 4; ++i) {
        ipe_row_group<kFmt, kX3>(p, g, ray, i * 32 + lane, tq[0][0], tq[0][1], myF);
#pragma unroll
        for (int r = 0; r < 3; ++r) tq[r][0] = tq[r + 1][0], tq[r][1] = tq[r + 1][1];  // rotate: static indexing
      }
      fence_proxy_async_smem();
      __syncwarp();
      if (lane == 0) {
        if (kPair) mbar_arrive_remote(f_ready_leader);
        else mbar_arrive(&f_ready[slot]);
      }
      TRACE(EV(3, 1, 0, slot));
    }
#ifdef MIPNERF_TC_TRACE
    if (slot == 0 && lane == 0) tracer.finish(4);
#endif
  } else {
    // ============================ slot workers ============================
    // split modes (one ray in flight per CTA): both worker groups share that ray's epilogues — group g takes columns
    // [128 g, 128 g + 128) of every trunk layer (64 g .. of the view layer), so the epilogue, which is fully exposed
    // with a single slot, takes half as long; group 1 hands its partial head sums to group 0 through four spare
    // TMEM columns, group 0 composites.
    const int grp = (warp - 2) >> 2;
    const int slot = kX3 ? 0 : grp;
    const int q = warp & 3;  // TMEM lane quarter this warp may access == sample quarter
    const int row = q * 32 + lane;
    uint8_t* myA = sA + slot * kABytes;
    const uint32_t t_acc = tmem_base + ((uint32_t)(q * 32) << 16) + slot * 256;
    uint32_t ph_acc = 0;
#ifdef MIPNERF_TC_TRACE
    Tracer tracer;
    if (q == 0 && lane == 0) tracer.init(2 + slot);
#endif
    const uint32_t a_ready_leader = kPair ? mapa_u32(smem_u32(&a_ready[slot]), 0) : 0u;
    auto arrive_a_ready = [&]() {
      __syncwarp();
      if (lane == 0) {
        if (kPair) mbar_arrive_remote(a_ready_leader);
        else mbar_arrive(&a_ready[slot]);
      }
    };
    const uint32_t acc_drained_leader = kTS ? mapa_u32(smem_u32(&acc_drained[slot]), 0) : 0u;
    auto arrive_acc_drained = [&]() {  // kTS: half 0 of the accumulator is in registers
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive_remote(acc_drained_leader);
    };
    const uint32_t t_act = t_acc + 128;  // kTS: the slot's 16-bit activation row (128 TMEM columns)
    const int my_rounds = slot < kSlots ? rounds : 0;
    const int kk0 = kX3 ? 2 * grp : 0, kk1 = kX3 ? 2 * grp + 2 : 4;  // this group's share of an epilogue
    const uint32_t t_xchg = tmem_base + ((uint32_t)(q * 32) << 16) + 256;  // split modes: slot 1's columns are unused
    const SmallParams* __restrict__ gsp = reinterpret_cast<const SmallParams*>(p.wimage + kSmallOffset);
    V4_DECL();
    constexpr bool dumping = kTrain;  // a separate instantiation: the inference kernel carries none of this
    const uint64_t dump_policy = kTrain ? l2_policy_evict_first() : 0ull;
    bool dump_pending = false;
    if (slot < kSlots) arrive_a_ready();  // accumulator of this slot is free for the first ray
    for (int round = 0; round < my_rounds; ++round) {
      const int64_t tile = tile_of(round, slot);
      const bool valid = tile < p.num_rays;
      const int64_t ray = valid ? tile : p.num_rays - 1;
      float t0 = 0.f, t1 = 0.f, dnorm = 0.f, vb = 0.f;
      TRACE(EV(2, 0, 0, slot));

      float dens = 0.f, rgb0 = 0.f, rgb1 = 0.f, rgb2 = 0.f;
      for (int l = 0; l < kNumLayers; ++l) {
        const long long tw0_ = V4_CLK();
        mbar_wait(&acc_full[slot], ph_acc);
        ph_acc ^= 1;
        tc_fence_after();
        V4_ADD(0, tw0_);
        TRACE(EV(2, 2, l, slot));
        if (l == 8) {
          // per-ray operands of the view epilogue / compositing: issued one epilogue early so the latency hides
          // behind the bottleneck layer; read through L2 because in the fused-prologue modes they were stored
          // by this CTA's IPE warp (ordered before us by f_ready -> MMA -> acc_full)
          vb = __ldcg(p.view_bias + ray * kCond + row);
          if (!p.raw_rgb_out) {
            t0 = __ldcg(p.t + ray * (kN + 1) + row), t1 = __ldcg(p.t + ray * (kN + 1) + row + 1);
            const float dx = __ldg(p.directions + ray * 3), dy = __ldg(p.directions + ray * 3 + 1),
                        dz = __ldg(p.directions + ray * 3 + 2);
            dnorm = sqrtf(dx * dx + dy * dy + dz * dz);
          }
        }
        if (kTS && l < 9) {
          // two N = 128 halves through the one accumulator; the first half's result waits in registers
          uint32_t held[64];
          const long long te0_ = V4_CLK();
#define MIPNERF_TS_HALF(LL, HH) epilogue_half_ts<kFmt, LL, HH>(t_acc, t_act, held, dens, arrive_acc_drained)
#define MIPNERF_TS_SWITCH(HH)                 \
  switch (l) {                                \
    case 0: MIPNERF_TS_HALF(0, HH); break;    \
    case 1: MIPNERF_TS_HALF(1, HH); break;    \
    case 2: MIPNERF_TS_HALF(2, HH); break;    \
    case 3: MIPNERF_TS_HALF(3, HH); break;    \
    case 4: MIPNERF_TS_HALF(4, HH); break;    \
    case 5: MIPNERF_TS_HALF(5, HH); break;    \
    case 6: MIPNERF_TS_HALF(6, HH); break;    \
    case 7: MIPNERF_TS_HALF(7, HH); break;    \
    default: MIPNERF_TS_HALF(8, HH); break;   \
  }
          MIPNERF_TS_SWITCH(0)
          V4_ADD(1, te0_);
          const long long tw1_ = V4_CLK();
          mbar_wait(&acc_full[slot], ph_acc);  // second half's accumulator; every MMA that read the activations is done
          ph_acc ^= 1;
          tc_fence_after();
          V4_ADD(2, tw1_);
          const long long te1_ = V4_CLK();
          MIPNERF_TS_SWITCH(1)
#undef MIPNERF_TS_SWITCH
#undef MIPNERF_TS_HALF
          tmem_st_wait();
          tc_fence_before();
          arrive_a_ready();
          V4_ADD(3, te1_);
        } else if (l < 9) {
          if (dumping) {  // the previous layer's bulk store must have READ the tile before anyone overwrites it
            if (row == 0 && dump_pending) {
              bulk_store_wait_read();
              dump_pending = false;
            }
            named_bar_sync(1 + slot, 128);
          }
          if (kX3 || MIPNERF_TC_ROLLED_EPILOGUE) {
            epilogue_trunk_rolled<kFmt, kX3, kA32>(t_acc, myA, row, dens, l, gsp, kk0, kk1);
          } else {
            switch (l) {
              case 0: epilogue_trunk<kFmt, 0, kX3, kA32>(t_acc, myA, row, dens); break;
              case 1: epilogue_trunk<kFmt, 1, kX3, kA32>(t_acc, myA, row, dens); break;
              case 2: epilogue_trunk<kFmt, 2, kX3, kA32>(t_acc, myA, row, dens); break;
              case 3: epilogue_trunk<kFmt, 3, kX3, kA32>(t_acc, myA, row, dens); break;
              case 4: epilogue_trunk<kFmt, 4, kX3, kA32>(t_acc, myA, row, dens); break;
              case 5: epilogue_trunk<kFmt, 5, kX3, kA32>(t_acc, myA, row, dens); break;
              case 6: epilogue_trunk<kFmt, 6, kX3, kA32>(t_acc, myA, row, dens); break;
              case 7: epilogue_trunk<kFmt, 7, kX3, kA32>(t_acc, myA, row, dens); break;
              default: epilogue_trunk<kFmt, 8, kX3, kA32>(t_acc, myA, row, dens); break;
            }
          }
          TRACE(EV(2, 3, l, slot));
          fence_proxy_async_smem();
          tc_fence_before();
          arrive_a_ready();
          TRACE(EV(2, 4, l, slot));
          if (dumping) {
            named_bar_sync(1 + slot, 128);  // the whole tile is written (and fenced towards the async proxy)
#ifndef MIPNERF_TRAIN_EXPERIMENT_NO_STORE  // timing experiments only (the dump is then incomplete)
            if (row == 0 && valid) {  // evict-first: the dump must not push the weight image out of L2
              bulk_s2g_hint(p.act_dump + ((size_t)l * p.dump_tiles + ray) * kABytes, myA, kABytes, dump_policy);
              dump_pending = true;
            }
#endif
          }
        } else {
          if (!kX3 || grp == 0) vb_s[slot * 128 + row] = vb;
          if (kX3) named_bar_sync(3, 256);       // both groups read it
          else named_bar_sync(1 + slot, 128);    // vb_s of this ray visible to the whole slot
          epilogue_view<kFmt>(t_acc, vb_s + slot * 128, rgb0, rgb1, rgb2,
#ifdef MIPNERF_TRAIN_EXPERIMENT_NO_VDUMP
                              nullptr, row, kk0, kk1);
#else
                              (dumping && valid) ? p.v_dump + (size_t)ray * (2 * kStageBytes) : nullptr, row, kk0, kk1);
#endif
          tc_fence_before();
          arrive_a_ready();  // accumulator drained: the next ray's layer 0 may start while we composite
          TRACE(EV(2, 3, l, slot));
        }
      }
      if (kX3) {  // partial density / colour dots of group 1 -> group 0 (same TMEM lanes, four spare columns)
        if (grp == 1) {
          tmem_st4(t_xchg, __float_as_uint(dens), __float_as_uint(rgb0), __float_as_uint(rgb1), __float_as_uint(rgb2));
          tmem_st_wait();
        }
        tc_fence_before();
        named_bar_sync(3, 256);
        tc_fence_after();
        if (grp == 1) continue;  // next ray
        uint32_t x0, x1, x2, x3;
        tmem_ld4(t_xchg, x0, x1, x2, x3);
        tmem_ld_wait();
        dens += __uint_as_float(x0), rgb0 += __uint_as_float(x1), rgb1 += __uint_as_float(x2), rgb2 += __uint_as_float(x3);
      }
      if (p.raw_rgb_out) {  // MLP-only mode: hand back the raw heads (models/mip_nerf.py:98,110)
        if (valid) {
          const int64_t sidx = ray * kN + row;
          p.raw_rgb_out[sidx * 3 + 0] = rgb0 + c_small.b_color[0];
          p.raw_rgb_out[sidx * 3 + 1] = rgb1 + c_small.b_color[1];
          p.raw_rgb_out[sidx * 3 + 2] = rgb2 + c_small.b_color[2];
          p.raw_density_out[sidx] = dens + c_small.b_density;
        }
        named_bar_sync(1 + slot, 128);  // vb_s is rewritten before the next ray's view epilogue
        continue;
      }
      float raw_dens = dens + c_small.b_density;
      if (kNoise || kTrain) {  // models/mip_nerf.py:232-233 (randomized and density_noise > 0)
        if (draws_active(p.dnoise) && valid)
          raw_dens = noisy_raw_density(raw_dens, draws_at_state<kTrain>(p.dnoise, p.rng_state), ray, row);
      }
      if (kTrain && valid) {  // training: the raw heads as well (render_backward recomputes the rest; the density
        const int64_t sidx = ray * kN + row;  // head WITH its noise, so that softplus' is taken at the same point)
        p.raw_rgb_keep[sidx * 3 + 0] = rgb0 + c_small.b_color[0];
        p.raw_rgb_keep[sidx * 3 + 1] = rgb1 + c_small.b_color[1];
        p.raw_rgb_keep[sidx * 3 + 2] = rgb2 + c_small.b_color[2];
        p.raw_density_keep[sidx] = raw_dens;
      }
      // ---- activations + compositing over the ray's 128 samples (4 warps of this slot)
      const float density = density_activation(raw_dens, p.density_bias);
      const float cr = rgb_activation(rgb0 + c_small.b_color[0], p.rgb_scale, p.rgb_padding);
      const float cg = rgb_activation(rgb1 + c_small.b_color[1], p.rgb_scale, p.rgb_padding);
      const float cb = rgb_activation(rgb2 + c_small.b_color[2], p.rgb_scale, p.rgb_padding);
      const float dd = density * ((t1 - t0) * dnorm);
      float incl = dd;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const float n = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += n;
      }
      float excl = __shfl_up_sync(0xffffffffu, incl, 1);
      if (lane == 0) excl = 0.f;
      if (lane == 31) cs[slot * 4 + q] = incl;
      named_bar_sync(1 + slot, 128);
      float before = 0.f;
      for (int qq = 0; qq < q; ++qq) before += cs[slot * 4 + qq];
      const float w = -expm1f(-dd) * expf(-(before + excl));
      if (valid) p.weights[ray * kN + row] = w;
      float pr = warp_sum(w * cr), pg = warp_sum(w * cg), pb = warp_sum(w * cb), pw = warp_sum(w),
            pd = warp_sum(w * (0.5f * (t0 + t1)));
      if (lane == 0) {
        float* dst = ps + (slot * 4 + q) * 8;
        dst[0] = pr, dst[1] = pg, dst[2] = pb, dst[3] = pw, dst[4] = pd;
      }
      named_bar_sync(1 + slot, 128);
      TRACE(EV(2, 5, 0, slot));
      if (row == 0 && valid) {
        float s[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
        for (int qq = 0; qq < 4; ++qq)
          for (int k = 0; k < 5; ++k) s[k] += ps[(slot * 4 + qq) * 8 + k];
        const float t_first = __ldcg(p.t + ray * (kN + 1)), t_last = __ldcg(p.t + ray * (kN + 1) + kN);
        float d = s[4];
        if (isnan(d)) d = 0.f;
        else if (isinf(d)) d = d > 0 ? 3.4028234663852886e38f : -3.4028234663852886e38f;
        d = fminf(fmaxf(d, t_first), t_last);
        const float bg = p.white_bkgd ? 1.0f - s[3] : 0.f;
        p.comp_rgb[ray * 3 + 0] = s[0] + bg;
        p.comp_rgb[ray * 3 + 1] = s[1] + bg;
        p.comp_rgb[ray * 3 + 2] = s[2] + bg;
        p.distance[ray] = d;
        p.acc[ray] = s[3];
      }
      named_bar_sync(1 + slot, 128);  // row 0 has consumed ps / everyone cs before the next ray reuses them
    }
    if (kTS && slot == 0 && q == 0 && lane == 0) { V4_FLUSH(8); }
    if (dump_pending) bulk_store_wait_all();  // the last tile's store has left shared memory and reached global
#ifdef MIPNERF_TC_TRACE
    if (q == 0 && lane == 0) tracer.finish(2 + slot);
#endif
  }
  tc_fence_before();
  __syncthreads();
  if (kPair) cluster_sync_all();  // no CTA exits while its peer may still signal it
  if (warp == 0) {
    if (kPair) tmem_dealloc_pair(tmem_base, 512);
    else tmem_dealloc(tmem_base, 512);
  }
}


// =================================================================================================
// v2 ("shared weight stream"): same tile / slot / epilogue structure as mlp_level_kernel<.,true>, but
//   * every weight stage is consumed by BOTH slots before it is released (the producer streams each
//     layer once per round instead of once per slot: half the L2->SMEM weight traffic, half the
//     supply rate the ring has to sustain);
//   * the ring has 12 x 8 KB stages; the 48 KB for that come from not keeping feature tiles in SMEM:
//     the IPE warps write the (pre-swizzled, 16-bit) feature K-slabs of the next ray to a per-CTA
//     global scratch (L2 resident) and the producer streams them through the same ring as A-operand
//     stages for layer 0 and for the skip part of layer 5 (group 6 accumulates onto group 5; the
//     workers are not involved in that split).
// =================================================================================================
constexpr int kStages2 = 12;
constexpr int kNumGroups2 = 11;
constexpr uint32_t kSmemW2 = 2 * kABytes;
constexpr uint32_t kSmemMisc2 = kSmemW2 + kStages2 * kWStage;
constexpr uint32_t kMisc2Bytes = 512 + 16 + 2 * 128 * 4 + 8 * 4 + 2 * 4 * 8 * 4;
constexpr uint32_t kSmemTotal2 = kSmemMisc2 + kMisc2Bytes + 1024;
static_assert(kSmemTotal2 <= 232448, "exceeds 227 KB of shared memory per CTA");
constexpr uint32_t kFeatSlotBytes = 3 * kWStage;                 // K 0..31 | 32..63 | 64..95, [128 x 64 B] SW64 each
constexpr uint32_t kFeatScratchPerCta = 2 * 2 * kFeatSlotBytes;  // 2 slots x 2 (ray parity)
constexpr int kMaxCtas2 = 192;

__host__ __device__ constexpr int g2_layer(int g) { return g < 6 ? g : g - 1; }
__host__ __device__ constexpr int g2_nw(int g) { return (g == 0 || g == 6) ? 3 : 8; }
__host__ __device__ constexpr int g2_wslab0(int g) { return g == 6 ? 8 : 0; }
__host__ __device__ constexpr bool g2_feat(int g) { return g == 0 || g == 6; }

// position in the 12-stage ring + the mbarrier parity of that stage's current fill (fill #n goes to
// stage n % 12 with parity (n / 12) & 1, so both follow by add-and-wrap, no division, no masks)
struct RingPos {
  uint32_t st, par;
};
__device__ __forceinline__ RingPos ring_at(RingPos b, uint32_t off) {  // off < kStages2
  RingPos r{b.st + off, b.par};
  if (r.st >= (uint32_t)kStages2) {
    r.st -= kStages2;
    r.par ^= 1u;
  }
  return r;
}

// MMAs of one (group, slot): kNw weight stages (shared by both slots: waited for by slot 0, released
// after slot 1) and, for the feature groups, the slot's 3 private feature stages as the A operand.
template <int kNw, bool kFeat, int kSlot>
__device__ __forceinline__ void v2_issue(RingPos base, uint32_t bars_u, uint32_t sW_u, uint32_t a_base,
                                         uint32_t d_tmem, uint32_t idesc, bool accumulate_all) {
#pragma unroll
  for (int i = 0; i < kNw; ++i) {
    const RingPos w = ring_at(base, i);
    if (kSlot == 0) mbar_wait_fast(bars_u + w.st * 8, w.par);
    uint32_t a_lo, a_hi, f_empty = 0;
    if (kFeat) {
      const RingPos f = ring_at(base, kNw + kSlot * 3 + i);
      mbar_wait_fast(bars_u + f.st * 8, f.par);
      a_lo = desc_lo(sW_u + f.st * kWStage);
      a_hi = kDescHiSw64;
      f_empty = bars_u + (kStages2 + f.st) * 8;
    } else {
      a_lo = desc_lo(a_base + (i >> 1) * kStageBytes + (i & 1) * 64);
      a_hi = kDescHiSw128;
    }
    tc_fence_after();
    const uint32_t b_lo = desc_lo(sW_u + w.st * kWStage);
    umma_ss_pair_lohi(d_tmem, a_lo, a_hi, b_lo, kDescHiSw64, idesc, (accumulate_all || i > 0) ? 1u : 0u);
    umma_ss_pair_lohi(d_tmem, a_lo + 2, a_hi, b_lo + 2, kDescHiSw64, idesc, 1u);
    if (kFeat) umma_commit_pair_addr(f_empty);                                       // private stage: free now
    if (kSlot == 1) umma_commit_pair_addr(bars_u + (kStages2 + w.st) * 8);  // last use of the shared stage
  }
}

template <int kFmt>
__global__ void __launch_bounds__(kThreads, 1) mlp_level_kernel_v2(const LevelParams p) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t raw = smem_u32(smem_raw);
  uint8_t* smem = smem_raw + (((raw + 1023u) & ~1023u) - raw);
  uint8_t* sA = smem + kSmemA;
  uint8_t* sW = smem + kSmemW2;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + kSmemMisc2);
  uint64_t* w_full = bars;                       // [12] producer (+ peer relay) -> MMA
  uint64_t* w_empty = bars + kStages2;           // [12] MMA -> producer (after the LAST use of the stage)
  uint64_t* a_ready = bars + 2 * kStages2;       // [2]
  uint64_t* acc_full = bars + 2 * kStages2 + 2;  // [2]
  uint64_t* f_ready = bars + 2 * kStages2 + 4;   // [2] IPE warp -> producer: feature slabs of the ray are in the scratch
  uint64_t* f_free = bars + 2 * kStages2 + 6;    // [2] MMA -> IPE warp: group 6 has consumed the ray's feature stages
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(smem + kSmemMisc2 + 512);
  float* vb_s = reinterpret_cast<float*>(smem + kSmemMisc2 + 528);
  float* cs = vb_s + 256;
  float* ps = cs + 8;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const uint32_t rank = cluster_ctarank();
  const bool leader = rank == 0;
  if (tid == 0) {
    for (int i = 0; i < kStages2; ++i) {
      mbar_init(&w_full[i], leader ? 2 : 1);
      mbar_init(&w_empty[i], 1);
    }
    for (int s = 0; s < 2; ++s) {
      mbar_init(&a_ready[s], 8);
      mbar_init(&acc_full[s], 1);
      mbar_init(&f_ready[s], 1);
      mbar_init(&f_free[s], 1);
    }
    fence_mbar_init();
  }
  if (warp == 0) tmem_alloc_pair(tmem_slot, 512);
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const int rounds = p.rounds;
  uint8_t* my_scratch = p.feat_scratch + (size_t)blockIdx.x * kFeatScratchPerCta;
  auto tile_of = [&](int round, int slot) -> int64_t {
    return (((int64_t)round * (gridDim.x >> 1) + (blockIdx.x >> 1)) * 2 + slot) * 2 + rank;
  };

  if (warp == 0) {
    // ============================ producer: weights once per round + per-slot feature slabs ============
    if (lane == 0) {
      TRACER_DECL(0);
      RingPos cur{0u, 0u};
      uint32_t ph_fr0 = 0, ph_fr1 = 0;
      auto fill = [&](const void* src, uint32_t bytes, int tag) {  // fills happen in ring order
        mbar_wait(&w_empty[cur.st], cur.par ^ 1u);
        mbar_arrive_expect_tx(&w_full[cur.st], bytes);
        bulk_g2s(sW + cur.st * kWStage, src, bytes, &w_full[cur.st]);
        TRACE(EV(0, 0, tag, cur.st));
        cur = ring_at(cur, 1u);
      };
      for (int round = 0; round < rounds; ++round)
        for (int g = 0; g < kNumGroups2; ++g) {
          const int l = g2_layer(g), nw = g2_nw(g);
          const uint32_t bytes = l == 9 ? kViewPairStage : kWStage;
          const uint8_t* src = l == 9 ? p.wimage + kViewPairOffset + rank * 8 * kViewPairStage
                                      : p.wimage + layer_offset(l) + rank * (layer_bytes(l) / 2) + g2_wslab0(g) * kWStage;
          for (int i = 0; i < nw; ++i) fill(src + i * bytes, bytes, g);
          if (g2_feat(g)) {
            for (int slot = 0; slot < 2; ++slot) {
              if (g == 0) {  // the IPE warp has published this ray's slabs
                if (slot == 0) {
                  mbar_wait(&f_ready[0], ph_fr0);
                  ph_fr0 ^= 1;
                } else {
                  mbar_wait(&f_ready[1], ph_fr1);
                  ph_fr1 ^= 1;
                }
              }
              const uint8_t* fsrc = my_scratch + (slot * 2 + (round & 1)) * kFeatSlotBytes;
              for (int i = 0; i < 3; ++i) fill(fsrc + i * kWStage, kWStage, g);
            }
          }
        }
      TRACER_DONE(0);
    }
  } else if (warp == 1) {
    // ============================ MMA issuer (leader) / stage relay (peer) ============================
    const uint32_t tm_u = __shfl_sync(0xffffffffu, tmem_base, 0);
    const uint32_t sA_u = __shfl_sync(0xffffffffu, smem_u32(sA), 0);
    const uint32_t sW_u = __shfl_sync(0xffffffffu, smem_u32(sW), 0);
    const uint32_t bars_u = __shfl_sync(0xffffffffu, smem_u32(bars), 0);
    const uint32_t rank_u = __shfl_sync(0xffffffffu, rank, 0);
    if (elect_one_sync()) {
      if (rank_u == 0) {
        TRACER_DECL(1);
        const uint32_t idesc = make_idesc_f16(256, 256, kFmt);
        const uint32_t idesc_view = make_idesc_f16(256, 128, kFmt);
        RingPos base{0u, 0u};
        uint32_t ph_ready0 = 0, ph_ready1 = 0;
        const uint32_t acc_full_u = bars_u + (2 * kStages2 + 2) * 8, f_free_u = bars_u + (2 * kStages2 + 6) * 8;
        for (int round = 0; round < rounds; ++round)
          for (int g = 0; g < kNumGroups2; ++g) {
            const int l = g2_layer(g);
            const bool feat = g2_feat(g);
            const uint32_t id = l == 9 ? idesc_view : idesc;
            // ---- slot 0
            if (g != 6) {  // group 6 continues group 5's accumulation: same A-operand epoch
              mbar_wait_fast(bars_u + (2 * kStages2) * 8, ph_ready0);
              ph_ready0 ^= 1;
              tc_fence_after();
            }
            TRACE(EV(1, 0, g, 0));
            if (feat) v2_issue<3, true, 0>(base, bars_u, sW_u, sA_u, tm_u, id, g == 6);
            else v2_issue<8, false, 0>(base, bars_u, sW_u, sA_u, tm_u, id, false);
            if (g != 5) umma_commit_pair_addr(acc_full_u);
            if (g == 6) umma_commit_pair_addr(f_free_u);
            TRACE(EV(1, 2, g, 0));
            // ---- slot 1
            if (g != 6) {
              mbar_wait_fast(bars_u + (2 * kStages2 + 1) * 8, ph_ready1);
              ph_ready1 ^= 1;
              tc_fence_after();
            }
            TRACE(EV(1, 0, g, 1));
            if (feat) v2_issue<3, true, 1>(base, bars_u, sW_u, sA_u + kABytes, tm_u + 256, id, g == 6);
            else v2_issue<8, false, 1>(base, bars_u, sW_u, sA_u + kABytes, tm_u + 256, id, false);
            if (g != 5) umma_commit_pair_addr(acc_full_u + 8);
            if (g == 6) umma_commit_pair_addr(f_free_u + 8);
            TRACE(EV(1, 2, g, 1));
            base = ring_at(base, feat ? 9u : 8u);
          }
        TRACER_DONE(1);
      } else {
        // peer CTA: relay "stage landed here" to the leader's w_full, in the producer's fill order
        RingPos cur{0u, 0u};
        const uint32_t leader_w_full = mapa_u32(bars_u, 0);
        for (int round = 0; round < rounds; ++round)
          for (int g = 0; g < kNumGroups2; ++g) {
            const int n = g2_feat(g) ? 9 : 8;
            for (int i = 0; i < n; ++i) {
              mbar_wait_fast(bars_u + cur.st * 8, cur.par);
              mbar_arrive_remote(leader_w_full + cur.st * 8);
              cur = ring_at(cur, 1u);
            }
          }
      }
    }
    __syncwarp();
  } else if (warp >= 10) {
    // ============================ IPE warps: feature slabs of the slot's next ray -> global scratch ====
    const int slot = warp - 10;
    for (int round = 0; round < rounds; ++round) {
      const int64_t tile = tile_of(round, slot);
      const int64_t ray = tile < p.num_rays ? tile : p.num_rays - 1;
      // run at most one ray ahead: start once the previous ray's group 6 has consumed its feature stages
      // (keeps the single-count f_ready barrier from seeing two arrivals in one producer wait)
      if (round >= 1) mbar_wait(&f_free[slot], (uint32_t)((round - 1) & 1));
      uint8_t* dst = my_scratch + (slot * 2 + (round & 1)) * kFeatSlotBytes;
      const RayGeom g = load_ray_geom(p.origins, p.directions, p.radii, ray);
#pragma unroll 1
      for (int i = 0; i < 4; ++i) {
        const int row = i * 32 + lane;
        const float t0 = __ldg(p.t + ray * (kN + 1) + row), t1 = __ldg(p.t + ray * (kN + 1) + row + 1);
        float mean[3], cov[3], tm, tv, rv;
        frustum_moments(t0, t1, g.radius_sq, tm, tv, rv);
        lift_gaussian(g, tm, tv, rv, mean, cov);
        if (p.disable_integration) cov[0] = cov[1] = cov[2] = 0.f;
#pragma unroll
        for (int gi = 0; gi < 6; ++gi) {
          float fsin[8], fcos[8];
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int f = gi * 8 + e;  // feature index = degree*3 + coord   (models/mip.py:335-341)
            ipe_pair<true>(mean[f % 3], cov[f % 3], f / 3, fsin[e], fcos[e]);
          }
          const int ks = gi * 8, kc = 48 + gi * 8;  // K of the sin / cos halves
          store8<kFmt>(dst + (ks >> 5) * kWStage + sw64_offset(row, ks & 31), fsin);
          store8<kFmt>(dst + (kc >> 5) * kWStage + sw64_offset(row, kc & 31), fcos);
        }
      }
      __threadfence();                                     // slabs visible device-wide ...
      asm volatile("fence.proxy.async;" ::: "memory");      // ... and to the TMA engine (async proxy)
      __syncwarp();
      if (lane == 0) mbar_arrive(&f_ready[slot]);
    }
  } else {
    // ============================ slot workers (as in v1; 10 accumulator hand-offs per ray) ============
    const int slot = (warp - 2) >> 2;
    const int q = warp & 3;
    const int row = q * 32 + lane;
    uint8_t* myA = sA + slot * kABytes;
    const uint32_t t_acc = tmem_base + ((uint32_t)(q * 32) << 16) + slot * 256;
    uint32_t ph_acc = 0;
#ifdef MIPNERF_TC_TRACE
    Tracer tracer;
    if (q == 0 && lane == 0) tracer.init(2 + slot);
#endif
    const uint32_t a_ready_leader = mapa_u32(smem_u32(&a_ready[slot]), 0);
    auto arrive_a_ready = [&]() {
      __syncwarp();
      if (lane == 0) mbar_arrive_remote(a_ready_leader);
    };
    arrive_a_ready();
    for (int round = 0; round < rounds; ++round) {
      const int64_t tile = tile_of(round, slot);
      const bool valid = tile < p.num_rays;
      const int64_t ray = valid ? tile : p.num_rays - 1;
      const float t0 = __ldg(p.t + ray * (kN + 1) + row), t1 = __ldg(p.t + ray * (kN + 1) + row + 1);
      float dnorm;
      {
        const float dx = __ldg(p.directions + ray * 3), dy = __ldg(p.directions + ray * 3 + 1),
                    dz = __ldg(p.directions + ray * 3 + 2);
        dnorm = sqrtf(dx * dx + dy * dy + dz * dz);
      }
      vb_s[slot * 128 + row] = __ldg(p.view_bias + ray * kCond + row);
      TRACE(EV(2, 0, 0, slot));
      float dens = 0.f, rgb0 = 0.f, rgb1 = 0.f, rgb2 = 0.f;
      for (int l = 0; l < kNumLayers; ++l) {
        mbar_wait(&acc_full[slot], ph_acc);
        ph_acc ^= 1;
        tc_fence_after();
        TRACE(EV(2, 2, l, slot));
        if (l < 9) {
          switch (l) {
            case 0: epilogue_trunk<kFmt, 0, false>(t_acc, myA, row, dens); break;
            case 1: epilogue_trunk<kFmt, 1, false>(t_acc, myA, row, dens); break;
            case 2: epilogue_trunk<kFmt, 2, false>(t_acc, myA, row, dens); break;
            case 3: epilogue_trunk<kFmt, 3, false>(t_acc, myA, row, dens); break;
            case 4: epilogue_trunk<kFmt, 4, false>(t_acc, myA, row, dens); break;
            case 5: epilogue_trunk<kFmt, 5, false>(t_acc, myA, row, dens); break;
            case 6: epilogue_trunk<kFmt, 6, false>(t_acc, myA, row, dens); break;
            case 7: epilogue_trunk<kFmt, 7, false>(t_acc, myA, row, dens); break;
            default: epilogue_trunk<kFmt, 8, false>(t_acc, myA, row, dens); break;
          }
          TRACE(EV(2, 3, l, slot));
          fence_proxy_async_smem();
          tc_fence_before();
          arrive_a_ready();
          TRACE(EV(2, 4, l, slot));
        } else {
          named_bar_sync(1 + slot, 128);
          epilogue_view<kFmt>(t_acc, vb_s + slot * 128, rgb0, rgb1, rgb2);
          tc_fence_before();
          arrive_a_ready();
          TRACE(EV(2, 3, l, slot));
        }
      }
      const float density = density_activation(dens + c_small.b_density, p.density_bias);
      const float cr = rgb_activation(rgb0 + c_small.b_color[0], p.rgb_scale, p.rgb_padding);
      const float cg = rgb_activation(rgb1 + c_small.b_color[1], p.rgb_scale, p.rgb_padding);
      const float cb = rgb_activation(rgb2 + c_small.b_color[2], p.rgb_scale, p.rgb_padding);
      const float dd = density * ((t1 - t0) * dnorm);
      float incl = dd;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const float n = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += n;
      }
      float excl = __shfl_up_sync(0xffffffffu, incl, 1);
      if (lane == 0) excl = 0.f;
      if (lane == 31) cs[slot * 4 + q] = incl;
      named_bar_sync(1 + slot, 128);
      float before = 0.f;
      for (int qq = 0; qq < q; ++qq) before += cs[slot * 4 + qq];
      const float w = -expm1f(-dd) * expf(-(before + excl));
      if (valid) p.weights[ray * kN + row] = w;
      float pr = warp_sum(w * cr), pg = warp_sum(w * cg), pb = warp_sum(w * cb), pw = warp_sum(w),
            pd = warp_sum(w * (0.5f * (t0 + t1)));
      if (lane == 0) {
        float* dst = ps + (slot * 4 + q) * 8;
        dst[0] = pr, dst[1] = pg, dst[2] = pb, dst[3] = pw, dst[4] = pd;
      }
      named_bar_sync(1 + slot, 128);
      TRACE(EV(2, 5, 0, slot));
      if (row == 0 && valid) {
        float s[5] = {0.f, 0.f, 0.f, 0.f, 0.f};
        for (int qq = 0; qq < 4; ++qq)
          for (int k = 0; k < 5; ++k) s[k] += ps[(slot * 4 + qq) * 8 + k];
        const float t_first = __ldg(p.t + ray * (kN + 1)), t_last = __ldg(p.t + ray * (kN + 1) + kN);
        float d = s[4];
        if (isnan(d)) d = 0.f;
        else if (isinf(d)) d = d > 0 ? 3.4028234663852886e38f : -3.4028234663852886e38f;
        d = fminf(fmaxf(d, t_first), t_last);
        const float bg = p.white_bkgd ? 1.0f - s[3] : 0.f;
        p.comp_rgb[ray * 3 + 0] = s[0] + bg;
        p.comp_rgb[ray * 3 + 1] = s[1] + bg;
        p.comp_rgb[ray * 3 + 2] = s[2] + bg;
        p.distance[ray] = d;
        p.acc[ray] = s[3];
      }
      named_bar_sync(1 + slot, 128);
    }
#ifdef MIPNERF_TC_TRACE
    if (q == 0 && lane == 0) tracer.finish(2 + slot);
#endif
  }
  tc_fence_before();
  __syncthreads();
  cluster_sync_all();
  if (warp == 0) tmem_dealloc_pair(tmem_base, 512);
}

#include "mlp_tc_v3.cuh"

// view-direction term of the view layer as a per-ray bias: vb[r][n] = b[n] + W[n][256:283] . pos_enc(viewdir[r])
// (models/mip.py:353-363 + the `cat([bottleneck, viewenc])` half of view_layers.0, models/mip_nerf.py:106-108).
// Block = 128 threads (thread n = output n keeps its 27 weights in registers) x 16 rays whose 27-wide
// encodings are computed once into shared memory.
//
// The same launch ("ray prologue") also writes the coarse fenceposts of level 0 (models/mip.py:143-160):
// blocks past the view-bias range each produce kCoarsePerBlock values of t[B,129].  One launch instead
// of two in front of the level-0 kernel.
constexpr int kVbRays = 16;
constexpr int kCoarsePerBlock = 8 * kCond;
__global__ void __launch_bounds__(kCond) ray_prologue_kernel(const float* __restrict__ viewdirs,
                                                             const float* __restrict__ w, const float* __restrict__ b,
                                                             float* __restrict__ out, int64_t num_rays,
                                                             unsigned vb_blocks, const float* __restrict__ near,
                                                             const float* __restrict__ far, const Draws t_rand,
                                                             float* __restrict__ t_out, int disparity) {
  __shared__ float venc[kVbRays][kViewDim + 1];
  const int n = threadIdx.x;
  if (blockIdx.x >= vb_blocks) {
    const int64_t base = (int64_t)(blockIdx.x - vb_blocks) * kCoarsePerBlock, total = num_rays * (kN + 1);
#pragma unroll 1
    for (int i = 0; i < kCoarsePerBlock / kCond; ++i) {
      const int64_t idx = base + i * kCond + n;
      if (idx >= total) return;
      const int64_t ray = idx / (kN + 1);
      const int j = (int)(idx % (kN + 1));
      const bool jit = draws_active(t_rand);
      t_out[idx] = coarse_fencepost(__ldg(near + ray), __ldg(far + ray), j, kN, disparity, jit,
                                    jit ? draw_uniform(t_rand, ray, j, kN + 1) : 0.f);
    }
    return;
  }
  const int64_t ray0 = (int64_t)blockIdx.x * kVbRays;
  for (int idx = n; idx < kVbRays * kViewDim; idx += kCond) {
    const int r = idx / kViewDim, f = idx % kViewDim;
    const int64_t ray = ray0 + r < num_rays ? ray0 + r : num_rays - 1;
    float v;
    if (f < 3) {
      v = __ldg(viewdirs + ray * 3 + f);  // append_identity
    } else {
      const int g = f - 3, is_cos = g >= 12, h = is_cos ? g - 12 : g;  // scale-major, then xyz
      const float y = __fmul_rn(__ldg(viewdirs + ray * 3 + h % 3), __int_as_float((127 + h / 3) << 23));
      v = sinf(is_cos ? __fadd_rn(y, MIPNERF_HALF_PI_F32) : y);
    }
    venc[r][f] = v;
  }
  float wr[kViewDim];
#pragma unroll
  for (int k = 0; k < kViewDim; ++k) wr[k] = __ldg(w + (size_t)n * (kWidth + kViewDim) + kWidth + k);
  const float bias = __ldg(b + n);
  __syncthreads();
#pragma unroll 4
  for (int r = 0; r < kVbRays; ++r) {
    if (ray0 + r >= num_rays) break;
    float acc = bias;
#pragma unroll
    for (int k = 0; k < kViewDim; ++k) acc = fmaf(wr[k], venc[r][k], acc);
    out[(ray0 + r) * kCond + n] = acc;
  }
}

// MLP-only mode: same per-ray bias from a caller-supplied [B,27] view encoding
__global__ void view_bias_from_enc_kernel(const float* __restrict__ venc, const float* __restrict__ w,
                                          const float* __restrict__ b, float* __restrict__ out, int64_t num_rays) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= num_rays * kCond) return;
  const int64_t ray = idx / kCond;
  const int n = (int)(idx % kCond);
  float acc = __ldg(b + n);
#pragma unroll
  for (int k = 0; k < kViewDim; ++k)
    acc = fmaf(__ldg(w + (size_t)n * (kWidth + kViewDim) + kWidth + k), __ldg(venc + ray * kViewDim + k), acc);
  out[idx] = acc;
}

// ---- weight packing ---------------------------------------------------------------------------
// lo != 0: the low half  fl16(w - fl16(w))  of the split-operand modes instead of fl16(w)
template <int kFmt>
__global__ void pack_stage_kernel(const float* __restrict__ w, int in_features, int row0, int kbase, int kcount,
                                  uint8_t* __restrict__ dst, int nrows, int lo) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= nrows * kcount) return;
  const int i = idx / kcount, j = idx % kcount;
  float v = w[(size_t)(row0 + i) * in_features + kbase + j];
  if (lo) v = v - from16<kFmt>(to16<kFmt>(v));
  const uint32_t off = kcount == 64 ? sw128_offset(i, j) : sw64_offset(i, j);
  *reinterpret_cast<uint16_t*>(dst + off) = to16<kFmt>(v);
}

// All stages of one (hi or lo) v1 image in ONE launch: block = stage.  Main stages: layer l, N-half h, K-slab s of 32
// (K order of layer 5 is the reference's concat [h (256) | x (96)], mip_nerf.py:96-97) -> [128 x 64 B] SW64; then the
// 16 stages of the pair-mode view layer (two 64-row halves x 8 slabs).
struct PackV1Src {
  const float* weight[kNumLayers];
  int in_features[kNumLayers];
};
__host__ __device__ constexpr int v1_stage_begin(int l) {
  int n = 0;
  for (int i = 0; i < l; ++i) n += num_halves(i) * num_k32(i);
  return n;
}
constexpr int kV1MainStages = v1_stage_begin(kNumLayers);
template <int kFmt>
__global__ void __launch_bounds__(256) pack_v1_image_kernel(const PackV1Src src, uint8_t* __restrict__ base, int lo) {
  const int stage = blockIdx.x;
  const float* w;
  int in_features, row0, kbase, nrows;
  uint8_t* dst;
  if (stage < kV1MainStages) {
    int l = 0;
    while (l + 1 < kNumLayers && stage >= v1_stage_begin(l + 1)) ++l;
    const int local = stage - v1_stage_begin(l);
    const int h = local / num_k32(l), sl = local % num_k32(l);
    w = src.weight[l], in_features = src.in_features[l], row0 = h * 128, kbase = sl * 32, nrows = 128;
    dst = base + layer_offset(l) + (size_t)local * kWStage;
  } else {
    const int local = stage - kV1MainStages;
    w = src.weight[kNumLayers - 1], in_features = src.in_features[kNumLayers - 1];
    row0 = (local >> 3) * 64, kbase = (local & 7) * 32, nrows = 64;
    dst = base + kViewPairOffset + (size_t)local * kViewPairStage;
  }
  for (int idx = threadIdx.x; idx < nrows * 32; idx += 256) {
    const int i = idx >> 5, j = idx & 31;
    float v = w[(size_t)(row0 + i) * in_features + kbase + j];
    if (lo) v = v - from16<kFmt>(to16<kFmt>(v));
    *reinterpret_cast<uint16_t*>(dst + sw64_offset(i, j)) = to16<kFmt>(v);
  }
}

// dst [rows, in_dst] <- src [rows, in_src]: the first `prefix` columns copied; the rest is two halves (sin | shifted sin)
// of half_dst columns each, of which the model has the first half_src (lower encoding degrees); the others are zero
__global__ void expand_encoding_columns_kernel(const float* __restrict__ src, int in_src, float* __restrict__ dst,
                                               int in_dst, int rows, int prefix, int half_src, int half_dst) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * in_dst) return;
  const int r = idx / in_dst, c = idx % in_dst;
  float v = 0.f;
  if (c < prefix) {
    v = src[(size_t)r * in_src + c];
  } else {
    const int j = c - prefix, h = j / half_dst, i = j % half_dst;
    if (h < 2 && i < half_src) v = src[(size_t)r * in_src + prefix + h * half_src + i];
  }
  dst[idx] = v;
}

struct SmallSrc {
  const float* bias[9];
  const float* w_density;
  const float* b_density;
  const float* w_color;
  const float* b_color;
};
__global__ void pack_small_params_kernel(const SmallSrc src, SmallParams* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < 9 * kWidth) out->bias[i / kWidth][i % kWidth] = src.bias[i / kWidth][i % kWidth];
  if (i < kWidth) out->w_density[i] = src.w_density[i];
  if (i < 3 * kCond) out->w_color[i / kCond][i % kCond] = src.w_color[i];
  if (i == 0) out->b_density = src.b_density[0];
  if (i < 3) out->b_color[i] = src.b_color[i];
}

__global__ void pack_view_dir_kernel(const float* __restrict__ w, const float* __restrict__ b,
                                     float* __restrict__ out) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < kViewDim * kCond) {
    const int k = i / kCond, n = i % kCond;
    out[i] = w[(size_t)n * (kWidth + kViewDim) + kWidth + k];
  } else if (i < (kViewDim + 1) * kCond) {
    out[i] = b[i - kViewDim * kCond];
  }
}

// c_small is ONE constant bank per device, while the ABI lets callers run forwards of different models on different
// streams.  SmallUpload serialises those users: it holds a host lock for the duration of the enqueue, makes the
// stream wait for the previous user's kernels (on another stream) before overwriting the bank, and records an event
// after this call's launches.  Same-stream callers (the normal case) pay one event record.  During stream capture the
// cross-stream wait is skipped (a capture is single-stream by construction and the event lives outside the graph).
constexpr int kMaxDevices = 64;
struct SmallBankState {
  cudaEvent_t done = nullptr;
  cudaStream_t last = nullptr;
  bool used = false;
};
std::mutex g_small_mu;
SmallBankState g_small_state[kMaxDevices];

class SmallUpload {
 public:
  SmallUpload(const uint8_t* img, cudaStream_t st) : lock_(g_small_mu), st_(st) {
    int dev = 0;
    cudaGetDevice(&dev);
    state_ = &g_small_state[dev % kMaxDevices];
    cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
    if (cudaStreamIsCapturing(st, &cap) != cudaSuccess) cap = cudaStreamCaptureStatusNone;
    capturing_ = cap != cudaStreamCaptureStatusNone;
    if (!capturing_ && state_->used && state_->last != st) {
      err_ = cudaStreamWaitEvent(st, state_->done, 0);
      if (err_ != cudaSuccess) return;
    }
    err_ = cudaMemcpyToSymbolAsync(c_small, img + kSmallOffset, sizeof(SmallParams), 0, cudaMemcpyDeviceToDevice, st);
  }
  cudaError_t error() const { return err_; }
  ~SmallUpload() {
    if (capturing_ || err_ != cudaSuccess) return;
    if (!state_->done && cudaEventCreateWithFlags(&state_->done, cudaEventDisableTiming) != cudaSuccess) return;
    if (cudaEventRecord(state_->done, st_) == cudaSuccess) {
      state_->last = st_;
      state_->used = true;
    }
  }

 private:
  std::lock_guard<std::mutex> lock_;
  cudaStream_t st_;
  SmallBankState* state_ = nullptr;
  bool capturing_ = false;
  cudaError_t err_ = cudaSuccess;
};

struct TcScratch {
  float *vbias, *t[2], *w[2];
  uint8_t* feat;  // v2 kernel: kMaxCtas2 x kFeatScratchPerCta
  size_t bytes;
};
constexpr int64_t kChunkRaysTc = 65536;

inline size_t align_up(size_t v, size_t a = 256) { return (v + a - 1) / a * a; }

TcScratch carve_tc(int64_t rays, void* base) {
  TcScratch s{};
  size_t off = 0;
  auto take = [&](size_t elems) {
    float* p = base ? reinterpret_cast<float*>(static_cast<char*>(base) + off) : nullptr;
    off += align_up(elems * sizeof(float));
    return p;
  };
  s.vbias = take((size_t)rays * kCond);
  for (int i = 0; i < 2; ++i) {
    s.t[i] = take((size_t)rays * (kN + 1));
    s.w[i] = take((size_t)rays * kN);
  }
  s.feat = reinterpret_cast<uint8_t*>(take((size_t)kMaxCtas2 * kFeatScratchPerCta / sizeof(float)));
  s.bytes = off;
  return s;
}

int g_num_sms = 0;
bool g_attr_set[2][2][2] = {};

// operand format (0 fp16, 1 bf16) and split flag of a tensor-core precision
inline int fmt_of(int precision) { return (precision == MIPNERF_B200_BF16 || precision == MIPNERF_B200_BF16X3) ? 1 : 0; }
inline bool is_x3(int precision) { return precision == MIPNERF_B200_FP16X3 || precision == MIPNERF_B200_BF16X3; }

template <int kFmt, bool kPair, bool kX3 = false, bool kTrain = false, bool kTS = false, bool kNoise = false>
cudaError_t launch_level_t(const LevelParams& p, cudaStream_t st) {
  auto kern = mlp_level_kernel<kFmt, kPair, kX3, kTrain, kTS, kNoise>;
  static bool attr_set = false;  // one flag per instantiation
  if (!attr_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemTotal);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  if (g_num_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
  }
  LevelParams q = p;
  LaunchScope scope(p.feat_in ? kKernMlpTc : kKernMlpLevelTc, st);
  if (kPair) {
    constexpr int64_t kPerPair = kX3 ? 2 : 4;  // rays a CTA pair holds at a time (slots x 2 CTAs)
    const int64_t quads = (p.num_rays + kPerPair - 1) / kPerPair;
    const int pairs = (int)(quads < g_num_sms / 2 ? quads : g_num_sms / 2);
    q.rounds = (int)((p.num_rays + kPerPair * (int64_t)pairs - 1) / (kPerPair * (int64_t)pairs));
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(2 * pairs);
    cfg.blockDim = dim3(kThreads);
    cfg.dynamicSmemBytes = kSmemTotal;
    cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = 2;
    attr[0].val.clusterDim.y = 1;
    attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kern, q);
  }
  const int64_t pairs = (p.num_rays + 1) / 2;
  const int grid = (int)(pairs < g_num_sms ? pairs : g_num_sms);
  q.rounds = (int)((p.num_rays + 2 * (int64_t)grid - 1) / (2 * (int64_t)grid));
  kern<<<grid, kThreads, kSmemTotal, st>>>(q);
  return cudaGetLastError();
}

bool g_attr_set2[2] = {false, false};

template <int kFmt>
cudaError_t launch_level_v2(const LevelParams& p, cudaStream_t st) {
  auto kern = mlp_level_kernel_v2<kFmt>;
  if (!g_attr_set2[kFmt]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemTotal2);
    if (e != cudaSuccess) return e;
    g_attr_set2[kFmt] = true;
  }
  if (g_num_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
  }
  LevelParams q = p;
  LaunchScope scope(kKernMlpLevelTc, st);
  const int64_t quads = (p.num_rays + 3) / 4;
  int max_pairs = g_num_sms / 2;
  if (max_pairs > kMaxCtas2 / 2) max_pairs = kMaxCtas2 / 2;
  const int pairs = (int)(quads < max_pairs ? quads : max_pairs);
  q.rounds = (int)((p.num_rays + 4 * (int64_t)pairs - 1) / (4 * (int64_t)pairs));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(2 * pairs);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = kSmemTotal2;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, q);
}

bool g_attr_set3[2] = {false, false};

template <int kFmt>
cudaError_t launch_level_v3(const LevelParams& p, cudaStream_t st) {
  auto kern = mlp_level_kernel_v3<kFmt>;
  if (!g_attr_set3[kFmt]) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemTotal3);
    if (e != cudaSuccess) return e;
    g_attr_set3[kFmt] = true;
  }
  if (g_num_sms == 0) {
    int dev = 0;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev);
  }
  LevelParams q = p;
  LaunchScope scope(p.feat_in ? kKernMlpTc : kKernMlpLevelTc, st);
  const int64_t duos = (p.num_rays + 1) / 2;  // a CTA pair holds 2 rays at a time
  const int pairs = (int)(duos < g_num_sms / 2 ? duos : g_num_sms / 2);
  q.rounds = (int)((p.num_rays + 2 * (int64_t)pairs - 1) / (2 * (int64_t)pairs));
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = dim3(2 * pairs);
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = kSmemTotal3;
  cfg.stream = st;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = 2;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, q);
}

// MIPNERF_B200_TC_VARIANT: "v3" = activations in tensor memory, one ray per CTA (mlp_tc_v3.cuh), "shared" = CTA pair +
// shared weight stream (v2), "pair" = CTA pair (v1), "single" = 1-CTA kernel (cta_group::1).
int tc_variant() {
  const char* v = getenv("MIPNERF_B200_TC_VARIANT");
  if (v && v[0] == 'v' && v[1] == '4') return 4;
  if (v && v[0] == 'v' && v[1] == '3') return 3;
  if (v && v[0] == 's' && v[1] == 'i') return 0;
  if (v && v[0] == 's' && v[1] == 'h') return 2;
  if (v && v[0] == 'p') return 1;
  return MIPNERF_TC_DEFAULT_VARIANT;
}
bool use_pair_variant() { return tc_variant() != 0; }
// MIPNERF_B200_TC_PROLOGUE=separate keeps the ray prologue / resampler as their own launches (A/B measurements);
// default: produced inside the v1 level kernels.
bool fused_prologue_enabled(int precision) {
  const char* v = getenv("MIPNERF_B200_TC_PROLOGUE");
  return (is_x3(precision) || tc_variant() < 2 || tc_variant() == 4) && !(v && v[0] == 's');
}

cudaError_t launch_level(const LevelParams& p, int precision, cudaStream_t st) {
  if (p.act_dump)  // training forward: the CTA-pair kernel with the activation dump
    return precision == MIPNERF_B200_BF16 ? launch_level_t<1, true, false, true>(p, st)
                                          : launch_level_t<0, true, false, true>(p, st);
  if (draws_active(p.dnoise)) {  // density noise (randomized, density_noise > 0): the v1 CTA-pair kernels' kNoise build
    if (is_x3(precision))
      return fmt_of(precision) ? launch_level_t<1, true, true, false, false, true>(p, st)
                               : launch_level_t<0, true, true, false, false, true>(p, st);
    return precision == MIPNERF_B200_BF16 ? launch_level_t<1, true, false, false, false, true>(p, st)
                                          : launch_level_t<0, true, false, false, false, true>(p, st);
  }
  if (is_x3(precision))  // split-operand parity modes: the CTA-pair kernel, whatever variant is selected
    return fmt_of(precision) ? launch_level_t<1, true, true>(p, st) : launch_level_t<0, true, true>(p, st);
  if (tc_variant() == 4)  // "v4": the CTA-pair kernel with the activations in tensor memory (TS-form MMAs)
    return precision == MIPNERF_B200_BF16 ? launch_level_t<1, true, false, false, true>(p, st)
                                          : launch_level_t<0, true, false, false, true>(p, st);
  if (tc_variant() == 3)
    return precision == MIPNERF_B200_BF16 ? launch_level_v3<1>(p, st) : launch_level_v3<0>(p, st);
  if (tc_variant() == 2)
    return precision == MIPNERF_B200_BF16 ? launch_level_v2<1>(p, st) : launch_level_v2<0>(p, st);
  const bool pair = use_pair_variant();
  if (precision == MIPNERF_B200_BF16)
    return pair ? launch_level_t<1, true>(p, st) : launch_level_t<1, false>(p, st);
  return pair ? launch_level_t<0, true>(p, st) : launch_level_t<0, false>(p, st);
}

}  // namespace

#ifdef MIPNERF_TC_TRACE
int set_trace_ptr(unsigned long long* ptr);
}  // namespace mipnerf
extern "C" int mipnerf_b200_debug_set_trace_buffer(void* dev_ptr) {
  unsigned long long* ptr = static_cast<unsigned long long*>(dev_ptr);
  return mipnerf::set_trace_ptr(ptr);
}
namespace mipnerf {
int set_trace_ptr(unsigned long long* ptr) {
  return cudaMemcpyToSymbol(g_trace, &ptr, sizeof(ptr)) == cudaSuccess ? 0 : -3;
}
#endif

// Encoding degrees below the kernels' own (max_deg_point < 16, deg_view < 4; min_deg_point = 0): the level kernels always
// compute the 96 IPE features of degrees 0..15 and the 27 view features of degrees 0..3, and the MODEL's narrower
// layers.0 / layers.5 / view_layers.0 weights are zero-padded to those widths when the operand image is packed (feature
// column 3 l + c of the sin half and 48 + 3 l + c of the shifted-sin half <- the model's columns 3 l + c and
// 3 L + 3 l + c; models/mip.py:322-341, :353-363).  The extra features meet exact zeros in the GEMM, so the result is the
// narrower model's, at the default model's speed.
bool tc_default_degrees(const mipnerf_b200_config* c) { return c->max_deg_point == 16 && c->deg_view == 4; }
bool tc_supported(const mipnerf_b200_config* c, int precision) {
  return (precision == MIPNERF_B200_BF16 || precision == MIPNERF_B200_FP16 || is_x3(precision)) &&
         c->num_samples == kN &&
         c->min_deg_point == 0 && c->max_deg_point >= 1 && c->max_deg_point <= 16 && c->deg_view >= 1 &&
         c->deg_view <= 4 && c->use_viewdirs &&
         c->net_depth == 8 && c->net_width == kWidth && c->net_depth_condition == 1 &&
         c->net_width_condition == kCond && c->skip_index == 4 && c->num_rgb_channels == 3 &&
         c->num_density_channels == 1;
}
bool tc_mlp_supported(const mipnerf_b200_config* c, int samples_per_ray, int precision) {
  mipnerf_b200_config c2 = *c;
  c2.num_samples = kN;  // MLP-only mode takes the caller's [B,128,96] / [B,27] encodings as they are: default degrees only
  return samples_per_ray == kN && tc_default_degrees(c) && tc_supported(&c2, precision);
}

// zero-padded fp32 copies of layers.0 [256,96], layers.5 [256,352], view_layers.0 [128,283] behind the operand image
constexpr size_t kPad0Bytes = (size_t)kWidth * kFeat * sizeof(float);
constexpr size_t kPad5Bytes = (size_t)kWidth * (kWidth + kFeat) * sizeof(float);
constexpr size_t kPadViewBytes = (size_t)kCond * (kWidth + kViewDim) * sizeof(float);
constexpr size_t kPadOffset = (kV3Offset + kV3Bytes + 255) / 256 * 256;
constexpr size_t kPadBytes = kPad0Bytes + kPad5Bytes + kPadViewBytes;

size_t tc_packed_bytes(const mipnerf_b200_config* c, int precision) {
  if (!tc_supported(c, precision)) return 0;
  return tc_default_degrees(c) ? kV3Offset + kV3Bytes : kPadOffset + kPadBytes;
}

size_t tc_workspace_bytes(const mipnerf_b200_config* c, int64_t num_rays, int precision) {
  if (!tc_supported(c, precision)) return 0;
  const int64_t r = num_rays < kChunkRaysTc ? num_rays : kChunkRaysTc;
  return carve_tc(r > 0 ? r : 1, nullptr).bytes;
}

cudaError_t tc_pack_weights(const mipnerf_b200_config* c, const mipnerf_b200_weights* w, int precision,
                            void* packed_out, cudaStream_t st, bool with_v3) {
  if (!tc_supported(c, precision)) return cudaErrorNotSupported;
  uint8_t* img = static_cast<uint8_t*>(packed_out);
  const bool bf = fmt_of(precision) == 1;
  const int parts = is_x3(precision) ? 2 : 1;  // hi image, then (split modes) the lo stage image
  cudaError_t e = cudaMemsetAsync(img, 0, with_v3 ? kV3Offset + kV3Bytes : kV3Offset, st);
  if (e != cudaSuccess) return e;
  LaunchScope scope(kKernPackWeights, st);
  mipnerf_b200_linear lin[12];
  for (int i = 0; i < 12; ++i) lin[i] = w->linears[i];
  if (!tc_default_degrees(c)) {  // lower encoding degrees: pack from zero-padded copies of the three encoding-fed layers
    float* pad0 = reinterpret_cast<float*>(img + kPadOffset);
    float* pad5 = reinterpret_cast<float*>(img + kPadOffset + kPad0Bytes);
    float* padv = reinterpret_cast<float*>(img + kPadOffset + kPad0Bytes + kPad5Bytes);
    const int hx = 3 * c->max_deg_point, hv = 3 * c->deg_view;
    auto expand = [&](int li, float* dst, int in_dst, int rows, int prefix, int half_src, int half_dst) {
      expand_encoding_columns_kernel<<<(rows * in_dst + 255) / 256, 256, 0, st>>>(lin[li].weight, lin[li].in_features, dst,
                                                                                  in_dst, rows, prefix, half_src, half_dst);
      lin[li].weight = dst, lin[li].in_features = in_dst;
    };
    expand(0, pad0, kFeat, kWidth, 0, hx, kFeat / 2);
    expand(5, pad5, kWidth + kFeat, kWidth, kWidth, hx, kFeat / 2);
    expand(10, padv, kWidth + kViewDim, kCond, kWidth + 3, hv, (kViewDim - 3) / 2);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  PackV1Src v1{};
  for (int l = 0; l < kNumLayers; ++l) {
    const int li = l < 8 ? l : (l == 8 ? 9 : 10);  // layers.l | extra_layer | view_layers.0
    v1.weight[l] = lin[li].weight, v1.in_features[l] = lin[li].in_features;
  }
  for (int part = 0; part < parts; ++part) {
    uint8_t* base = img + (part ? kLoOffset : 0);
    if (bf) pack_v1_image_kernel<1><<<kV1MainStages + 16, 256, 0, st>>>(v1, base, part);
    else pack_v1_image_kernel<0><<<kV1MainStages + 16, 256, 0, st>>>(v1, base, part);
  }
  // v3 blocks: per layer, per CTA rank, in the kernel's issue order (mlp_tc_v3.cuh: Sched3); the training step
  // repacks every optimiser step and runs the v1 pair kernel only, so it skips them
  for (int l = 0; with_v3 && l < kNumLayers; ++l) {
    const int li = l < 8 ? l : (l == 8 ? 9 : 10);
    const mipnerf_b200_linear& lin3 = lin[li];
    const int type = layer_type3(l), nb = sched_count3(type);
    const int fbase = l == 5 ? kWidth : 0;  // K offset of the feature columns: layer 5 is [h (256) | x (96)]
    for (int r = 0; r < 2; ++r) {
      uint8_t* dst = img + kV3Offset + layer_offset3(l) + (size_t)r * (layer_bytes3(l) / 2);
      for (int b = 0; b < nb; ++b, dst += kBlk3) {
        const Blk3 blk = kSched3Host.blk[type][b];
        const int row0 = 64 * blk.nq + 32 * r;
        const int kbase = blk.kind < 4 ? 64 * blk.kind : (blk.kind == 4 ? fbase : fbase + 64);
        const int kcount = blk.kind == 5 ? 32 : 64;
        if (bf)
          pack_stage_kernel<1><<<(32 * kcount + 255) / 256, 256, 0, st>>>(lin3.weight, lin3.in_features, row0, kbase, kcount,
                                                                         dst, 32, 0);
        else
          pack_stage_kernel<0><<<(32 * kcount + 255) / 256, 256, 0, st>>>(lin3.weight, lin3.in_features, row0, kbase, kcount,
                                                                         dst, 32, 0);
      }
    }
  }
  SmallSrc src;
  for (int l = 0; l < 8; ++l) src.bias[l] = lin[l].bias;
  src.bias[8] = lin[9].bias;  // extra_layer
  src.w_density = lin[8].weight;
  src.b_density = lin[8].bias;
  src.w_color = lin[11].weight;
  src.b_color = lin[11].bias;
  pack_small_params_kernel<<<(9 * kWidth + 255) / 256, 256, 0, st>>>(src,
                                                                      reinterpret_cast<SmallParams*>(img + kSmallOffset));
  pack_view_dir_kernel<<<((kViewDim + 1) * kCond + 255) / 256, 256, 0, st>>>(
      lin[10].weight, lin[10].bias, reinterpret_cast<float*>(img + kViewDirOffset));
  return cudaGetLastError();
}

// The uniforms of one launch: rows `off..` of the caller's array, or the in-kernel generator (stream 0 = t_rand,
// 1 + level = that level's u_jitter, scaled like uniform_(to = 1/ncols - eps), models/mip.py:201-202).
Draws level_draws(int randomized, const float* array, const mipnerf_b200_rng* rng, int64_t off, int stream, int ncols) {
  if (!randomized) return draws_from_array(nullptr);
  if (array) return draws_from_array(array + off * ncols);
  if (!rng) return draws_from_array(nullptr);
  const float scale = stream == 0 ? 1.0f : (float)(1.0 / (double)ncols) - MIPNERF_F32_EPS;
  return draws_philox(rng->seed, rng->offset, off, stream, scale);
}

// The density-noise normals of one launch of level `level` (models/mip_nerf.py:232-233): rows `off..` of the caller's
// [B,n] array, or the in-kernel generator (stream 32 + level); inactive unless randomized and density_noise > 0.
Draws density_noise_draws(const mipnerf_b200_config* c, int randomized, const float* normal, const mipnerf_b200_rng* rng,
                          int64_t off, int level, int n) {
  if (!randomized || !(c->density_noise > 0.f)) return draws_from_array(nullptr);
  Draws d = normal ? draws_from_array(normal + off * n)
                   : (rng ? draws_philox(rng->seed, rng->offset, off, kDensityNoiseStream + level, 1.f)
                          : draws_from_array(nullptr));
  d.scale = c->density_noise;
  return d;
}

cudaError_t tc_forward(const mipnerf_b200_config* c, const mipnerf_b200_weights* w, const mipnerf_b200_rays* rays,
                       int randomized, const float* t_rand, const float* u_jitter, const mipnerf_b200_rng* rng,
                       int white_bkgd, int precision, mipnerf_b200_level_out* outs, void* workspace,
                       size_t workspace_bytes, cudaStream_t st, const TcTrainDump* dump, int64_t ray_base) {
  const uint8_t* img = static_cast<const uint8_t*>(w->packed);
  SmallUpload small(img, st);  // biases / heads -> constant bank, ordered against other streams' forwards
  cudaError_t e = small.error();
  if (e != cudaSuccess) return e;
  const mipnerf_b200_linear& view = w->linears[10];
  const float rgb_scale = (float)(1.0 + 2.0 * (double)c->rgb_padding);
  for (int64_t off = 0; off < rays->num_rays; off += kChunkRaysTc) {
    const int64_t cnt = (rays->num_rays - off) < kChunkRaysTc ? (rays->num_rays - off) : kChunkRaysTc;
    const TcScratch s = carve_tc(cnt, workspace);
    if (s.bytes > workspace_bytes) return cudaErrorInvalidValue;
    const float* origins = rays->origins + off * 3;
    const float* directions = rays->directions + off * 3;
    const float* radii = rays->radii + off;
    // v1 kernels produce fenceposts and the view bias inside the level kernels (IPE warps); the shared-stream
    // variant keeps the separate prologue / resample launches.
    const bool fused_prologue = dump != nullptr || fused_prologue_enabled(precision);  // training: always the v1 pair kernel
    if (!fused_prologue && !tc_default_degrees(c)) return cudaErrorNotSupported;  // the stand-alone prologue reads the
                                                                                  // model's own (narrower) view layer
    // in-kernel Philox: the counter is the ray index of the caller's whole batch (ray_base = offset of `rays` in it)
    auto draws = [&](const float* array, int stream) {
      Draws d = level_draws(randomized, array, rng, off, stream, kN + 1);
      if (!array) d.ray_base += ray_base;
      return d;
    };
    if (!fused_prologue) {
      LaunchScope scope(kKernRayPrologue, st);
      float* t0 = outs[0].t_samples ? outs[0].t_samples + off * (kN + 1) : s.t[0];
      const unsigned vb_blocks = (unsigned)((cnt + kVbRays - 1) / kVbRays);
      const unsigned ct_blocks = (unsigned)((cnt * (kN + 1) + kCoarsePerBlock - 1) / kCoarsePerBlock);
      ray_prologue_kernel<<<vb_blocks + ct_blocks, kCond, 0, st>>>(
          rays->viewdirs + off * 3, view.weight, view.bias, s.vbias, cnt, vb_blocks, rays->near + off, rays->far + off,
          draws(t_rand, 0), t0, c->disparity);
      if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    const float *t_prev = nullptr, *w_prev = nullptr;
    for (int l = 0; l < c->num_levels; ++l) {
      float* t_cur = outs[l].t_samples ? outs[l].t_samples + off * (kN + 1) : s.t[l & 1];
      float* w_cur = outs[l].weights ? outs[l].weights + off * kN : s.w[l & 1];
      const Draws jit = draws(u_jitter, 1 + l);  // one stream per level
      int64_t* inds = outs[l].inds ? outs[l].inds + off * (kN + 1) : nullptr;
      if (l > 0 && !fused_prologue) {
        e = launch_resample(t_prev, w_prev, jit, t_cur, inds, cnt, kN, kN + 1, randomized, 1, c->resample_padding, st);
        if (e != cudaSuccess) return e;
      }
      LevelParams p{};
      p.wimage = img;
      p.origins = origins, p.directions = directions, p.radii = radii;
      p.t = t_cur;
      p.view_bias = s.vbias;
      if (fused_prologue) {
        p.t_mode = l == 0 ? 1 : 2;
        p.vb_mode = l == 0 ? 1 : 0;  // level 0 leaves the per-ray bias in s.vbias for the later levels
        p.near = rays->near + off, p.far = rays->far + off;
        p.t_rand = draws(t_rand, 0);
        p.disparity = c->disparity;
        p.t_prev = t_prev, p.w_prev = w_prev;
        p.u_jitter = jit;
        p.inds = inds;
        p.randomized = randomized;
        p.resample_padding = c->resample_padding;
        p.viewdirs = rays->viewdirs + off * 3;
      }
      p.feat_scratch = s.feat;
      if (dump) {  // training forward: one chunk only (the caller chunks), tile index = ray index
        p.act_dump = dump->act[l], p.v_dump = dump->v[l];
        p.raw_rgb_keep = dump->raw_rgb[l], p.raw_density_keep = dump->raw_density[l];
        p.dump_tiles = cnt;
      }
      p.comp_rgb = outs[l].comp_rgb + off * 3;
      p.distance = outs[l].distance + off;
      p.acc = outs[l].acc + off;
      p.weights = w_cur;
      p.num_rays = cnt;
      p.white_bkgd = white_bkgd;
      p.disable_integration = c->disable_integration;
      p.density_bias = c->density_bias, p.rgb_scale = rgb_scale, p.rgb_padding = c->rgb_padding;
      p.dnoise = density_noise_draws(c, randomized, outs[l].density_normal, rng, off, l, kN);
      if (!outs[l].density_normal) p.dnoise.ray_base += ray_base;
      p.rng_state = dump ? dump->rng_state : nullptr;
      e = launch_level(p, precision, st);
      if (e != cudaSuccess) return e;
      t_prev = t_cur;
      w_prev = w_cur;
    }
  }
  return cudaSuccess;
}

cudaError_t tc_mlp_forward(const mipnerf_b200_config* c, const mipnerf_b200_weights* w, const float* x,
                           const float* view_enc, int64_t num_rays, int precision, float* raw_rgb, float* raw_density,
                           void* workspace, cudaStream_t st) {
  (void)c;
  const uint8_t* img = static_cast<const uint8_t*>(w->packed);
  SmallUpload small(img, st);
  cudaError_t e = small.error();
  if (e != cudaSuccess) return e;
  float* vbias = static_cast<float*>(workspace);  // [num_rays, 128]
  const mipnerf_b200_linear& view = w->linears[10];
  {
    LaunchScope scope(kKernPosEnc, st);
    view_bias_from_enc_kernel<<<(unsigned)((num_rays * kCond + 255) / 256), 256, 0, st>>>(view_enc, view.weight,
                                                                                           view.bias, vbias, num_rays);
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
  }
  LevelParams p{};
  p.wimage = img;
  p.view_bias = vbias;
  p.feat_in = x;
  p.raw_rgb_out = raw_rgb;
  p.raw_density_out = raw_density;
  p.num_rays = num_rays;
  // MLP-only mode lives in the v1 kernels (CTA pair unless MIPNERF_B200_TC_VARIANT=single)
  if (is_x3(precision))
    return fmt_of(precision) ? launch_level_t<1, true, true>(p, st) : launch_level_t<0, true, true>(p, st);
  if (tc_variant() == 3) return precision == MIPNERF_B200_BF16 ? launch_level_v3<1>(p, st) : launch_level_v3<0>(p, st);
  const bool pair = tc_variant() != 0;
  if (precision == MIPNERF_B200_BF16) return pair ? launch_level_t<1, true>(p, st) : launch_level_t<1, false>(p, st);
  return pair ? launch_level_t<0, true>(p, st) : launch_level_t<0, false>(p, st);
}

cudaError_t launch_view_bias_from_enc(const float* venc, const float* w, const float* b, float* out,
                                      int64_t num_rays, cudaStream_t st) {
  if (num_rays == 0) return cudaSuccess;
  LaunchScope scope(kKernPosEnc, st);
  view_bias_from_enc_kernel<<<(unsigned)((num_rays * kCond + 255) / 256), 256, 0, st>>>(venc, w, b, out, num_rays);
  return cudaGetLastError();
}

size_t tc_mlp_workspace_bytes(int64_t num_rays) { return (size_t)(num_rays > 0 ? num_rays : 1) * kCond * sizeof(float); }

}  // namespace mipnerf
