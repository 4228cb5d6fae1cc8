// CUDA-core direct convolution (NHWC bf16, fp32 accumulate).
//
// Role: (1) the tiny-channel layers of the C3k interiors (C = 4/8/16) and the 3-channel
// stem, which cannot feed tcgen05 (N >= 16, K % 16 == 0); (2) the depth-wise 3x3 convs of
// the Detect cls branch; (3) the on-device cross-check for the tensor-core kernels.
// Arithmetic follows ConvBlock.forward (model.py:49-50) / Ultralytics Conv with BN folded:
//   out = [res +] relu(sum_{tap,ci} x * w + bias)
// One thread = one output pixel x CO_T output channels.
#include <type_traits>

#include "camera.cuh"
#include "common.cuh"
#include "stem_v2.cuh"

namespace uyd {

namespace {

constexpr int kThreads = 128;
constexpr size_t kSmemWeightLimit = 96 * 1024;

__device__ __forceinline__ float bf2f(__nv_bfloat16 v) { return __bfloat162float(v); }

template <int V>
struct Vec;
template <>
struct Vec<8> { using T = uint4; };
template <>
struct Vec<4> { using T = uint2; };

template <int V>
__device__ __forceinline__ void load_bf16(const __nv_bfloat16 *p, float (&x)[V]) {
  typename Vec<V>::T raw = *reinterpret_cast<const typename Vec<V>::T *>(p);
  const __nv_bfloat162 *h = reinterpret_cast<const __nv_bfloat162 *>(&raw);
#pragma unroll
  for (int i = 0; i < V / 2; ++i) {
    float2 f = __bfloat1622float2(h[i]);
    x[2 * i] = f.x;
    x[2 * i + 1] = f.y;
  }
}

// weights: bf16 [tap][ci][co]
template <int CO_T, int IN_VEC, bool W_SMEM>
__global__ void __launch_bounds__(kThreads) conv_direct_kernel(ConvArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const __nv_bfloat16 *wg = reinterpret_cast<const __nv_bfloat16 *>(a.w);
  const int taps = a.k * a.k;
  if (W_SMEM) {
    __nv_bfloat16 *ws = reinterpret_cast<__nv_bfloat16 *>(smem_raw);
    const int total = taps * a.cin * a.cout;
    for (int i = threadIdx.x; i < total; i += kThreads) ws[i] = wg[i];
    __syncthreads();
    wg = ws;
  }
  const long long npix = (long long)a.n * a.oh * a.ow;
  const long long p = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (p >= npix) return;
  const int co0 = blockIdx.y * CO_T;
  const int ox = (int)(p % a.ow);
  const int oy = (int)((p / a.ow) % a.oh);
  const int n = (int)(p / ((long long)a.ow * a.oh));
  const int pad = a.k / 2;

  float acc[CO_T];
#pragma unroll
  for (int i = 0; i < CO_T; ++i) acc[i] = 0.f;

  const __nv_bfloat16 *in = reinterpret_cast<const __nv_bfloat16 *>(a.in);
  for (int ky = 0; ky < a.k; ++ky) {
    const int iy = oy * a.stride + ky - pad;
    if (iy < 0 || iy >= a.ih) continue;
    for (int kx = 0; kx < a.k; ++kx) {
      const int ix = ox * a.stride + kx - pad;
      if (ix < 0 || ix >= a.iw) continue;
      const __nv_bfloat16 *px = in + (((long long)n * a.ih + iy) * a.iw + ix) * a.in_pitch;
      const __nv_bfloat16 *wt = wg + (size_t)(ky * a.k + kx) * a.cin * a.cout + co0;
      for (int ci = 0; ci < a.cin; ci += IN_VEC) {
        float x[IN_VEC];
        load_bf16<IN_VEC>(px + ci, x);
#pragma unroll
        for (int v = 0; v < IN_VEC; ++v) {
          const __nv_bfloat16 *wr = wt + (size_t)(ci + v) * a.cout;
          if (CO_T >= 8) {
#pragma unroll
            for (int c8 = 0; c8 < CO_T; c8 += 8) {
              float wv[8];
              load_bf16<8>(wr + c8, wv);
#pragma unroll
              for (int j = 0; j < 8; ++j) acc[c8 + j] = fmaf(x[v], wv[j], acc[c8 + j]);
            }
          } else {
            float wv[4];
            load_bf16<4>(wr, wv);
#pragma unroll
            for (int j = 0; j < 4; ++j) acc[j] = fmaf(x[v], wv[j], acc[j]);
          }
        }
      }
    }
  }

  const long long opix = ((long long)n * a.oh + oy) * a.ow + ox;
  float r[CO_T];
#pragma unroll
  for (int i = 0; i < CO_T; ++i) {
    float v = acc[i] + a.bias[co0 + i];
    if (a.relu) v = fmaxf(v, 0.f);
    r[i] = v;
  }
  if (a.res) {
    const __nv_bfloat16 *rp = reinterpret_cast<const __nv_bfloat16 *>(a.res) + opix * a.res_pitch + co0;
#pragma unroll
    for (int i = 0; i < CO_T; ++i) r[i] += bf2f(rp[i]);
  }
  if (a.out_f32) {
    float *op = reinterpret_cast<float *>(a.out) + opix * a.out_pitch + co0;
#pragma unroll
    for (int i = 0; i < CO_T; ++i) op[i] = r[i];
  } else {
    __nv_bfloat16 *op = reinterpret_cast<__nv_bfloat16 *>(a.out) + opix * a.out_pitch + co0;
    if (CO_T % 4 == 0 && (reinterpret_cast<uintptr_t>(op) & 7) == 0) {
#pragma unroll
      for (int i = 0; i < CO_T; i += 4) {
        __nv_bfloat162 lo = __floats2bfloat162_rn(r[i], r[i + 1]);
        __nv_bfloat162 hi = __floats2bfloat162_rn(r[i + 2], r[i + 3]);
        uint2 pk;
        pk.x = *reinterpret_cast<uint32_t *>(&lo);
        pk.y = *reinterpret_cast<uint32_t *>(&hi);
        *reinterpret_cast<uint2 *>(op + i) = pk;
      }
    } else {
#pragma unroll
      for (int i = 0; i < CO_T; ++i) op[i] = __float2bfloat16_rn(r[i]);
    }
  }
}

// Stem: network input NCHW fp32 (the reference forward signature), Cin = 3.
// weights bf16 [tap][ci][co]; one thread = one output pixel x CO_T channels.
template <int CO_T, typename TIn>
__global__ void __launch_bounds__(kThreads) conv_stem_nchw_kernel(ConvArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  __nv_bfloat16 *ws = reinterpret_cast<__nv_bfloat16 *>(smem_raw);
  const int total = a.k * a.k * a.cin * a.cout;
  for (int i = threadIdx.x; i < total; i += kThreads) ws[i] = reinterpret_cast<const __nv_bfloat16 *>(a.w)[i];
  __syncthreads();
  const long long npix = (long long)a.n * a.oh * a.ow;
  const long long p = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (p >= npix) return;
  const int co0 = blockIdx.y * CO_T;
  const int ox = (int)(p % a.ow);
  const int oy = (int)((p / a.ow) % a.oh);
  const int n = (int)(p / ((long long)a.ow * a.oh));
  const int pad = a.k / 2;
  const TIn *in = reinterpret_cast<const TIn *>(a.in);
  float acc[CO_T];
#pragma unroll
  for (int i = 0; i < CO_T; ++i) acc[i] = 0.f;
  for (int ky = 0; ky < a.k; ++ky) {
    const int iy = oy * a.stride + ky - pad;
    if (iy < 0 || iy >= a.ih) continue;
    for (int kx = 0; kx < a.k; ++kx) {
      const int ix = ox * a.stride + kx - pad;
      if (ix < 0 || ix >= a.iw) continue;
      for (int ci = 0; ci < a.cin; ++ci) {
        // the frame stays fp32 (fp32 x bf16-weight -> fp32): no input rounding at all.
        // uint8 frames are normalised exactly like the reference pre-process (x / 255).
        float x = (float)in[(((long long)n * a.cin + ci) * a.ih + iy) * a.iw + ix];
        if (sizeof(TIn) == 1) x = __fdiv_rn(x, 255.0f);
        const __nv_bfloat16 *wr = ws + (size_t)((ky * a.k + kx) * a.cin + ci) * a.cout + co0;
#pragma unroll
        for (int j = 0; j < CO_T; ++j) acc[j] = fmaf(x, bf2f(wr[j]), acc[j]);
      }
    }
  }
  const long long opix = ((long long)n * a.oh + oy) * a.ow + ox;
  __nv_bfloat16 *op = reinterpret_cast<__nv_bfloat16 *>(a.out) + opix * a.out_pitch + co0;
#pragma unroll
  for (int i = 0; i < CO_T; ++i) {
    float v = acc[i] + a.bias[co0 + i];
    if (a.relu) v = fmaxf(v, 0.f);
    op[i] = __float2bfloat16_rn(v);
  }
}

// Depth-wise 3x3 (Detect cv3 branch, DWConv): weights bf16 [tap][c]; thread = pixel x 8 ch.
__global__ void __launch_bounds__(kThreads) conv_dw_kernel(ConvArgs a) {
  const int cg = a.cin / 8;
  const long long total = (long long)a.n * a.oh * a.ow * cg;
  const long long t = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (t >= total) return;
  const int c0 = (int)(t % cg) * 8;
  const long long p = t / cg;
  const int ox = (int)(p % a.ow);
  const int oy = (int)((p / a.ow) % a.oh);
  const int n = (int)(p / ((long long)a.ow * a.oh));
  const int pad = a.k / 2;
  const __nv_bfloat16 *in = reinterpret_cast<const __nv_bfloat16 *>(a.in);
  const __nv_bfloat16 *w = reinterpret_cast<const __nv_bfloat16 *>(a.w);
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.f;
  for (int ky = 0; ky < a.k; ++ky) {
    const int iy = oy * a.stride + ky - pad;
    if (iy < 0 || iy >= a.ih) continue;
    for (int kx = 0; kx < a.k; ++kx) {
      const int ix = ox * a.stride + kx - pad;
      if (ix < 0 || ix >= a.iw) continue;
      float x[8], wv[8];
      load_bf16<8>(in + (((long long)n * a.ih + iy) * a.iw + ix) * a.in_pitch + c0, x);
      load_bf16<8>(w + (size_t)(ky * a.k + kx) * a.cin + c0, wv);
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[j] = fmaf(x[j], wv[j], acc[j]);
    }
  }
  __nv_bfloat16 *op = reinterpret_cast<__nv_bfloat16 *>(a.out) + (((long long)n * a.oh + oy) * a.ow + ox) * a.out_pitch + c0;
  uint4 pk;
  uint32_t *pw = reinterpret_cast<uint32_t *>(&pk);
#pragma unroll
  for (int i = 0; i < 8; i += 2) {
    float v0 = acc[i] + a.bias[c0 + i], v1 = acc[i + 1] + a.bias[c0 + i + 1];
    if (a.relu) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); }
    __nv_bfloat162 h = __floats2bfloat162_rn(v0, v1);
    pw[i / 2] = *reinterpret_cast<uint32_t *>(&h);
  }
  *reinterpret_cast<uint4 *>(op) = pk;
}

// Tiled stem for the shapes the networks actually have (3 -> 16 of the YAML graph when it is not fused, 3 -> 32 of
// model.py's backbone.stem, model.py:173): 3x3, stride 2.  A CTA stages the
// 33 x 65 x 3 input patch of a 16 x 32 output tile in shared memory with coalesced row reads
// (the frame is read once from HBM instead of 9x through L1); each thread computes two
// horizontally adjacent output pixels x 16 channels so that every weight vector read from
// shared memory feeds two FMAs (the kernel is FMA-bound, not LSU-bound).
constexpr int kStemTH = 16, kStemTW = 32, kStemThreads = 256;
template <typename TIn, int COUT>
__global__ void __launch_bounds__(kStemThreads) conv_stem_tiled_kernel(ConvArgs a) {
  // shared tile column j holds image column ox0*2 - 4 + j (4-element aligned so that rows are fetched
  // as 16-byte / 4-byte vectors); the conv reads columns 3 .. 67
  constexpr int IH = 2 * kStemTH + 1, NV = (2 * kStemTW) / 4 + 2, IP = NV * 4;
  __shared__ __align__(16) float sx[3][IH][IP];
  __shared__ __align__(16) float sw[27][COUT];
  const int tid = threadIdx.x;
  const int ox0 = blockIdx.x * kStemTW, oy0 = blockIdx.y * kStemTH, n = blockIdx.z;
  for (int i = tid; i < 27 * COUT; i += kStemThreads)
    sw[i / COUT][i % COUT] = __bfloat162float(reinterpret_cast<const __nv_bfloat16 *>(a.w)[i]);
  const TIn *in = reinterpret_cast<const TIn *>(a.in) + (long long)n * 3 * a.ih * a.iw;
  const bool vec_ok = a.iw % 4 == 0 && (reinterpret_cast<uintptr_t>(in) & 15) == 0;
#pragma unroll 4
  for (int i = tid; i < 3 * IH * NV; i += kStemThreads) {
    const int c = i / (IH * NV), r = (i / NV) % IH, j = i % NV;
    const int iy = oy0 * 2 - 1 + r, ix = ox0 * 2 - 4 + 4 * j;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (iy >= 0 && iy < a.ih) {
      const TIn *src = in + ((long long)c * a.ih + iy) * a.iw + ix;
      if (vec_ok && ix >= 0 && ix + 3 < a.iw) {
        if (sizeof(TIn) == 4) {
          v = *reinterpret_cast<const float4 *>(src);
        } else {
          const uchar4 u = *reinterpret_cast<const uchar4 *>(src);
          v = make_float4(__fdiv_rn((float)u.x, 255.f), __fdiv_rn((float)u.y, 255.f), __fdiv_rn((float)u.z, 255.f),
                          __fdiv_rn((float)u.w, 255.f));
        }
      } else {
        float t[4];
#pragma unroll
        for (int e = 0; e < 4; ++e) {
          t[e] = 0.f;
          if (ix + e >= 0 && ix + e < a.iw) {
            t[e] = (float)src[e];
            if (sizeof(TIn) == 1) t[e] = __fdiv_rn(t[e], 255.0f);
          }
        }
        v = make_float4(t[0], t[1], t[2], t[3]);
      }
    }
    *reinterpret_cast<float4 *>(&sx[c][r][4 * j]) = v;
  }
  __syncthreads();
  const int tx = tid % (kStemTW / 2), ty = tid / (kStemTW / 2);
  const int ox = ox0 + 2 * tx, oy = oy0 + ty;
  if (ox >= a.ow || oy >= a.oh) return;
  float acc[2][COUT];
#pragma unroll
  for (int i = 0; i < COUT; ++i) acc[0][i] = acc[1][i] = 0.f;
#pragma unroll
  for (int ky = 0; ky < 3; ++ky)
#pragma unroll
    for (int ci = 0; ci < 3; ++ci) {
      const float *row = &sx[ci][2 * ty + ky][4 * tx + 3];  // image column 2*ox - 1
      const float x[5] = {row[0], row[1], row[2], row[3], row[4]};
#pragma unroll
      for (int kx = 0; kx < 3; ++kx) {
        const float4 *wr = reinterpret_cast<const float4 *>(sw[(ky * 3 + kx) * 3 + ci]);
#pragma unroll
        for (int q = 0; q < COUT / 4; ++q) {
          const float4 w4 = wr[q];
          acc[0][4 * q] = fmaf(x[kx], w4.x, acc[0][4 * q]);
          acc[0][4 * q + 1] = fmaf(x[kx], w4.y, acc[0][4 * q + 1]);
          acc[0][4 * q + 2] = fmaf(x[kx], w4.z, acc[0][4 * q + 2]);
          acc[0][4 * q + 3] = fmaf(x[kx], w4.w, acc[0][4 * q + 3]);
          acc[1][4 * q] = fmaf(x[kx + 2], w4.x, acc[1][4 * q]);
          acc[1][4 * q + 1] = fmaf(x[kx + 2], w4.y, acc[1][4 * q + 1]);
          acc[1][4 * q + 2] = fmaf(x[kx + 2], w4.z, acc[1][4 * q + 2]);
          acc[1][4 * q + 3] = fmaf(x[kx + 2], w4.w, acc[1][4 * q + 3]);
        }
      }
    }
#pragma unroll
  for (int px = 0; px < 2; ++px) {
    if (ox + px >= a.ow) break;
    __nv_bfloat16 *op = reinterpret_cast<__nv_bfloat16 *>(a.out) + (((long long)n * a.oh + oy) * a.ow + ox + px) * a.out_pitch;
    uint4 o[COUT / 8];
    uint32_t *pw = reinterpret_cast<uint32_t *>(o);
#pragma unroll
    for (int i = 0; i < COUT; i += 2) {
      float v0 = acc[px][i] + a.bias[i], v1 = acc[px][i + 1] + a.bias[i + 1];
      if (a.relu) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); }
      __nv_bfloat162 h = __floats2bfloat162_rn(v0, v1);
      pw[i / 2] = *reinterpret_cast<uint32_t *>(&h);
    }
#pragma unroll
    for (int i = 0; i < COUT / 8; ++i) reinterpret_cast<uint4 *>(op)[i] = o[i];
  }
}

// model.py's backbone.stem (Conv 3 -> 32, 3x3, stride 2, model.py:173) on the legacy tensor path.  The tiled CUDA-core
// kernel above spent 0.59 ms per batch of 64 (19 TFLOP/s, 12 % of the model.py step).  Here the GEMM is TRANSPOSED as in
// stem_v2.cuh: output channels are the mma rows (A = weights, 2 m-tiles of 16, kept in registers by persistent CTAs),
// eight horizontally adjacent output pixels the columns (B = the frame patch), K = 9 (channel, ky) combinations of
// four consecutive patch columns (image columns 2 ox - 2 .. 2 ox + 1; the first has zero weights), four combinations
// per mma.m16n8k16.bf16 k-step, so a B register is ONE LDS.32 of the bf16 patch.
//   * A first version on mma.m16n8k8.tf32 (fp32 patch, 10 HMMA.1688 + 5 LDS.64 per 8 pixels) took 232 us; bf16 operands with
//     the frame SPLIT into hi + lo planes (x = hi + lo up to 2^-17: finer than tf32) take 212 us (12 HMMA.16816 + 12 LDS.32).
//     Both instructions issue at 2.0 cycles per SM (ncu, profiles/r03_issue.md section 4) and the HMMA pipe is 20-36 % busy:
//     the kernel is bound by its integer / staging instructions; the bf16 form stages half the bytes and keeps 24 instead
//     of 40 weight registers.
//   * Rows of m-tile mt are assigned to channels 4 (r & 7) + 2 mt + (r >> 3), so lane (g, t) ends up with channels
//     4g .. 4g + 3 of pixels 2t and 2t + 1: two 8-byte stores, 64 contiguous bytes per pixel across the warp.
//   * The loads of tile i + 1 are issued before tile i is computed (tiles strided by the grid).
//   * TIn = CamIn reads camera frames (camera.cuh) instead of a frame tensor: one 4-pixel vector of a patch row holds all
//     three channels, so the map runs over (row, vector), 3 raw uint4 per thread in flight (NV12 / BGRA at the model's
//     extent; converted in stage_cam()).  Resampled BGRA is read and blended in stage_cam(): its 16 taps per vector would not
//     fit the register budget of two CTAs per SM.  TIn = CamLetterboxIn (UYD_CAM_BGRA_LETTERBOX) reads and blends its
//     taps in stage_cam() the same way.
constexpr int kSmTH = 8, kSmTW = 64, kSmThreads = 256;          // output tile: one row of 64 pixels per warp
constexpr int kSmIH = 2 * kSmTH + 1, kSmNV = (2 * kSmTW) / 4 + 2;
constexpr int kSmIP = 152;  // bf16 per patch row (>= 4 kSmNV): row / plane strides of 12 and 20 banks keep the two
                            // combinations one LDS.32 touches in disjoint banks
static_assert(kSmIP >= 4 * kSmNV && kSmIP % 4 == 0, "patch pitch");

// the camera instantiation's arguments carry the frames
struct CamConvArgs : ConvArgs {
  CamFrames f;
};
template <typename TIn>
using StemMmaArgs = typename std::conditional<std::is_same<TIn, CamIn>::value || std::is_same<TIn, CamLetterboxIn>::value, CamConvArgs,
                                              ConvArgs>::type;

template <typename TIn, bool SPLIT>
__global__ void __launch_bounds__(kSmThreads) conv_stem_mma_kernel(StemMmaArgs<TIn> a, int tiles_x, int tiles_y, int total_tiles) {
  constexpr int NP = SPLIT ? 2 : 1;  // planes: hi (| lo)
  constexpr bool kLetterbox = std::is_same<TIn, CamLetterboxIn>::value;
  constexpr bool kCam = std::is_same<TIn, CamIn>::value || kLetterbox;
  __shared__ __align__(16) __nv_bfloat16 sx[NP][3][kSmIH][kSmIP];
  __shared__ float sw[27][32];
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  for (int i = tid; i < 27 * 32; i += kSmThreads) sw[i / 32][i % 32] = __bfloat162float(reinterpret_cast<const __nv_bfloat16 *>(a.w)[i]);
  const bool vec_ok = a.iw % 4 == 0 && (reinterpret_cast<uintptr_t>(a.in) & 15) == 0 && ((long long)a.ih * a.iw * sizeof(TIn)) % 16 == 0;
  // Patch staging: every load of a thread is issued before the first is used (7 x 16 B in flight per thread); the
  // (channel, row, vector) of element i = tid + 256 k advances incrementally (256 = 7 * 34 + 18)
  constexpr int kIters = kCam ? (kSmIH * kSmNV + kSmThreads - 1) / kSmThreads : (3 * kSmIH * kSmNV + kSmThreads - 1) / kSmThreads;
  static_assert(kSmThreads / kSmNV < kSmIH, "incremental (c, r, j) update");
  typename std::conditional<kCam, uint4, float4>::type pv[kIters];
  auto tile_origin = [&](int tile, int &n, int &oy0, int &ox0) {
    n = tile / (tiles_x * tiles_y);
    const int tr = tile - n * tiles_x * tiles_y;
    oy0 = (tr / tiles_x) * kSmTH;
    ox0 = (tr % tiles_x) * kSmTW;
  };
  auto issue = [&](int tile) {
    int n, oy0, ox0;
    tile_origin(tile, n, oy0, ox0);
    if constexpr (kCam) {
      const uint8_t *frame = reinterpret_cast<const uint8_t *>(a.in) + (long long)n * a.f.frame_stride;
      const uint8_t *uvp = a.f.uv ? a.f.uv + (long long)n * a.f.uv_frame_stride : nullptr;
      const bool raw = !kLetterbox && !cam_resampled(a, a.f);
      int j = tid % kSmNV, r = tid / kSmNV;
#pragma unroll
      for (int k = 0; k < kIters; ++k) {
        const int iy = oy0 * 2 - 1 + r, ix = ox0 * 2 - 4 + 4 * j;
        uint32_t w[4] = {0u, 0u, 0u, 0u};
        if (raw && r < kSmIH && iy >= 0 && iy < a.ih && ix >= 0 && ix + 3 < a.iw) cam_load4(a.f, frame, uvp, iy, ix, w);
        pv[k] = make_uint4(w[0], w[1], w[2], w[3]);
        j += kSmThreads % kSmNV;
        r += kSmThreads / kSmNV;
        if (j >= kSmNV) { j -= kSmNV; ++r; }
      }
    } else {
    const TIn *in = reinterpret_cast<const TIn *>(a.in) + (long long)n * 3 * a.ih * a.iw;
    int j = tid % kSmNV, r = tid / kSmNV, c = 0;
#pragma unroll
    for (int k = 0; k < kIters; ++k) {
      const int iy = oy0 * 2 - 1 + r, ix = ox0 * 2 - 4 + 4 * j;  // patch column 4 j = image column 2 ox0 - 4 + 4 j
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (c < 3 && iy >= 0 && iy < a.ih) {
        const TIn *src = in + ((long long)c * a.ih + iy) * a.iw + ix;
        if (vec_ok && ix >= 0 && ix + 3 < a.iw) {
          if (sizeof(TIn) == 4) {
            v = __ldg(reinterpret_cast<const float4 *>(src));
          } else {
            const uchar4 u = __ldg(reinterpret_cast<const uchar4 *>(src));
            v = make_float4((float)u.x, (float)u.y, (float)u.z, (float)u.w);
          }
        } else {
          float e4[4];
#pragma unroll
          for (int e = 0; e < 4; ++e) e4[e] = (ix + e >= 0 && ix + e < a.iw) ? (float)src[e] : 0.f;
          v = make_float4(e4[0], e4[1], e4[2], e4[3]);
        }
      }
      pv[k] = v;
      j += kSmThreads % kSmNV;
      r += kSmThreads / kSmNV;
      if (j >= kSmNV) { j -= kSmNV; ++r; }
      if (r >= kSmIH) { r -= kSmIH; ++c; }
    }
    }
  };
  __nv_bfloat16 *sx0 = &sx[0][0][0][0];
  constexpr int kPlane = 3 * kSmIH * kSmIP;  // bf16 elements of the hi plane set
  // the four values of patch vector (c, r, j) -> hi (| lo) bf16 planes
  auto put = [&](int c, int r, int j, const float4 &v) {
    const uint32_t h01 = c3kf::pack_bf16(v.x, v.y), h23 = c3kf::pack_bf16(v.z, v.w);
    __nv_bfloat16 *d = sx0 + (c * kSmIH + r) * kSmIP + 4 * j;
    *reinterpret_cast<uint2 *>(d) = make_uint2(h01, h23);
    if (SPLIT) {  // lo = bf16(x - hi): x = hi + lo up to 2^-17 relative
      const uint32_t l01 = c3kf::pack_bf16(v.x - c3kf::bf16_lo(h01), v.y - c3kf::bf16_hi(h01));
      const uint32_t l23 = c3kf::pack_bf16(v.z - c3kf::bf16_lo(h23), v.w - c3kf::bf16_hi(h23));
      *reinterpret_cast<uint2 *>(d + kPlane) = make_uint2(l01, l23);
    }
  };
  auto stage_cam = [&](int tile) {
    if constexpr (kCam) {  // zero outside the image (the conv's padding), normalised camera values inside
      int n, oy0, ox0;
      tile_origin(tile, n, oy0, ox0);
      const uint8_t *frame = reinterpret_cast<const uint8_t *>(a.in) + (long long)n * a.f.frame_stride;
      const CamNorm nm = cam_norm(a.f);
      const bool resampled = cam_resampled(a, a.f);
      CamLetterbox lb;
      if constexpr (kLetterbox) lb = cam_letterbox(a, a.f);
      int j = tid % kSmNV, r = tid / kSmNV;
#pragma unroll
      for (int k = 0; k < kIters; ++k) {
        if (r < kSmIH) {
          const int iy = oy0 * 2 - 1 + r, ix = ox0 * 2 - 4 + 4 * j;
          float px[4][3];
#pragma unroll
          for (int e = 0; e < 4; ++e) px[e][0] = px[e][1] = px[e][2] = 0.f;
          if (iy >= 0 && iy < a.ih && ix >= 0 && ix + 3 < a.iw) {
            if constexpr (kLetterbox) {
              cam_letterbox4(lb, a.f, nm, frame, iy, ix, px);
            } else if (resampled) {
              cam_resize4(a, a.f, nm, frame, iy, ix, px);
            } else {
              const uint32_t w[4] = {pv[k].x, pv[k].y, pv[k].z, pv[k].w};
              cam_convert4(a.f, nm, w, px);
            }
          }
#pragma unroll
          for (int c = 0; c < 3; ++c) put(c, r, j, make_float4(px[0][c], px[1][c], px[2][c], px[3][c]));
        }
        j += kSmThreads % kSmNV;
        r += kSmThreads / kSmNV;
        if (j >= kSmNV) { j -= kSmNV; ++r; }
      }
    }
  };
  auto stage = [&]() {
    if constexpr (!kCam) {
    int j = tid % kSmNV, r = tid / kSmNV, c = 0;
#pragma unroll
    for (int k = 0; k < kIters; ++k) {
      float4 v = pv[k];
      if (sizeof(TIn) == 1) v = make_float4(stemv2::div255(v.x), stemv2::div255(v.y), stemv2::div255(v.z), stemv2::div255(v.w));
      if (c < 3) put(c, r, j, v);
      j += kSmThreads % kSmNV;
      r += kSmThreads / kSmNV;
      if (j >= kSmNV) { j -= kSmNV; ++r; }
      if (r >= kSmIH) { r -= kSmIH; ++c; }
    }
    }
  };
  int tile = blockIdx.x;
  if (tile < total_tiles) issue(tile);
  __syncthreads();  // sw
  // A fragments (m16n8k16): a0 (g, 2t..) a1 (g + 8, 2t..) a2 (g, 2t + 8..) a3 (g + 8, 2t + 8..); logical k = 4 cl + slot with
  // cl = the combination inside the k-step (combination 4 s + cl = 3 channel + ky) and slot = kx + 1: registers a0 / a1
  // pair with the LDS.32 of combination 4 s + (t >> 1), a2 / a3 with that of combination 4 s + 2 + (t >> 1)
  uint32_t af[3][2][4];
  float bz[2][2];
#pragma unroll
  for (int mt = 0; mt < 2; ++mt) {
#pragma unroll
    for (int h = 0; h < 2; ++h) bz[mt][h] = a.bias[4 * g + 2 * mt + h];
#pragma unroll
    for (int s = 0; s < 3; ++s)
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int co = 4 * g + 2 * mt + (i & 1), combo = 4 * s + 2 * (i >> 1) + (t >> 1);
        float w[2];
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int kx = 2 * (t & 1) + e - 1;
          w[e] = (combo < 9 && kx >= 0) ? sw[((combo % 3) * 3 + kx) * 3 + combo / 3][co] : 0.f;
        }
        af[s][mt][i] = c3kf::pack_bf16(w[0], w[1]);  // already bf16 values: exact
      }
  }
  // bf16 offset of this lane's two LDS.32 in k-step s, relative to 2 (8 grp + g): patch column 2 ox - 2 = 2 (ox - ox0) + 2
  int koff[3][2];
#pragma unroll
  for (int s = 0; s < 3; ++s)
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      int combo = 4 * s + 2 * h + (t >> 1);
      if (combo > 8) combo = 8;  // zero-weight combinations re-read the last real one
      koff[s][h] = ((combo / 3) * kSmIH + 2 * warp + combo % 3) * kSmIP + 2 + 2 * (t & 1);
    }
  for (; tile < total_tiles; tile += gridDim.x) {
    if constexpr (kCam) stage_cam(tile);
    else stage();
    __syncthreads();
    if (tile + (int)gridDim.x < total_tiles) issue(tile + gridDim.x);  // in flight while this tile is computed
    int n, oy0, ox0;
    tile_origin(tile, n, oy0, ox0);
    const int oy = oy0 + warp;
    if (oy < a.oh) {
      __nv_bfloat16 *orow = reinterpret_cast<__nv_bfloat16 *>(a.out) + ((long long)n * a.oh + oy) * a.ow * a.out_pitch + 4 * g;
      __nv_bfloat16 *po = orow + (long long)(ox0 + 2 * t) * a.out_pitch;
#pragma unroll 4
      for (int grp = 0; grp < kSmTW / 8; ++grp) {
        float acc[2][4];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt) { acc[mt][0] = acc[mt][1] = bz[mt][0]; acc[mt][2] = acc[mt][3] = bz[mt][1]; }
        const __nv_bfloat16 *px = sx0 + 2 * (8 * grp + g);
#pragma unroll
        for (int pl = 0; pl < NP; ++pl)
#pragma unroll
          for (int s = 0; s < 3; ++s) {
            const uint32_t b0 = *reinterpret_cast<const uint32_t *>(px + pl * kPlane + koff[s][0]);
            const uint32_t b1 = *reinterpret_cast<const uint32_t *>(px + pl * kPlane + koff[s][1]);
#pragma unroll
            for (int mt = 0; mt < 2; ++mt)
              asm("mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
                  : "+f"(acc[mt][0]), "+f"(acc[mt][1]), "+f"(acc[mt][2]), "+f"(acc[mt][3])
                  : "r"(af[s][mt][0]), "r"(af[s][mt][1]), "r"(af[s][mt][2]), "r"(af[s][mt][3]), "r"(b0), "r"(b1));  // not volatile: the chains of unrolled groups interleave
          }
        // lane (g, t): channels 4g .. 4g + 3 = (mt 0 row g, mt 0 row g + 8, mt 1 row g, mt 1 row g + 8) of pixels 2t | 2t + 1
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          const int ox = ox0 + 8 * grp + 2 * t + e;
          if (ox >= a.ow) continue;
          uint32_t h0, h1;
          if (a.relu) {
            h0 = c3kf::relu_pack_bf16(acc[0][e], acc[0][2 + e]);
            h1 = c3kf::relu_pack_bf16(acc[1][e], acc[1][2 + e]);
          } else {
            h0 = c3kf::pack_bf16(acc[0][e], acc[0][2 + e]);
            h1 = c3kf::pack_bf16(acc[1][e], acc[1][2 + e]);
          }
          *reinterpret_cast<uint2 *>(po + (8 * grp + e) * a.out_pitch) = make_uint2(h0, h1);
        }
      }
    }
    __syncthreads();  // the patch is overwritten by the next stage()
  }
}

// Depth-wise 3x3 stride 1, four horizontally adjacent pixels x 8 channels per thread: the 3 x 6
// input window is loaded once (18 x 16 B) for 4 outputs instead of 36 loads.
__global__ void __launch_bounds__(kThreads) conv_dw4_kernel(ConvArgs a) {
  pdl_trigger();
  const int cg = a.cin / 8, wq = a.ow / 4;
  const long long total = (long long)a.n * a.oh * wq * cg;
  const long long t = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (t >= total) return;
  const int c0 = (int)(t % cg) * 8;
  const long long p = t / cg;
  const int ox0 = (int)(p % wq) * 4;
  const int oy = (int)((p / wq) % a.oh);
  const int n = (int)(p / ((long long)wq * a.oh));
  const __nv_bfloat16 *in = reinterpret_cast<const __nv_bfloat16 *>(a.in);
  const __nv_bfloat16 *w = reinterpret_cast<const __nv_bfloat16 *>(a.w);
  float acc[4][8];
#pragma unroll
  for (int q = 0; q < 4; ++q)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[q][j] = 0.f;
#pragma unroll
  for (int ky = 0; ky < 3; ++ky) {
    const int iy = oy + ky - 1;
    if (iy < 0 || iy >= a.ih) continue;
    float wv[3][8];
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) load_bf16<8>(w + (size_t)(ky * 3 + kx) * a.cin + c0, wv[kx]);
    const __nv_bfloat16 *row = in + ((long long)n * a.ih + iy) * a.iw * a.in_pitch + c0;
#pragma unroll
    for (int col = 0; col < 6; ++col) {
      const int ix = ox0 + col - 1;
      if (ix < 0 || ix >= a.iw) continue;
      float x[8];
      load_bf16<8>(row + (long long)ix * a.in_pitch, x);
#pragma unroll
      for (int q = 0; q < 4; ++q) {
        const int kx = col - q;  // output pixel q uses this column as tap kx
        if (kx >= 0 && kx < 3) {
#pragma unroll
          for (int j = 0; j < 8; ++j) acc[q][j] = fmaf(x[j], wv[kx][j], acc[q][j]);
        }
      }
    }
  }
  float bias[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) bias[j] = a.bias[c0 + j];
#pragma unroll
  for (int q = 0; q < 4; ++q) {
    __nv_bfloat16 *op = reinterpret_cast<__nv_bfloat16 *>(a.out) + (((long long)n * a.oh + oy) * a.ow + ox0 + q) * a.out_pitch + c0;
    uint4 pk;
    uint32_t *pw = reinterpret_cast<uint32_t *>(&pk);
#pragma unroll
    for (int i = 0; i < 8; i += 2) {
      float v0 = acc[q][i] + bias[i], v1 = acc[q][i + 1] + bias[i + 1];
      if (a.relu) { v0 = fmaxf(v0, 0.f); v1 = fmaxf(v1, 0.f); }
      __nv_bfloat162 h = __floats2bfloat162_rn(v0, v1);
      pw[i / 2] = *reinterpret_cast<uint32_t *>(&h);
    }
    *reinterpret_cast<uint4 *>(op) = pk;
  }
}

// Depth-wise 3x3 stride 1, column formulation (the P4 class branch's 128-channel conv at 40 x 40): a thread owns a
// channel QUAD of one output column over R rows.  The 36 weights stay in registers as fp32 pairs, every input row is
// loaded once (three 8-byte loads: columns x - 1, x, x + 1) and feeds the three output rows it is a tap row of,
// accumulators of three rows in flight (ring-indexed), packed FFMA2.  Per 32 outputs: 30 x 8 bytes loaded, 60
// unpack and 144 FFMA2 instructions -- conv_dw4_kernel above needs 29 x 16 bytes, 216 unpacks and 288 FFMAs.
// Lanes run over the channel quads first: a warp reads / writes whole pixels (256 contiguous bytes at C = 128).
__device__ __forceinline__ float2 dw_ffma2(float2 a, float2 b, float2 c) {
  float2 d;
  asm("{\n\t.reg .b64 ra, rb, rc, rd;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
      "fma.rn.f32x2 rd, ra, rb, rc;\n\tmov.b64 {%0, %1}, rd;\n\t}"
      : "=f"(d.x), "=f"(d.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
  return d;
}
template <int R>
__global__ void __launch_bounds__(kThreads) conv_dw_col_kernel(ConvArgs a) {
  pdl_trigger();
  const int nq = a.cin / 4, segs = (a.oh + R - 1) / R;
  const long long total = (long long)a.n * segs * a.ow * nq;
  const long long t = (long long)blockIdx.x * kThreads + threadIdx.x;
  if (t >= total) return;
  const int q = (int)(t % nq);
  long long p = t / nq;
  const int x = (int)(p % a.ow);
  p /= a.ow;
  const int oy0 = (int)(p % segs) * R, n = (int)(p / segs);
  const __nv_bfloat16 *in = reinterpret_cast<const __nv_bfloat16 *>(a.in) + (long long)n * a.ih * a.iw * a.in_pitch + 4 * q;
  __nv_bfloat16 *out = reinterpret_cast<__nv_bfloat16 *>(a.out) + (long long)n * a.oh * a.ow * a.out_pitch + 4 * q;
  const __nv_bfloat16 *w = reinterpret_cast<const __nv_bfloat16 *>(a.w) + 4 * q;
  auto lo2 = [](uint32_t v) { return make_float2(__uint_as_float(v << 16), __uint_as_float(v & 0xffff0000u)); };
  float2 wlo[9], whi[9];
#pragma unroll
  for (int tap = 0; tap < 9; ++tap) {
    const uint2 h = __ldg(reinterpret_cast<const uint2 *>(w + (size_t)tap * a.cin));
    wlo[tap] = lo2(h.x);
    whi[tap] = lo2(h.y);
  }
  const float4 b4 = __ldg(reinterpret_cast<const float4 *>(a.bias + 4 * q));
  const float2 blo = make_float2(b4.x, b4.y), bhi = make_float2(b4.z, b4.w);
  const bool left = x > 0, right = x + 1 < a.iw;
  auto load_row = [&](int i, uint2 (&h)[3]) {  // input row oy0 - 1 + i, columns x - 1 .. x + 1 (zero outside the image)
    const int iy = oy0 - 1 + i;
    h[0] = h[1] = h[2] = make_uint2(0u, 0u);
    if (iy >= 0 && iy < a.ih) {
      const __nv_bfloat16 *r = in + ((long long)iy * a.iw + x) * a.in_pitch;
      if (left) h[0] = __ldg(reinterpret_cast<const uint2 *>(r - a.in_pitch));
      h[1] = __ldg(reinterpret_cast<const uint2 *>(r));
      if (right) h[2] = __ldg(reinterpret_cast<const uint2 *>(r + a.in_pitch));
    }
  };
  float2 a0[3], a1[3];
  uint2 cur[3], nxt[3];
  load_row(0, cur);
#pragma unroll
  for (int i = 0; i < R + 2; ++i) {
    if (i + 1 < R + 2) load_row(i + 1, nxt);  // in flight while row i is consumed
    float2 v0[3], v1[3];
#pragma unroll
    for (int dx = 0; dx < 3; ++dx) { v0[dx] = lo2(cur[dx].x); v1[dx] = lo2(cur[dx].y); }
#pragma unroll
    for (int tr = 0; tr < 3; ++tr) {  // input row i is tap row tr of output row i - tr
      const int r = i - tr;
      if (r < 0 || r >= R) continue;
      float2 &o0 = a0[r % 3], &o1 = a1[r % 3];
      if (tr == 0) { o0 = blo; o1 = bhi; }
#pragma unroll
      for (int dx = 0; dx < 3; ++dx) {
        o0 = dw_ffma2(v0[dx], wlo[tr * 3 + dx], o0);
        o1 = dw_ffma2(v1[dx], whi[tr * 3 + dx], o1);
      }
      if (tr == 2 && oy0 + r < a.oh) {
        float2 y0 = o0, y1 = o1;
        if (a.relu) { y0.x = fmaxf(y0.x, 0.f); y0.y = fmaxf(y0.y, 0.f); y1.x = fmaxf(y1.x, 0.f); y1.y = fmaxf(y1.y, 0.f); }
        const __nv_bfloat162 h0 = __floats2bfloat162_rn(y0.x, y0.y), h1 = __floats2bfloat162_rn(y1.x, y1.y);
        *reinterpret_cast<uint2 *>(out + ((long long)(oy0 + r) * a.ow + x) * a.out_pitch) =
            make_uint2(*reinterpret_cast<const uint32_t *>(&h0), *reinterpret_cast<const uint32_t *>(&h1));
      }
    }
#pragma unroll
    for (int dx = 0; dx < 3; ++dx) cur[dx] = nxt[dx];
  }
}

template <int CO_T, int IN_VEC>
int launch_generic(const ConvArgs &a, cudaStream_t s) {
  const long long npix = (long long)a.n * a.oh * a.ow;
  dim3 grid((unsigned)((npix + kThreads - 1) / kThreads), a.cout / CO_T);
  const size_t wbytes = (size_t)a.k * a.k * a.cin * a.cout * 2;
  if (wbytes <= kSmemWeightLimit) {
    auto kern = conv_direct_kernel<CO_T, IN_VEC, true>;
    if (wbytes > 48 * 1024) cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemWeightLimit);
    kern<<<grid, kThreads, wbytes, s>>>(a);
  } else {
    conv_direct_kernel<CO_T, IN_VEC, false><<<grid, kThreads, 0, s>>>(a);
  }
  return (int)cudaGetLastError();
}

}  // namespace

size_t direct_weight_bytes(const uyd_conv &d) {
  return d.depthwise ? (size_t)d.k * d.k * d.cin * 2 : (size_t)d.k * d.k * d.cin * d.cout * 2;
}

// PyTorch [cout][cin/g][k][k] fp32 -> bf16 [tap][ci][co]  (depth-wise: [tap][c])
void direct_pack_weights(const uyd_conv &d, const float *w, void *dst_host) {
  __nv_bfloat16 *o = reinterpret_cast<__nv_bfloat16 *>(dst_host);
  const int taps = d.k * d.k;
  if (d.depthwise) {
    for (int t = 0; t < taps; ++t)
      for (int c = 0; c < d.cin; ++c) o[(size_t)t * d.cin + c] = __float2bfloat16_rn(w[(size_t)c * taps + t]);
    return;
  }
  for (int t = 0; t < taps; ++t)
    for (int ci = 0; ci < d.cin; ++ci)
      for (int co = 0; co < d.cout; ++co)
        o[((size_t)t * d.cin + ci) * d.cout + co] = __float2bfloat16_rn(w[((size_t)co * d.cin + ci) * taps + t]);
}

static unsigned stem_mma_grid(const ConvArgs &a, int &tx, int &ty, int &total) {
  tx = ceil_div(a.ow, kSmTW); ty = ceil_div(a.oh, kSmTH); total = tx * ty * a.n;
  const int resident = 2 * current_sm_count();  // 256 threads x <= 128 registers: two CTAs per SM
  return (unsigned)(total < resident ? total : resident);
}

bool stem_camera_supported(const ConvArgs &a) {
  return a.cin == 3 && a.cout == 32 && a.k == 3 && a.stride == 2 && !a.out_f32 && !a.res && a.iw % 4 == 0 && a.out_pitch % 8 == 0 &&
         (reinterpret_cast<uintptr_t>(a.out) & 15) == 0;
}

int stem_camera_launch(const ConvArgs &a, const CamFrames &f, cudaStream_t s) {
  UYD_REQUIRE(stem_camera_supported(a), UYD_E_UNSUPPORTED, "camera frames feed only the 3 -> 32 3x3 stride-2 mma stem (16-byte aligned output)");
  int tx, ty, total;
  const unsigned mgrid = stem_mma_grid(a, tx, ty, total);
  CamConvArgs ca;
  static_cast<ConvArgs &>(ca) = a;
  ca.f = f;
  if (f.cam == UYD_CAM_BGRA_LETTERBOX) conv_stem_mma_kernel<CamLetterboxIn, true><<<mgrid, kSmThreads, 0, s>>>(ca, tx, ty, total);
  else conv_stem_mma_kernel<CamIn, true><<<mgrid, kSmThreads, 0, s>>>(ca, tx, ty, total);
  return (int)cudaGetLastError();
}

int direct_conv_launch(const ConvArgs &a, bool depthwise, cudaStream_t s) {
  if (depthwise) {
    UYD_REQUIRE(a.cin % 8 == 0 && a.in_pitch % 8 == 0 && a.out_pitch % 8 == 0 && !a.out_f32 && !a.res &&
                    (reinterpret_cast<uintptr_t>(a.in) & 15) == 0 && (reinterpret_cast<uintptr_t>(a.out) & 15) == 0,
                UYD_E_UNSUPPORTED, "depthwise conv needs C %% 8 == 0 and 16-byte aligned slices");
    if (a.k == 3 && a.stride == 1 && a.ih == a.oh && a.iw == a.ow && getenv("UYD_DW_OLD") == nullptr) {
      auto go = [&](auto kern, int R) {
        const long long totalc = (long long)a.n * ((a.oh + R - 1) / R) * a.ow * (a.cin / 4);
        kern<<<(unsigned)((totalc + kThreads - 1) / kThreads), kThreads, 0, s>>>(a);
        return (int)cudaGetLastError();
      };
      // rows per thread (measured at 64 x 40 x 40 x 128: R = 4 / 8 / 10 / 20 -> 30.8 / 25.6 / 24.6 / 23.4 us): the tallest
      // strip that still leaves 1024 threads per SM
      const long long cols = (long long)a.n * a.ow * (a.cin / 4), want = 1024ll * current_sm_count();
      if (a.oh % 20 == 0 && cols * (a.oh / 20) >= want) return go(conv_dw_col_kernel<20>, 20);
      if (a.oh % 10 == 0 && cols * (a.oh / 10) >= want) return go(conv_dw_col_kernel<10>, 10);
      return go(conv_dw_col_kernel<8>, 8);
    }
    if (a.k == 3 && a.stride == 1 && a.ow % 4 == 0) {
      const long long total4 = (long long)a.n * a.oh * (a.ow / 4) * (a.cin / 8);
      conv_dw4_kernel<<<(unsigned)((total4 + kThreads - 1) / kThreads), kThreads, 0, s>>>(a);
      return (int)cudaGetLastError();
    }
    const long long total = (long long)a.n * a.oh * a.ow * (a.cin / 8);
    conv_dw_kernel<<<(unsigned)((total + kThreads - 1) / kThreads), kThreads, 0, s>>>(a);
    return (int)cudaGetLastError();
  }
  if (a.in_nchw_f32) {
    UYD_REQUIRE(!a.out_f32 && !a.res, UYD_E_UNSUPPORTED, "stem conv writes bf16 without residual");
    const long long npix = (long long)a.n * a.oh * a.ow;
    const size_t wbytes = (size_t)a.k * a.k * a.cin * a.cout * 2;
    UYD_REQUIRE(wbytes <= 48 * 1024, UYD_E_UNSUPPORTED, "stem weights too large");
    const bool u8 = a.in_nchw_f32 == 2;
    if (a.cin == 3 && (a.cout == 16 || a.cout == 32) && a.k == 3 && a.stride == 2 && a.out_pitch % 8 == 0 &&
        (reinterpret_cast<uintptr_t>(a.out) & 15) == 0) {
      if (a.cout == 32 && a.out_pitch % 4 == 0 && getenv("UYD_STEM_TILED") == nullptr) {
        int tx, ty, total;
        const unsigned mgrid = stem_mma_grid(a, tx, ty, total);
        static const bool split = getenv("UYD_STEM_NO_SPLIT") == nullptr;  // probe: hi plane only (bf16-rounded frame)
        if (split) {
          if (u8) conv_stem_mma_kernel<uint8_t, true><<<mgrid, kSmThreads, 0, s>>>(a, tx, ty, total);
          else conv_stem_mma_kernel<float, true><<<mgrid, kSmThreads, 0, s>>>(a, tx, ty, total);
        } else {
          if (u8) conv_stem_mma_kernel<uint8_t, false><<<mgrid, kSmThreads, 0, s>>>(a, tx, ty, total);
          else conv_stem_mma_kernel<float, false><<<mgrid, kSmThreads, 0, s>>>(a, tx, ty, total);
        }
        return (int)cudaGetLastError();
      }
      dim3 grid(ceil_div(a.ow, kStemTW), ceil_div(a.oh, kStemTH), a.n);
      if (a.cout == 16) {
        if (u8) conv_stem_tiled_kernel<uint8_t, 16><<<grid, kStemThreads, 0, s>>>(a);
        else conv_stem_tiled_kernel<float, 16><<<grid, kStemThreads, 0, s>>>(a);
      } else {
        if (u8) conv_stem_tiled_kernel<uint8_t, 32><<<grid, kStemThreads, 0, s>>>(a);
        else conv_stem_tiled_kernel<float, 32><<<grid, kStemThreads, 0, s>>>(a);
      }
      return (int)cudaGetLastError();
    }
    if (a.cout % 16 == 0) {
      dim3 grid((unsigned)((npix + kThreads - 1) / kThreads), a.cout / 16);
      if (u8) conv_stem_nchw_kernel<16, uint8_t><<<grid, kThreads, wbytes, s>>>(a);
      else conv_stem_nchw_kernel<16, float><<<grid, kThreads, wbytes, s>>>(a);
    } else {
      UYD_REQUIRE(a.cout % 4 == 0, UYD_E_UNSUPPORTED, "stem cout must be a multiple of 4");
      dim3 grid((unsigned)((npix + kThreads - 1) / kThreads), a.cout / 4);
      if (u8) conv_stem_nchw_kernel<4, uint8_t><<<grid, kThreads, wbytes, s>>>(a);
      else conv_stem_nchw_kernel<4, float><<<grid, kThreads, wbytes, s>>>(a);
    }
    return (int)cudaGetLastError();
  }
  UYD_REQUIRE(a.cin % 4 == 0 && a.cout % 4 == 0, UYD_E_UNSUPPORTED, "direct conv needs cin, cout %% 4 == 0 (got %d, %d)", a.cin, a.cout);
  const bool in16 = a.cin % 8 == 0 && a.in_pitch % 8 == 0 && (reinterpret_cast<uintptr_t>(a.in) & 15) == 0;
  UYD_REQUIRE(in16 || (a.in_pitch % 4 == 0 && (reinterpret_cast<uintptr_t>(a.in) & 7) == 0), UYD_E_UNSUPPORTED,
              "input slice must be 8-byte aligned");
  // weight rows are read as 8-byte (CO_T=4) or 16-byte vectors
  if (a.cout % 16 == 0) return in16 ? launch_generic<16, 8>(a, s) : launch_generic<16, 4>(a, s);
  if (a.cout % 8 == 0) return in16 ? launch_generic<8, 8>(a, s) : launch_generic<8, 4>(a, s);
  return in16 ? launch_generic<4, 8>(a, s) : launch_generic<4, 4>(a, s);
}

}  // namespace uyd

// ---- INT8 (dp4a) path ----------------------------------------------------------------------------
// Same requant epilogue as the tensor-core int8 kernel (oracle/quant.py): exact int32
// accumulation, y = float(acc) * m_c + b_c (separate RN multiply / add), ReLU, + residual (bf16,
// added in fp32 after the activation), then bf16 / fp32 / int8 re-quantised with out_scale.
// weights: int8 [tap][co][ci]  (depth-wise: [tap][c]).
namespace uyd {
namespace {

__device__ __forceinline__ void store_s8_result(const ConvArgs &a, long long o, float y, float out_scale, int out_kind) {
  if (out_kind >= 2) {  // 3: the activation is a bf16 tensor in the graph -- round it to bf16 first, then the consumer's quantiser
    if (out_kind == 3) y = __bfloat162float(__float2bfloat16_rn(y));
    const int q = max(-127, min(127, __float2int_rn(__fmul_rn(y, out_scale))));
    reinterpret_cast<int8_t *>(a.out)[o] = (int8_t)q;
  } else if (out_kind == 1) {
    reinterpret_cast<float *>(a.out)[o] = y;
  } else {
    reinterpret_cast<__nv_bfloat16 *>(a.out)[o] = __float2bfloat16_rn(y);
  }
}

__global__ void __launch_bounds__(128) conv_s8_direct_kernel(ConvArgs a, const float *mult, float out_scale, int out_kind) {
  const long long npix = (long long)a.n * a.oh * a.ow;
  const long long p = (long long)blockIdx.x * 128 + threadIdx.x;
  if (p >= npix) return;
  const int co0 = blockIdx.y * 4;
  const int ox = (int)(p % a.ow), oy = (int)((p / a.ow) % a.oh), n = (int)(p / ((long long)a.ow * a.oh));
  const int pad = a.k / 2;
  const int8_t *in = reinterpret_cast<const int8_t *>(a.in);
  const int8_t *w = reinterpret_cast<const int8_t *>(a.w);
  int acc[4] = {0, 0, 0, 0};
  for (int ky = 0; ky < a.k; ++ky) {
    const int iy = oy * a.stride + ky - pad;
    if (iy < 0 || iy >= a.ih) continue;
    for (int kx = 0; kx < a.k; ++kx) {
      const int ix = ox * a.stride + kx - pad;
      if (ix < 0 || ix >= a.iw) continue;
      const int *px = reinterpret_cast<const int *>(in + (((long long)n * a.ih + iy) * a.iw + ix) * a.in_pitch);
      const int8_t *wt = w + ((size_t)(ky * a.k + kx) * a.cout + co0) * a.cin;
      for (int c4 = 0; c4 < a.cin / 4; ++c4) {
        const int x = px[c4];
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (co0 + j < a.cout) acc[j] = __dp4a(x, reinterpret_cast<const int *>(wt + (size_t)j * a.cin)[c4], acc[j]);
      }
    }
  }
  const long long opix = ((long long)n * a.oh + oy) * a.ow + ox;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    if (co0 + j >= a.cout) break;
    float y = __fadd_rn(__fmul_rn(__int2float_rn(acc[j]), mult[co0 + j]), a.bias[co0 + j]);
    if (a.relu) y = fmaxf(y, 0.f);
    if (a.res) y = __fadd_rn(y, __bfloat162float(reinterpret_cast<const __nv_bfloat16 *>(a.res)[opix * a.res_pitch + co0 + j]));
    store_s8_result(a, opix * a.out_pitch + co0 + j, y, out_scale, out_kind);
  }
}

// 4 -> 4 channels, 3x3, stride 1, bf16 output (the bottleneck convs of the 160 x 160 C3k blocks in the INT8 graph): the
// general kernel above spends its time on 64-bit index arithmetic, per-tap weight loads and four 2-byte stores
// (0.27 ms per launch at batch 256 = 0.3 TB/s).  Here: 32-bit indices, the 36 weight words in registers, one 8-byte
// store per pixel.  Identical arithmetic per element (exact int32 sums, the same fp32 epilogue ops in the same order).
// Q8: the output is the int8 input of the next QuantConv2d (round to bf16, multiply by its scale, round, clamp): 4 bytes per pixel
template <bool Q8>
__global__ void __launch_bounds__(256) conv_s8_c4_kernel(ConvArgs a, const float *__restrict__ mult, float out_scale) {
  const unsigned npix = (unsigned)a.n * a.oh * a.ow;
  const unsigned p = blockIdx.x * 256u + threadIdx.x;
  int wr[9][4];
#pragma unroll
  for (int t = 0; t < 9; ++t)
#pragma unroll
    for (int j = 0; j < 4; ++j) wr[t][j] = __ldg(reinterpret_cast<const int *>(a.w) + t * 4 + j);  // [tap][cout][cin = 4]
  if (p >= npix) return;
  const unsigned hw = (unsigned)a.oh * a.ow;
  const unsigned n = p / hw, r = p - n * hw, oy = r / (unsigned)a.ow, ox = r - oy * (unsigned)a.ow;
  const int8_t *in = reinterpret_cast<const int8_t *>(a.in);
  int acc[4] = {0, 0, 0, 0};
#pragma unroll
  for (int ky = 0; ky < 3; ++ky) {
    const int iy = (int)oy + ky - 1;
    if (iy < 0 || iy >= a.ih) continue;
#pragma unroll
    for (int kx = 0; kx < 3; ++kx) {
      const int ix = (int)ox + kx - 1;
      if (ix < 0 || ix >= a.iw) continue;
      const int x = *reinterpret_cast<const int *>(in + (size_t)((n * a.ih + iy) * a.iw + ix) * a.in_pitch);
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[j] = __dp4a(x, wr[ky * 3 + kx][j], acc[j]);
    }
  }
  float y[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    y[j] = __fadd_rn(__fmul_rn(__int2float_rn(acc[j]), __ldg(mult + j)), __ldg(a.bias + j));
    if (a.relu) y[j] = fmaxf(y[j], 0.f);
  }
  if (a.res) {
    const uint2 rv = *reinterpret_cast<const uint2 *>(reinterpret_cast<const __nv_bfloat16 *>(a.res) + (size_t)p * a.res_pitch);
    y[0] = __fadd_rn(y[0], __uint_as_float(rv.x << 16)); y[1] = __fadd_rn(y[1], __uint_as_float(rv.x & 0xffff0000u));
    y[2] = __fadd_rn(y[2], __uint_as_float(rv.y << 16)); y[3] = __fadd_rn(y[3], __uint_as_float(rv.y & 0xffff0000u));
  }
  if (Q8) {
    uint32_t pk = 0;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float yb = __bfloat162float(__float2bfloat16_rn(y[j]));
      const int q = max(-127, min(127, __float2int_rn(__fmul_rn(yb, out_scale))));
      pk |= (uint32_t)(q & 0xFF) << (8 * j);
    }
    *reinterpret_cast<uint32_t *>(reinterpret_cast<int8_t *>(a.out) + (size_t)p * a.out_pitch) = pk;
    return;
  }
  const __nv_bfloat162 h0 = __floats2bfloat162_rn(y[0], y[1]), h1 = __floats2bfloat162_rn(y[2], y[3]);
  *reinterpret_cast<uint2 *>(reinterpret_cast<__nv_bfloat16 *>(a.out) + (size_t)p * a.out_pitch) =
      make_uint2(*reinterpret_cast<const uint32_t *>(&h0), *reinterpret_cast<const uint32_t *>(&h1));
}

// depth-wise 3x3 (any stride), thread = pixel x 4 channels
__global__ void __launch_bounds__(128) conv_s8_dw_kernel(ConvArgs a, const float *mult, float out_scale, int out_kind) {
  const int cg = a.cin / 4;
  const long long total = (long long)a.n * a.oh * a.ow * cg;
  const long long t = (long long)blockIdx.x * 128 + threadIdx.x;
  if (t >= total) return;
  const int c0 = (int)(t % cg) * 4;
  const long long p = t / cg;
  const int ox = (int)(p % a.ow), oy = (int)((p / a.ow) % a.oh), n = (int)(p / ((long long)a.ow * a.oh));
  const int pad = a.k / 2;
  const int8_t *in = reinterpret_cast<const int8_t *>(a.in);
  const int8_t *w = reinterpret_cast<const int8_t *>(a.w);
  int acc[4] = {0, 0, 0, 0};
  for (int ky = 0; ky < a.k; ++ky) {
    const int iy = oy * a.stride + ky - pad;
    if (iy < 0 || iy >= a.ih) continue;
    for (int kx = 0; kx < a.k; ++kx) {
      const int ix = ox * a.stride + kx - pad;
      if (ix < 0 || ix >= a.iw) continue;
      const char4 x = *reinterpret_cast<const char4 *>(in + (((long long)n * a.ih + iy) * a.iw + ix) * a.in_pitch + c0);
      const char4 wv = *reinterpret_cast<const char4 *>(w + (size_t)(ky * a.k + kx) * a.cin + c0);
      acc[0] += (int)x.x * wv.x; acc[1] += (int)x.y * wv.y; acc[2] += (int)x.z * wv.z; acc[3] += (int)x.w * wv.w;
    }
  }
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    float y = __fadd_rn(__fmul_rn(__int2float_rn(acc[j]), mult[c0 + j]), a.bias[c0 + j]);
    if (a.relu) y = fmaxf(y, 0.f);
    store_s8_result(a, p * a.out_pitch + c0 + j, y, out_scale, out_kind);
  }
}

// q = clamp(rne(x * scale), -127, 127): the input quantiser of a QuantConv2d (qat.py:109-124), one
// thread = 4 channels of one pixel (the narrowest slices of the graph are 4 channels wide).
__global__ void __launch_bounds__(256) quantize_s8_kernel(const __nv_bfloat16 *__restrict__ in, int in_pitch,
                                                          int8_t *__restrict__ out, int out_pitch, long long npix, int c,
                                                          float scale) {
  const int cg = c / 4;
  const long long t = (long long)blockIdx.x * 256 + threadIdx.x;
  if (t >= npix * cg) return;
  const int c0 = (int)(t % cg) * 4;
  const long long p = t / cg;
  const uint2 raw = *reinterpret_cast<const uint2 *>(in + p * in_pitch + c0);
  const __nv_bfloat162 *h = reinterpret_cast<const __nv_bfloat162 *>(&raw);
  uint32_t w = 0u;
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const float2 f = __bfloat1622float2(h[i]);
    const int q0 = max(-127, min(127, __float2int_rn(__fmul_rn(f.x, scale))));
    const int q1 = max(-127, min(127, __float2int_rn(__fmul_rn(f.y, scale))));
    w |= ((uint32_t)(q0 & 0xFF) << (16 * i)) | ((uint32_t)(q1 & 0xFF) << (16 * i + 8));
  }
  *reinterpret_cast<uint32_t *>(out + p * out_pitch + c0) = w;
}

// 16 channels per thread (two 16-byte loads, one 16-byte store), four items per thread in flight, 32-bit indexing:
// the 4-channel kernel above reached 3.1 TB/s (121 quantize launches = 35 % of the INT8 step).  Same arithmetic per element.
__device__ __forceinline__ uint32_t quant4(uint32_t lo, uint32_t hi, float scale) {
  const float f0 = __uint_as_float(lo << 16), f1 = __uint_as_float(lo & 0xffff0000u);
  const float f2 = __uint_as_float(hi << 16), f3 = __uint_as_float(hi & 0xffff0000u);
  const int q0 = max(-127, min(127, __float2int_rn(__fmul_rn(f0, scale))));
  const int q1 = max(-127, min(127, __float2int_rn(__fmul_rn(f1, scale))));
  const int q2 = max(-127, min(127, __float2int_rn(__fmul_rn(f2, scale))));
  const int q3 = max(-127, min(127, __float2int_rn(__fmul_rn(f3, scale))));
  return (uint32_t)(q0 & 0xFF) | ((uint32_t)(q1 & 0xFF) << 8) | ((uint32_t)(q2 & 0xFF) << 16) | ((uint32_t)(q3 & 0xFF) << 24);
}
__global__ void __launch_bounds__(256) quantize_s8_x16_kernel(const __nv_bfloat16 *__restrict__ in, int in_pitch,
                                                              int8_t *__restrict__ out, int out_pitch, unsigned total, int cg,
                                                              float scale) {
  constexpr int U = 4;
  const unsigned t0 = blockIdx.x * (256u * U) + threadIdx.x;
  uint4 a[U], b[U];
  unsigned px[U], c0[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    const unsigned t = t0 + u * 256u;
    px[u] = t / (unsigned)cg;
    c0[u] = (t - px[u] * (unsigned)cg) * 16u;
    if (t < total) {
      const uint4 *src = reinterpret_cast<const uint4 *>(in + (size_t)px[u] * in_pitch + c0[u]);
      a[u] = src[0];
      b[u] = src[1];
    }
  }
#pragma unroll
  for (int u = 0; u < U; ++u) {
    if (t0 + u * 256u < total)
      *reinterpret_cast<uint4 *>(out + (size_t)px[u] * out_pitch + c0[u]) =
          make_uint4(quant4(a[u].x, a[u].y, scale), quant4(a[u].z, a[u].w, scale), quant4(b[u].x, b[u].y, scale), quant4(b[u].z, b[u].w, scale));
  }
}

// |x| maximum of a bf16 slice (max calibration of the input quantisers, qat.py:129-220): the bit pattern of a
// non-negative float orders like an unsigned integer, so one atomicMax per block suffices.
__global__ void __launch_bounds__(256) absmax_kernel(const __nv_bfloat16 *__restrict__ in, int in_pitch, long long npix, int c,
                                                     unsigned int *__restrict__ out_bits) {
  const int cg = c / 4;
  float m = 0.f;
  for (long long t = (long long)blockIdx.x * 256 + threadIdx.x; t < npix * cg; t += (long long)gridDim.x * 256) {
    const int c0 = (int)(t % cg) * 4;
    const uint2 raw = *reinterpret_cast<const uint2 *>(in + (t / cg) * in_pitch + c0);
    const __nv_bfloat162 *h = reinterpret_cast<const __nv_bfloat162 *>(&raw);
    const float2 f0 = __bfloat1622float2(h[0]), f1 = __bfloat1622float2(h[1]);
    m = fmaxf(m, fmaxf(fmaxf(fabsf(f0.x), fabsf(f0.y)), fmaxf(fabsf(f1.x), fabsf(f1.y))));
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, o));
  if ((threadIdx.x & 31) == 0 && m > 0.f) atomicMax(out_bits, __float_as_uint(m));
}

// Histogram of |x| over a bf16 slice (histogram / entropy calibration, qat.py:91-126: the reference's default
// calibrator is pytorch-quantization's HistogramCalibrator): bin = min(floor(|x| * inv_width), nbins - 1), counts
// privatised per block in shared memory and flushed with one global atomic per non-empty bin.
__global__ void __launch_bounds__(256) abs_histogram_kernel(const __nv_bfloat16 *__restrict__ in, int in_pitch, long long npix, int c,
                                                            float inv_width, int nbins, unsigned int *__restrict__ hist) {
  extern __shared__ unsigned int sh[];
  for (int i = threadIdx.x; i < nbins; i += 256) sh[i] = 0u;
  __syncthreads();
  const int cg = c / 4;
  for (long long t = (long long)blockIdx.x * 256 + threadIdx.x; t < npix * cg; t += (long long)gridDim.x * 256) {
    const int c0 = (int)(t % cg) * 4;
    const uint2 raw = *reinterpret_cast<const uint2 *>(in + (t / cg) * in_pitch + c0);
    const __nv_bfloat162 *h = reinterpret_cast<const __nv_bfloat162 *>(&raw);
    const float2 f0 = __bfloat1622float2(h[0]), f1 = __bfloat1622float2(h[1]);
    const float v[4] = {f0.x, f0.y, f1.x, f1.y};
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int b = min((int)__fmul_rn(fabsf(v[i]), inv_width), nbins - 1);
      atomicAdd(&sh[b], 1u);
    }
  }
  __syncthreads();
  for (int i = threadIdx.x; i < nbins; i += 256)
    if (sh[i]) atomicAdd(&hist[i], sh[i]);
}
}  // namespace

int abs_histogram_launch(const __nv_bfloat16 *in, int in_pitch, long long npix, int c, float inv_width, int nbins, unsigned int *hist,
                         cudaStream_t s) {
  UYD_REQUIRE(c % 4 == 0 && in_pitch % 4 == 0 && (reinterpret_cast<uintptr_t>(in) & 7) == 0, UYD_E_UNSUPPORTED,
              "histogram: C %% 4 == 0 and 8-byte aligned slices");
  UYD_REQUIRE(nbins > 0 && nbins <= 12288 && inv_width > 0.f, UYD_E_ARG, "histogram: 0 < nbins <= 12288, positive bin width");
  long long blocks = (npix * (c / 4) + 255) / 256;
  if (blocks > 148 * 4) blocks = 148 * 4;
  abs_histogram_kernel<<<(unsigned)blocks, 256, (size_t)nbins * 4, s>>>(in, in_pitch, npix, c, inv_width, nbins, hist);
  return (int)cudaGetLastError();
}

size_t direct_weight_bytes_s8(int cin, int cout, int k) { return (size_t)cin * cout * k * k; }

void direct_pack_weights_s8(int cin, int cout, int k, const int8_t *w, void *dst_host) {
  int8_t *o = reinterpret_cast<int8_t *>(dst_host);
  const int taps = k * k;
  for (int t = 0; t < taps; ++t)
    for (int co = 0; co < cout; ++co)
      for (int ci = 0; ci < cin; ++ci) o[((size_t)t * cout + co) * cin + ci] = w[((size_t)co * cin + ci) * taps + t];
}

// depth-wise: [c][1][k][k] -> [tap][c]
void direct_pack_weights_s8_dw(int c, int k, const int8_t *w, void *dst_host) {
  int8_t *o = reinterpret_cast<int8_t *>(dst_host);
  const int taps = k * k;
  for (int t = 0; t < taps; ++t)
    for (int ch = 0; ch < c; ++ch) o[(size_t)t * c + ch] = w[(size_t)ch * taps + t];
}

int direct_conv_s8_launch(const ConvArgs &a, const float *mult, float out_scale, int out_kind, cudaStream_t s) {
  UYD_REQUIRE(a.cin % 4 == 0 && a.in_pitch % 4 == 0 && (reinterpret_cast<uintptr_t>(a.in) & 3) == 0, UYD_E_UNSUPPORTED,
              "int8 direct conv needs cin %% 4 == 0 and 4-byte aligned input slices");
  const long long npix = (long long)a.n * a.oh * a.ow;
  const auto al8 = [](const void *q) { return (reinterpret_cast<uintptr_t>(q) & 7) == 0; };
  if (a.cin == 4 && a.cout == 4 && a.k == 3 && a.stride == 1 && (out_kind == 0 || out_kind == 3) && a.oh == a.ih && a.ow == a.iw &&
      npix < (1ll << 31) && npix * a.in_pitch < (1ll << 32) && a.out_pitch % 4 == 0 && (out_kind == 3 || al8(a.out)) &&
      (reinterpret_cast<uintptr_t>(a.out) & 3) == 0 && (!a.res || (a.res_pitch % 4 == 0 && al8(a.res)))) {
    if (out_kind == 3) conv_s8_c4_kernel<true><<<(unsigned)((npix + 255) / 256), 256, 0, s>>>(a, mult, out_scale);
    else conv_s8_c4_kernel<false><<<(unsigned)((npix + 255) / 256), 256, 0, s>>>(a, mult, out_scale);
    return (int)cudaGetLastError();
  }
  dim3 grid((unsigned)((npix + 127) / 128), (unsigned)ceil_div(a.cout, 4));
  conv_s8_direct_kernel<<<grid, 128, 0, s>>>(a, mult, out_scale, out_kind);
  return (int)cudaGetLastError();
}

int direct_conv_s8_dw_launch(const ConvArgs &a, const float *mult, float out_scale, int out_kind, cudaStream_t s) {
  UYD_REQUIRE(a.cin == a.cout && a.cin % 4 == 0 && a.in_pitch % 4 == 0 && (reinterpret_cast<uintptr_t>(a.in) & 3) == 0 && !a.res,
              UYD_E_UNSUPPORTED, "int8 depth-wise conv needs C %% 4 == 0, 4-byte aligned slices and no residual");
  const long long total = (long long)a.n * a.oh * a.ow * (a.cin / 4);
  conv_s8_dw_kernel<<<(unsigned)((total + 127) / 128), 128, 0, s>>>(a, mult, out_scale, out_kind);
  return (int)cudaGetLastError();
}

int quantize_s8_launch(const __nv_bfloat16 *in, int in_pitch, int8_t *out, int out_pitch, long long npix, int c, float scale,
                       cudaStream_t s) {
  UYD_REQUIRE(c % 4 == 0 && in_pitch % 4 == 0 && out_pitch % 4 == 0 && (reinterpret_cast<uintptr_t>(in) & 7) == 0 &&
                  (reinterpret_cast<uintptr_t>(out) & 3) == 0, UYD_E_UNSUPPORTED, "quantize: C %% 4 == 0 and aligned slices");
  if (c % 16 == 0 && in_pitch % 8 == 0 && out_pitch % 16 == 0 && (reinterpret_cast<uintptr_t>(in) & 15) == 0 &&
      (reinterpret_cast<uintptr_t>(out) & 15) == 0 && npix * (c / 16) < (1ll << 31)) {
    const unsigned total16 = (unsigned)(npix * (c / 16));
    quantize_s8_x16_kernel<<<(total16 + 1023u) / 1024u, 256, 0, s>>>(in, in_pitch, out, out_pitch, total16, c / 16, scale);
    return (int)cudaGetLastError();
  }
  const long long total = npix * (c / 4);
  quantize_s8_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(in, in_pitch, out, out_pitch, npix, c, scale);
  return (int)cudaGetLastError();
}

int absmax_launch(const __nv_bfloat16 *in, int in_pitch, long long npix, int c, unsigned int *out_bits, cudaStream_t s) {
  UYD_REQUIRE(c % 4 == 0 && in_pitch % 4 == 0 && (reinterpret_cast<uintptr_t>(in) & 7) == 0, UYD_E_UNSUPPORTED,
              "absmax: C %% 4 == 0 and 8-byte aligned slices");
  long long blocks = (npix * (c / 4) + 255) / 256;
  if (blocks > 148 * 8) blocks = 148 * 8;
  absmax_kernel<<<(unsigned)blocks, 256, 0, s>>>(in, in_pitch, npix, c, out_bits);
  return (int)cudaGetLastError();
}
}  // namespace uyd
