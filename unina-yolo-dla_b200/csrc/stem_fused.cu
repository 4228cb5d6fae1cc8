// Fused stem: model.0 Conv(3,16,3,2) + model.1 Conv(16,32,3,2) (unina-yolo-dla-m.yaml:24-25, both Conv+BN+ReLU, BN
// folded), optionally + model.2.cv1, in one launch.  Unfused, the 320x320x16 tensor between them costs 6.6 MB of HBM
// traffic per frame and a 16-channel layer cannot feed tcgen05 (32-byte TMA rows).  The design and the per-lane maps
// are in stem_v2.cuh, the camera-frame loaders (BGRA / NV12 read and normalised on load, SURVEY 8f-1) in camera.cuh;
// this file holds the kernel and the host side.  (The first-generation hi/lo-split kernel was removed after a round of soak.)
#include <type_traits>

#include "camera.cuh"
#include "stem_v2.cuh"

#include "common.cuh"

namespace uyd {

struct StemArgs {
  const void *in;      // NCHW frames, fp32 or uint8
  __nv_bfloat16 *out;  // NHWC slice base of image 0
  const uint32_t *wfrag;  // stemv2::pack fragments: [L0 | L1 | 1x1]
  const float *bias;      // [16 | 32]
  int n, ih, iw, oh, ow, out_pitch, u8;
  int pw;  // 1: the 1x1 Conv(32,16) follows in the same launch (second-generation kernel only); out has 16 channels
  // camera frames straight into the patch (f.cam != 0, camera.cuh); `in` = BGRA pixels / Y plane
  CamFrames f;
};

namespace stemv2 {
__device__ __forceinline__ void mma1688_tf32(float (&d)[4], const uint4 &a, uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void mma16816v(float (&d)[4], const uint4 &a, uint32_t b0, uint32_t b1) {
  asm volatile(
      "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
      : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
      : "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t movmatrix_trans(uint32_t v) {
  uint32_t r;
  asm volatile("movmatrix.sync.aligned.m8n8.trans.b16 %0, %1;" : "=r"(r) : "r"(v));
  return r;
}

// PERSIST: two CTAs per SM walk the tiles and keep the 18 layer-1 A fragments in registers (the per-tile re-read of
// those 9 KB by each of the eight warps is 576 of the ~3100 L1/shared wavefronts a tile costs, the kernel's bound).
template <typename TIn, bool PW, bool PERSIST>
__global__ void __launch_bounds__(stemv2::kThreads, PERSIST ? 2 : 3) stem_v2_kernel(StemArgs a) {
  pdl_trigger();
  extern __shared__ __align__(16) unsigned char smem[];
  unsigned char *patch = smem;                             // [3][38 lines: even rows at 0, odd rows at 20][68] fp32 (tf32)
  unsigned char *l0s = smem + kPatchBytes;                 // [584 pixels q = 34 y + x][48 B]: word w = channels (w, w+8)
  unsigned char *w1s = smem + kPatchBytes + kL0Bytes;      // layer-1 A fragments [tap][m-tile][lane] x 16 B (!PERSIST)

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t = lane & 3;
  uint4 w1r[PERSIST ? 18 : 1];
  if (PERSIST) {
#pragma unroll
    for (int i = 0; i < (PERSIST ? 18 : 0); ++i) w1r[i] = __ldg(reinterpret_cast<const uint4 *>(a.wfrag + kW0Words) + i * 32 + lane);
  }
  const int tiles_x = (a.ow + kTW - 1) / kTW, tiles_y = (a.oh + kTH - 1) / kTH;
  const int total_tiles = PERSIST ? tiles_x * tiles_y * a.n : 1;
  for (int tile = PERSIST ? (int)blockIdx.x : 0; tile < total_tiles; tile += PERSIST ? (int)gridDim.x : 1) {
  int ox0, oy0, n;
  if (PERSIST) {
    const int per = tiles_x * tiles_y, r = tile % per;
    n = tile / per; oy0 = (r / tiles_x) * kTH; ox0 = (r % tiles_x) * kTW;
  } else {
    ox0 = blockIdx.x * kTW; oy0 = blockIdx.y * kTH; n = blockIdx.z;
  }
  const int ix0 = 4 * ox0 - 4, iy0 = 4 * oy0 - 3;  // frame coordinates of the patch origin (16-byte aligned columns)

  // ---- all global loads first: layer-1 fragments and this thread's 7 patch vectors (column j, lines rl + 15 i) ----
  constexpr int kW1Vec = kW1Words / 4, kWIters = (kW1Vec + kThreads - 1) / kThreads;
  const uint4 *w1g = reinterpret_cast<const uint4 *>(a.wfrag + kW0Words);
  uint4 wv[kWIters];
#pragma unroll
  for (int it = 0; it < kWIters; ++it) {
    const int i = tid + it * kThreads;
    wv[it] = (!PERSIST && i < kW1Vec) ? __ldg(w1g + i) : make_uint4(0u, 0u, 0u, 0u);
  }
  // thread (pj, prl): column vector pj of patch rows prl, prl + 15 and (prl < 5) prl + 30 of each channel
  constexpr int kVecPerRow = kInW / 4, kRowLanes = 15;  // 17 vectors per row, 255 loading threads
  static_assert(2 * kRowLanes <= kInH && 3 * kRowLanes >= kInH && kRowLanes * kVecPerRow <= kThreads, "patch load map");
  constexpr bool kLetterbox = std::is_same<TIn, CamLetterboxIn>::value;
  constexpr bool kCam = std::is_same<TIn, CamIn>::value || kLetterbox;
  const TIn *img = reinterpret_cast<const TIn *>(a.in) + (kCam ? 0ll : (long long)n * 3 * a.ih * a.iw);
  asm volatile("" : "+l"(img));  // keep the per-load address arithmetic 32-bit: one IMAD.WIDE.U32 on this base
  const int pj = tid % kVecPerRow, prl = tid / kVecPerRow;
  const int ix = ix0 + 4 * pj;
  const bool col_ok = prl < kRowLanes && ix >= 0 && ix + 3 < a.iw;
  const unsigned plane = (unsigned)(a.ih * a.iw);
  bool ok[3];
  unsigned off[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int r = prl + kRowLanes * k, iy = iy0 + r;
    ok[k] = col_ok && r < kInH && (unsigned)iy < (unsigned)a.ih;
    off[k] = (unsigned)(iy * a.iw + ix);  // meaningful only when ok[k]
  }
  uint4 pv[3][3];
  if constexpr (kCam) {  // camera bytes -> normalised fp32 bit patterns of the four columns of every row this thread owns
    const uint8_t *frame = reinterpret_cast<const uint8_t *>(a.in) + (long long)n * a.f.frame_stride;
    const uint8_t *uvp = a.f.uv ? a.f.uv + (long long)n * a.f.uv_frame_stride : nullptr;
    const CamNorm nm = cam_norm(a.f);
    CamLetterbox lb;
    if constexpr (kLetterbox) lb = cam_letterbox(a, a.f);
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      float px[4][3];
#pragma unroll
      for (int j = 0; j < 4; ++j) px[j][0] = px[j][1] = px[j][2] = 0.f;
      if (ok[k]) {
        if constexpr (kLetterbox) cam_letterbox4(lb, a.f, nm, frame, iy0 + prl + kRowLanes * k, ix, px);
        else cam_row4(a, a.f, nm, frame, uvp, iy0 + prl + kRowLanes * k, ix, px);
      }
#pragma unroll
      for (int c = 0; c < 3; ++c)
        pv[c][k] = make_uint4(__float_as_uint(px[0][c]), __float_as_uint(px[1][c]), __float_as_uint(px[2][c]), __float_as_uint(px[3][c]));
    }
  } else {
#pragma unroll
  for (int c = 0; c < 3; ++c)
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      pv[c][k] = make_uint4(0u, 0u, 0u, 0u);
      if (ok[k]) {
        const TIn *src = img + (off[k] + c * plane);
        if (sizeof(TIn) == 4) pv[c][k] = __ldg(reinterpret_cast<const uint4 *>(src));
        else pv[c][k].x = __ldg(reinterpret_cast<const unsigned int *>(src));
      }
    }
  }
#pragma unroll
  for (int it = 0; it < kWIters; ++it) {
    const int i = tid + it * kThreads;
    if (!PERSIST && i < kW1Vec) reinterpret_cast<uint4 *>(w1s)[i] = wv[it];
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const int r = prl + kRowLanes * k;
    if (prl < kRowLanes && r < kInH) {
      unsigned char *dst = patch + (patch_line(0, r) * kInW + 4 * pj) * 4;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const uint4 v = pv[c][k];
        uint4 o;
        if (sizeof(TIn) == 4 || kCam) {  // round to nearest tf32: the mma reads the upper 19 bits
          o = ok[k] ? make_uint4(v.x + 0x1000u, v.y + 0x1000u, v.z + 0x1000u, v.w + 0x1000u) : v;
        } else {                 // x / 255 exactly as the float pre-process computes it, then the same rounding
          auto cv = [&](uint32_t b) { return ok[k] ? __float_as_uint(div255((float)b)) + 0x1000u : 0u; };
          o = make_uint4(cv(v.x & 0xffu), cv((v.x >> 8) & 0xffu), cv((v.x >> 16) & 0xffu), cv(v.x >> 24));
        }
        *reinterpret_cast<uint4 *>(dst + c * kChanLines * kInW * 4) = o;
      }
    }
  }
  __syncthreads();

  // ---- layer 0: 73 groups of 8 flat pixels, 16 channels = the 16 mma rows, mma.m16n8k8.tf32 ----
  {
    const uint4 *w0g = reinterpret_cast<const uint4 *>(a.wfrag);
    uint4 af[5];
#pragma unroll
    for (int s = 0; s < 5; ++s) af[s] = __ldg(w0g + s * 32 + lane);
    const float b_lo = __ldg(a.bias + g), b_hi = __ldg(a.bias + g + 8);
    const unsigned char *pb[5];
#pragma unroll
    for (int s = 0; s < 5; ++s)  // l0_k_off(s, t) from two compile-time constants
      pb[s] = patch + 64 * warp + 8 * g + 8 * (t & 1) + 4 * ((t >> 1) ? l0_k_off(s, 2) : l0_k_off(s, 0));
    unsigned char *sb = l0s + (8 * warp + 2 * t) * kL0Pitch + 4 * g;
    // groups warp + 8 i: pixels q = 8 (warp + 8 i) + (B: g | D: 2t, 2t+1); three independent mma chains at a time
    auto groups = [&](int i0, auto cnt) {
      constexpr int NG = decltype(cnt)::value;
      float acc[NG][4];
#pragma unroll
      for (int j = 0; j < NG; ++j) { acc[j][0] = acc[j][1] = b_lo; acc[j][2] = acc[j][3] = b_hi; }
#pragma unroll
      for (int s = 0; s < 5; ++s) {
        uint2 v[NG];
#pragma unroll
        for (int j = 0; j < NG; ++j) v[j] = ld64(pb[s] + 512 * (i0 + j));
#pragma unroll
        for (int j = 0; j < NG; ++j) mma1688_tf32(acc[j], af[s], v[j].x, v[j].y);
      }
#pragma unroll
      for (int j = 0; j < NG; ++j) {
        st32(sb + 64 * kL0Pitch * (i0 + j), relu_pack_bf16(acc[j][0], acc[j][2]));
        st32(sb + 64 * kL0Pitch * (i0 + j) + kL0Pitch, relu_pack_bf16(acc[j][1], acc[j][3]));
      }
    };
    static_assert(kGroups == 73, "nine groups per warp and one more for warp 0");
    groups(0, std::integral_constant<int, 3>{});
    groups(3, std::integral_constant<int, 3>{});
    groups(6, std::integral_constant<int, 3>{});
    if (warp == 0) groups(9, std::integral_constant<int, 1>{});
  }
  __syncthreads();
  // layer 1's zero padding: layer-0 row -1 / column -1 exist only in the tiles on the top / left image border
  if (oy0 == 0 || ox0 == 0) {
    if (oy0 == 0)
      for (int i = tid; i < kL0P * 8; i += kThreads) st32(l0s + (i >> 3) * kL0Pitch + 4 * (i & 7), 0u);
    if (ox0 == 0 && tid < kL0H * 8) st32(l0s + (tid >> 3) * kL0P * kL0Pitch + 4 * (tid & 7), 0u);
    __syncthreads();
  }

  // ---- layer 1: warp = output row oy0 + warp, two groups of 8 pixels x two 16-channel m-tiles, one tap per k-step ----
  {
    float acc[2][2][4];
#pragma unroll
    for (int mt = 0; mt < 2; ++mt) {
      const float2 bz = __ldg(reinterpret_cast<const float2 *>(a.bias + 16 + 4 * g + 2 * mt));
#pragma unroll
      for (int xg = 0; xg < 2; ++xg) { acc[xg][mt][0] = acc[xg][mt][1] = bz.x; acc[xg][mt][2] = acc[xg][mt][3] = bz.y; }
    }
    const unsigned char *bb = l0s + l1_b_off(warp, 0, g, t, 0);
    const uint4 *wf = reinterpret_cast<const uint4 *>(w1s) + lane;
#pragma unroll
    for (int tap = 0; tap < 9; ++tap) {
      const uint4 a0 = PERSIST ? w1r[PERSIST ? tap * 2 : 0] : wf[(tap * 2 + 0) * 32], a1 = PERSIST ? w1r[PERSIST ? tap * 2 + 1 : 0] : wf[(tap * 2 + 1) * 32];
#pragma unroll
      for (int xg = 0; xg < 2; ++xg) {
        const uint2 b = ld64(bb + ((tap / 3) * kL0P + 16 * xg + tap % 3) * kL0Pitch);
        mma16816v(acc[xg][0], a0, b.x, b.y);
        mma16816v(acc[xg][1], a1, b.x, b.y);
      }
    }
    const int oy = oy0 + warp;
    __nv_bfloat16 *orow = a.out + ((long long)n * a.oh + oy) * a.ow * a.out_pitch;
    if (!PW) {
#pragma unroll
      for (int xg = 0; xg < 2; ++xg)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int px = ox0 + 8 * xg + 2 * t + h;
          if (oy < a.oh && px < a.ow)
            *reinterpret_cast<uint2 *>(orow + (long long)px * a.out_pitch + 4 * g) =
                make_uint2(relu_pack_bf16(acc[xg][0][h], acc[xg][0][2 + h]), relu_pack_bf16(acc[xg][1][h], acc[xg][1][2 + h]));
        }
    } else {
      // 1x1 conv on the bf16-rounded layer-1 output: (channel x pixel) accumulator tiles -> movmatrix -> B fragments
      const uint4 *w2 = reinterpret_cast<const uint4 *>(a.wfrag + kW0Words + kW1Words) + lane;
      const uint4 p0 = __ldg(w2), p1 = __ldg(w2 + 32);
      const float2 bz = __ldg(reinterpret_cast<const float2 *>(a.bias + 48 + 2 * g));
#pragma unroll
      for (int xg = 0; xg < 2; ++xg) {
        float acc2[4] = {bz.x, bz.x, bz.y, bz.y};
        uint32_t bq[2][2];
#pragma unroll
        for (int mt = 0; mt < 2; ++mt)
#pragma unroll
          for (int hh = 0; hh < 2; ++hh) bq[mt][hh] = movmatrix_trans(relu_pack_bf16(acc[xg][mt][2 * hh], acc[xg][mt][2 * hh + 1]));
        mma16816v(acc2, p0, bq[0][0], bq[0][1]);
        mma16816v(acc2, p1, bq[1][0], bq[1][1]);
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int px = ox0 + 8 * xg + 2 * t + h;
          if (oy < a.oh && px < a.ow)
            *reinterpret_cast<uint32_t *>(orow + (long long)px * a.out_pitch + 2 * g) = relu_pack_bf16(acc2[h], acc2[2 + h]);
        }
      }
    }
  }
  }  // tile loop
}
}  // namespace stemv2
bool stem_fused_supported(int c0, int c1, int ih, int iw, int out_pitch, int out_coff) {
  return c0 == 16 && c1 == 32 && ih % 4 == 0 && iw % 4 == 0 && out_pitch % 8 == 0 && out_coff % 8 == 0;
}

// w0 [16][3][3][3], w1 [32][16][3][3] (BN folded, PyTorch layout)
// frags = stem_v2.cuh fragments, bias = [16 | 32 | 16 (1x1, zero without w2)]
void stem_fused_pack(const float *w0, const float *b0, const float *w1, const float *b1, const float *w2, const float *b2,
                     std::vector<uint32_t> &frags, std::vector<float> &bias) {
  frags.clear();
  bias.assign(64, 0.f);
  for (int i = 0; i < 16; ++i) bias[i] = b0[i];
  for (int i = 0; i < 32; ++i) bias[16 + i] = b1[i];
  for (int i = 0; i < 16 && b2; ++i) bias[48 + i] = b2[i];
  stemv2::pack(w0, w1, w2, frags);
}

static int stem_v2_launch(const StemArgs &a0, cudaStream_t s) {
  StemArgs a = a0;
  static const bool persist = [] { const char *v = getenv("UYD_STEM_PERSIST"); return !(v && *v == '0'); }();
  const int sms = current_sm_count();
  UYD_REQUIRE(sms > 0, UYD_E_NOGPU, "stem: no current CUDA device");
  const int tiles = ceil_div(a.ow, stemv2::kTW) * ceil_div(a.oh, stemv2::kTH) * a.n;
  const size_t smem = stemv2::kSmemBytes;
  auto go = [&](auto kern, bool pers) -> int {
    if (int e = smem_optin(kern, stemv2::kSmemBytes)) return e;
    if (pers) kern<<<tiles < 2 * sms ? tiles : 2 * sms, stemv2::kThreads, smem, s>>>(a);
    else kern<<<dim3(ceil_div(a.ow, stemv2::kTW), ceil_div(a.oh, stemv2::kTH), a.n), stemv2::kThreads, smem, s>>>(a);
    return (int)cudaGetLastError();
  };
  // persistent CTAs pay off once there are several tiles per CTA (batch-1 frames keep one tile per CTA)
  const bool pers = persist && tiles >= 8 * sms;
  using namespace stemv2;
  if (a.f.cam == UYD_CAM_BGRA_LETTERBOX) {
    if (a.pw) return pers ? go(stem_v2_kernel<CamLetterboxIn, true, true>, true) : go(stem_v2_kernel<CamLetterboxIn, true, false>, false);
    return pers ? go(stem_v2_kernel<CamLetterboxIn, false, true>, true) : go(stem_v2_kernel<CamLetterboxIn, false, false>, false);
  }
  if (a.f.cam) {
    if (a.pw) return pers ? go(stem_v2_kernel<CamIn, true, true>, true) : go(stem_v2_kernel<CamIn, true, false>, false);
    return pers ? go(stem_v2_kernel<CamIn, false, true>, true) : go(stem_v2_kernel<CamIn, false, false>, false);
  }
  if (a.u8) {
    if (a.pw) return pers ? go(stem_v2_kernel<uint8_t, true, true>, true) : go(stem_v2_kernel<uint8_t, true, false>, false);
    return pers ? go(stem_v2_kernel<uint8_t, false, true>, true) : go(stem_v2_kernel<uint8_t, false, false>, false);
  }
  if (a.pw) return pers ? go(stem_v2_kernel<float, true, true>, true) : go(stem_v2_kernel<float, true, false>, false);
  return pers ? go(stem_v2_kernel<float, false, true>, true) : go(stem_v2_kernel<float, false, false>, false);
}

int stem_fused_launch(const StemArgs &a, cudaStream_t s) { return stem_v2_launch(a, s); }

}  // namespace uyd
