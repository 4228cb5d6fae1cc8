// Camera frames read straight into a stem's input patch (SURVEY 8f-1: no CHW fp32 tensor in HBM).  Shared by the YAML
// network's fused stem (stem_fused.cu) and model.py's mma stem (conv_direct.cu), so both normalise and resample the
// same way: semantics of cuda_preprocess.cu:99-253.
#pragma once
#include "stem_v2.cuh"  // stemv2::div255

namespace uyd {

// The frame fields of uyd_camera_frames a stem kernel reads (by value, in the kernel's parameters).
// cam = 1 packed BGRA (bilinear resize when the frame extent differs from the network input), 2 = NV12, 3 = packed
// BGRA letterboxed (CamLetterboxIn instantiations, below);
// the BGRA pixels / the Y plane are the kernel's input pointer.
struct CamFrames {
  int cam, src_w, src_h, src_pitch, uv_pitch;
  long long frame_stride, uv_frame_stride;
  const uint8_t *uv;
  float mean[3], stdv[3];  // r, g, b
};

struct CamIn {};  // TIn tag of the camera instantiations of the stem kernels

// Camera frames -> normalised model-input values: ((v / 255) - mean) / std, BGRA bilinear taps with the half-pixel
// rule, BT.601 NV12.  v / 255 is q = v * r corrected by one FMA step (the IEEE quotient for every integer v,
// stemv2::div255; within an ulp otherwise); the mean / std step is skipped for the unit normalisation the YAML model is
// fed with and uses an IEEE division otherwise, so that a BGRA frame of the model's extent gives bit-identical results
// to the reference kernel's tensor.
struct CamNorm {
  float mean[3], stdv[3];
  bool unit;
  __device__ __forceinline__ float operator()(float v, int c) const {
    const float q = stemv2::div255(v);
    return unit ? q : __fdiv_rn(__fsub_rn(q, mean[c]), stdv[c]);
  }
};

__device__ __forceinline__ CamNorm cam_norm(const CamFrames &f) {
  CamNorm nm;
#pragma unroll
  for (int c = 0; c < 3; ++c) { nm.mean[c] = f.mean[c]; nm.stdv[c] = f.stdv[c]; }
  nm.unit = f.mean[0] == 0.f && f.mean[1] == 0.f && f.mean[2] == 0.f && f.stdv[0] == 1.f && f.stdv[1] == 1.f && f.stdv[2] == 1.f;
  return nm;
}

// The raw bytes of four horizontally adjacent model-input pixels (iy, ix .. ix + 3), ix % 4 == 0, and their conversion.
// NV12: 4 luma bytes + 2 (U, V) pairs = two 32-bit loads when the planes are 4-byte aligned; (y4, uv4, -, -)
__device__ __forceinline__ uint4 cam_load_nv12(const CamFrames &f, const uint8_t *frame, const uint8_t *uvp, int iy, int ix) {
  const uint8_t *yr = frame + (long long)iy * f.src_pitch + ix;
  const uint8_t *ur = uvp + (long long)(iy / 2) * f.uv_pitch + ix;
  uint32_t y4, uv4;
  if (((f.src_pitch | f.uv_pitch) & 3) == 0 && ((reinterpret_cast<uintptr_t>(frame) | reinterpret_cast<uintptr_t>(uvp)) & 3) == 0) {
    y4 = *reinterpret_cast<const uint32_t *>(yr);
    uv4 = *reinterpret_cast<const uint32_t *>(ur);
  } else {
    y4 = yr[0] | (yr[1] << 8) | (yr[2] << 16) | ((uint32_t)yr[3] << 24);
    uv4 = ur[0] | (ur[1] << 8) | (ur[2] << 16) | ((uint32_t)ur[3] << 24);
  }
  return make_uint4(y4, uv4, 0u, 0u);
}
__device__ __forceinline__ void cam_convert_nv12(const CamNorm &nm, const uint4 &v, float (&px)[4][3]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float Y = (float)((v.x >> (8 * j)) & 0xFF);
    const float U = (float)((v.y >> (16 * (j >> 1))) & 0xFF) - 128.0f, V = (float)((v.y >> (16 * (j >> 1) + 8)) & 0xFF) - 128.0f;
    float r = Y + 1.402f * V, g = Y - 0.344136f * U - 0.714136f * V, b = Y + 1.772f * U;
    r = fmaxf(0.0f, fminf(255.0f, r)); g = fmaxf(0.0f, fminf(255.0f, g)); b = fmaxf(0.0f, fminf(255.0f, b));
    px[j][0] = nm(r, 0); px[j][1] = nm(g, 1); px[j][2] = nm(b, 2);
  }
}
// BGRA at the model's extent: one pixel = one 32-bit word; one 16-byte load when pitch, frame stride and base are
// 16-byte aligned, else four 4-byte loads
__device__ __forceinline__ void cam_load_bgra(const CamFrames &f, const uint8_t *frame, int iy, int ix, uint32_t (&w)[4]) {
  const uint32_t *q = reinterpret_cast<const uint32_t *>(frame + (long long)iy * f.src_pitch + 4 * ix);
  if (((f.src_pitch | (int)(f.frame_stride & 15)) & 15) == 0 && (reinterpret_cast<uintptr_t>(frame) & 15) == 0) {
    const uint4 v = *reinterpret_cast<const uint4 *>(q);
    w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
  } else {
#pragma unroll
    for (int j = 0; j < 4; ++j) w[j] = q[j];
  }
}
__device__ __forceinline__ void cam_convert_bgra(const CamNorm &nm, const uint32_t (&w)[4], float (&px)[4][3]) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    px[j][0] = nm((float)((w[j] >> 16) & 0xFF), 0);
    px[j][1] = nm((float)((w[j] >> 8) & 0xFF), 1);
    px[j][2] = nm((float)(w[j] & 0xFF), 2);
  }
}

// BGRA + bilinear resize to the model's extent (m.ih x m.iw): the row terms once, four taps of 32-bit pixels per output
// pixel.  M: the kernel's argument struct (StemArgs, ConvArgs); the extent is read through it, in place.
template <class M>
__device__ __forceinline__ void cam_resize4(const M &m, const CamFrames &f, const CamNorm &nm, const uint8_t *frame, int iy, int ix,
                                            float (&px)[4][3]) {
  const float ratio_x = (float)f.src_w / m.iw, ratio_y = (float)f.src_h / m.ih;
  const float sy = fmaxf(0.0f, fminf((iy + 0.5f) * ratio_y - 0.5f, f.src_h - 1.0f));
  const int ya = (int)sy, yb = min(ya + 1, f.src_h - 1);
  const float fy = sy - ya;
  const uint8_t *ra = frame + (long long)ya * f.src_pitch, *rb = frame + (long long)yb * f.src_pitch;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const float sx = fmaxf(0.0f, fminf((ix + j + 0.5f) * ratio_x - 0.5f, f.src_w - 1.0f));
    const int xa = (int)sx, xb = min(xa + 1, f.src_w - 1);
    const float fx = sx - xa;
    const float waa = (1.0f - fx) * (1.0f - fy), wab = fx * (1.0f - fy), wba = (1.0f - fx) * fy, wbb = fx * fy;
    const uint32_t paa = *reinterpret_cast<const uint32_t *>(ra + 4 * xa), pab = *reinterpret_cast<const uint32_t *>(ra + 4 * xb);
    const uint32_t pba = *reinterpret_cast<const uint32_t *>(rb + 4 * xa), pbb = *reinterpret_cast<const uint32_t *>(rb + 4 * xb);
    auto mix = [&](int sh) {
      return waa * (float)((paa >> sh) & 0xFF) + wab * (float)((pab >> sh) & 0xFF) + wba * (float)((pba >> sh) & 0xFF) +
             wbb * (float)((pbb >> sh) & 0xFF);
    };
    px[j][0] = nm(mix(16), 0); px[j][1] = nm(mix(8), 1); px[j][2] = nm(mix(0), 2);
  }
}

// ---- BGRA letterboxed into the model input (f.cam == UYD_CAM_BGRA_LETTERBOX): the Ultralytics predictor's
// LetterBox(center=True, scaleup=True), i.e. cv2.resize(INTER_LINEAR) of the frame to (new_w, new_h), placed at
// (top, left), byte 114 around it.  The stem sees the numbers a uint8 tensor of the cv2-letterboxed frame gives.
struct CamLetterboxIn {};  // TIn tag of the letterboxing instantiations of the stem kernels

// The geometry of a src_w x src_h frame in a dst_w x dst_h model input, shared by the loader, uyd_letterbox_boxes and
// uyd_letterbox_geometry: r = min(dst_h / src_h, dst_w / src_w), new = round(src * r), pad = round((dst - new) / 2 - 0.1),
// Python's half-to-even round being nearbyint (1280 x 725 -> new_h = round(362.5) = 362).  gain = r (scale_boxes).
struct LetterboxGeom {
  int new_w, new_h, left, top;
  double gain;
};
__host__ __device__ inline LetterboxGeom letterbox_geometry(int src_w, int src_h, int dst_w, int dst_h) {
  const double r = fmin((double)dst_h / src_h, (double)dst_w / src_w);
  LetterboxGeom g;
  g.new_w = (int)nearbyint(src_w * r);
  g.new_h = (int)nearbyint(src_h * r);
  g.left = (int)nearbyint((dst_w - g.new_w) / 2.0 - 0.1);
  g.top = (int)nearbyint((dst_h - g.new_h) / 2.0 - 0.1);
  g.gain = r;
  return g;
}

// the geometry and cv2's source step per axis, scale = 1 / (new / src) in double, once per thread
struct CamLetterbox {
  LetterboxGeom g;
  double scale_x, scale_y;
};
template <class M>
__device__ __forceinline__ CamLetterbox cam_letterbox(const M &m, const CamFrames &f) {
  CamLetterbox lb;
  lb.g = letterbox_geometry(f.src_w, f.src_h, m.iw, m.ih);
  lb.scale_x = 1.0 / ((double)lb.g.new_w / f.src_w);
  lb.scale_y = 1.0 / ((double)lb.g.new_h / f.src_h);
  return lb;
}

// cv2 4.x INTER_LINEAR for uint8, output index d: f = (float)((d + 0.5) scale - 0.5), s = floor(f), f -= s; 11-bit
// weights rint((1 - f) 2048), rint(f 2048); source indices s, s + 1 clamped to [0, src).  The horizontal pass also
// zeroes the weight where s falls outside [0, src - 1); the vertical pass does not.  _rn intrinsics: no contraction.
struct CamTap {
  int s0, s1, w0, w1;
};
__device__ __forceinline__ CamTap cam_lin_tap(int d, double scale, int src, bool clamp_weight) {
  float f = (float)__dsub_rn(__dmul_rn((double)d + 0.5, scale), 0.5);
  int s = (int)floorf(f);
  f = __fsub_rn(f, (float)s);
  if (clamp_weight) {
    if (s < 0) { f = 0.f; s = 0; }
    if (s >= src - 1) { f = 0.f; s = src - 1; }
  }
  CamTap t;
  t.s0 = min(max(s, 0), src - 1);
  t.s1 = min(max(s + 1, 0), src - 1);
  t.w0 = __float2int_rn(__fmul_rn(__fsub_rn(1.f, f), 2048.f));
  t.w1 = __float2int_rn(__fmul_rn(f, 2048.f));
  return t;
}

// four horizontally adjacent model-input pixels (iy, ix .. ix + 3): 114 in the pad, else the two passes with cv2's SIMD
// vertical rounding (((b0 (h0 >> 4)) >> 16) + ((b1 (h1 >> 4)) >> 16) + 2) >> 2.  An exact 2x downscale, where cv2
// switches to INTER_AREA, gives weights 1024 / 1024 on the 2x2 block here: (a + b + c + d + 2) >> 2 as AREA; a frame
// already of extent (new_w, new_h) gives weights 2048 / 0: a copy.
__device__ __forceinline__ void cam_letterbox4(const CamLetterbox &lb, const CamFrames &f, const CamNorm &nm, const uint8_t *frame,
                                               int iy, int ix, float (&px)[4][3]) {
  const int y = iy - lb.g.top;
  const bool row_in = y >= 0 && y < lb.g.new_h;
  CamTap ty{};
  if (row_in) ty = cam_lin_tap(y, lb.scale_y, f.src_h, false);
  const uint8_t *ra = frame + (long long)ty.s0 * f.src_pitch, *rb = frame + (long long)ty.s1 * f.src_pitch;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int x = ix + j - lb.g.left;
    int v[3] = {114, 114, 114};
    if (row_in && x >= 0 && x < lb.g.new_w) {
      const CamTap tx = cam_lin_tap(x, lb.scale_x, f.src_w, true);
      const uint32_t paa = *reinterpret_cast<const uint32_t *>(ra + 4 * tx.s0), pab = *reinterpret_cast<const uint32_t *>(ra + 4 * tx.s1);
      const uint32_t pba = *reinterpret_cast<const uint32_t *>(rb + 4 * tx.s0), pbb = *reinterpret_cast<const uint32_t *>(rb + 4 * tx.s1);
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const int sh = 16 - 8 * c;  // R, G, B = bytes 2, 1, 0
        const int h0 = (int)((paa >> sh) & 0xFF) * tx.w0 + (int)((pab >> sh) & 0xFF) * tx.w1;
        const int h1 = (int)((pba >> sh) & 0xFF) * tx.w0 + (int)((pbb >> sh) & 0xFF) * tx.w1;
        v[c] = (((ty.w0 * (h0 >> 4)) >> 16) + ((ty.w1 * (h1 >> 4)) >> 16) + 2) >> 2;
      }
    }
    px[j][0] = nm((float)v[0], 0); px[j][1] = nm((float)v[1], 1); px[j][2] = nm((float)v[2], 2);
  }
}

// whether the frames are resampled (BGRA of another extent than the model's) or read by cam_load4 / cam_convert4
template <class M>
__device__ __forceinline__ bool cam_resampled(const M &m, const CamFrames &f) { return f.cam != 2 && !(f.src_w == m.iw && f.src_h == m.ih); }

// NV12 / BGRA at the model's extent, split into the loads and the arithmetic so that a kernel can issue the loads of a
// later tile early and keep 4 registers per 4 pixels in flight
__device__ __forceinline__ void cam_load4(const CamFrames &f, const uint8_t *frame, const uint8_t *uvp, int iy, int ix, uint32_t (&w)[4]) {
  if (f.cam == 2) {
    const uint4 v = cam_load_nv12(f, frame, uvp, iy, ix);
    w[0] = v.x; w[1] = v.y; w[2] = w[3] = 0u;
  } else {
    cam_load_bgra(f, frame, iy, ix, w);
  }
}
__device__ __forceinline__ void cam_convert4(const CamFrames &f, const CamNorm &nm, const uint32_t (&w)[4], float (&px)[4][3]) {
  if (f.cam == 2) cam_convert_nv12(nm, make_uint4(w[0], w[1], 0u, 0u), px);
  else cam_convert_bgra(nm, w, px);
}

// four horizontally adjacent model-input pixels (iy, ix .. ix + 3), ix % 4 == 0, loaded and converted in one go
template <class M>
__device__ __forceinline__ void cam_row4(const M &m, const CamFrames &f, const CamNorm &nm, const uint8_t *frame, const uint8_t *uvp,
                                         int iy, int ix, float (&px)[4][3]) {
  if (f.cam == 2) cam_convert_nv12(nm, cam_load_nv12(f, frame, uvp, iy, ix), px);
  else if (f.src_w == m.iw && f.src_h == m.ih) {
    uint32_t w[4];
    cam_load_bgra(f, frame, iy, ix, w);
    cam_convert_bgra(nm, w, px);
  }
  else cam_resize4(m, f, nm, frame, iy, ix, px);
}

}  // namespace uyd
