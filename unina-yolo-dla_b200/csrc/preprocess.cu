// Camera-frame pre-processing in front of model.0 (SURVEY.md section 8f row 1): packed BGRA / NV12 bytes ->
// RGB, (x / 255 - mean) / std, planar CHW fp32 -- the tensor uyd_plan_run consumes.  Drop-in for the
// reference's extern "C" entry points (ros2_ws/src/perception/include/cuda_preprocess.h:62-84, kernels
// cuda_preprocess.cu:99-253): same argument meaning, same arithmetic expression by expression (half-pixel
// bilinear sampling with clamped coordinates, BT.601 NV12 conversion), plus a batch dimension so that one
// launch feeds a whole plan batch.
//
// HBM-bound byte work: the no-resize kernels move 4 pixels per thread (one 16-byte BGRA load, three 16-byte
// plane stores); the resize kernel gathers four 4-byte pixels per output pixel.
#include "camera.cuh"  // letterbox_geometry
#include "common.cuh"

namespace uyd {
namespace {

__device__ __forceinline__ float norm1(float v, float mean, float stdv) { return ((v / 255.0f) - mean) / stdv; }

// 4 pixels per thread; requires width % 4 == 0, pitch % 16 == 0 and 16-byte aligned frames
__global__ void __launch_bounds__(256) bgra_vec4_kernel(const uint8_t *__restrict__ in, float *__restrict__ out, int width,
                                                        int height, int pitch, long long in_frame_stride, uyd_norm_params p) {
  const int x4 = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, n = blockIdx.z;
  if (x4 * 4 >= width) return;
  const uint4 q = *reinterpret_cast<const uint4 *>(in + n * in_frame_stride + (long long)y * pitch + x4 * 16);
  const uint32_t px[4] = {q.x, q.y, q.z, q.w};
  float r[4], g[4], b[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    b[i] = norm1((float)(px[i] & 0xFF), p.mean_b, p.std_b);
    g[i] = norm1((float)((px[i] >> 8) & 0xFF), p.mean_g, p.std_g);
    r[i] = norm1((float)((px[i] >> 16) & 0xFF), p.mean_r, p.std_r);
  }
  const long long plane = (long long)width * height;
  float *o = out + (long long)n * 3 * plane + (long long)y * width + x4 * 4;
  *reinterpret_cast<float4 *>(o) = make_float4(r[0], r[1], r[2], r[3]);
  *reinterpret_cast<float4 *>(o + plane) = make_float4(g[0], g[1], g[2], g[3]);
  *reinterpret_cast<float4 *>(o + 2 * plane) = make_float4(b[0], b[1], b[2], b[3]);
}

__global__ void __launch_bounds__(256) bgra_scalar_kernel(const uint8_t *__restrict__ in, float *__restrict__ out, int width,
                                                          int height, int pitch, long long in_frame_stride, uyd_norm_params p) {
  const int x = blockIdx.x * blockDim.x + threadIdx.x, y = blockIdx.y, n = blockIdx.z;
  if (x >= width) return;
  const uint8_t *px = in + n * in_frame_stride + (long long)y * pitch + x * 4;
  const long long plane = (long long)width * height;
  float *o = out + (long long)n * 3 * plane + (long long)y * width + x;
  o[0] = norm1((float)px[2], p.mean_r, p.std_r);
  o[plane] = norm1((float)px[1], p.mean_g, p.std_g);
  o[2 * plane] = norm1((float)px[0], p.mean_b, p.std_b);
}

// Half-pixel bilinear resize + normalise (semantics of cuda_preprocess.cu:140-199: sample position
// (d + 0.5) * src/dst - 0.5 clamped to the image, the four neighbours weighted (1-fx)(1-fy), fx(1-fy), (1-fx)fy, fx*fy).
// One thread owns PX horizontally adjacent output pixels of one row: the row terms (source rows, fy) are computed
// once, every source pixel is ONE 32-bit load (B | G<<8 | R<<16 | A<<24) instead of three byte loads per tap, and
// the three planes are written with one 16-byte store each (PX == 4) -- the fp32 CHW write is the HBM cost here.
template <int PX>
__global__ void __launch_bounds__(128) bgra_resize_kernel(const uint8_t *__restrict__ in, float *__restrict__ out, int sw, int sh,
                                                          int spitch, int dw, int dh, long long in_frame_stride,
                                                          uyd_norm_params p) {
  const int xq = (blockIdx.x * blockDim.x + threadIdx.x) * PX, dy = blockIdx.y, n = blockIdx.z;
  if (xq >= dw) return;
  const uint8_t *frame = in + n * in_frame_stride;
  const float ratio_x = (float)sw / dw, ratio_y = (float)sh / dh;
  const float sy = fmaxf(0.0f, fminf((dy + 0.5f) * ratio_y - 0.5f, sh - 1.0f));
  const int ya = (int)sy, yb = min(ya + 1, sh - 1);
  const float fy = sy - ya, gy = 1.0f - fy;
  const uint8_t *row_a = frame + (long long)ya * spitch, *row_b = frame + (long long)yb * spitch;
  float r[PX], g[PX], b[PX];
#pragma unroll
  for (int i = 0; i < PX; ++i) {
    const float sx = fmaxf(0.0f, fminf((xq + i + 0.5f) * ratio_x - 0.5f, sw - 1.0f));
    const int xa = (int)sx, xb = min(xa + 1, sw - 1);
    const float fx = sx - xa, gx = 1.0f - fx;
    const uint32_t paa = *reinterpret_cast<const uint32_t *>(row_a + 4 * xa), pab = *reinterpret_cast<const uint32_t *>(row_a + 4 * xb);
    const uint32_t pba = *reinterpret_cast<const uint32_t *>(row_b + 4 * xa), pbb = *reinterpret_cast<const uint32_t *>(row_b + 4 * xb);
    const float waa = gx * gy, wab = fx * gy, wba = gx * fy, wbb = fx * fy;
    auto mix = [&](int shift) {
      return waa * (float)((paa >> shift) & 0xFF) + wab * (float)((pab >> shift) & 0xFF) + wba * (float)((pba >> shift) & 0xFF) +
             wbb * (float)((pbb >> shift) & 0xFF);
    };
    r[i] = norm1(mix(16), p.mean_r, p.std_r);
    g[i] = norm1(mix(8), p.mean_g, p.std_g);
    b[i] = norm1(mix(0), p.mean_b, p.std_b);
  }
  const long long plane = (long long)dw * dh;
  float *o = out + (long long)n * 3 * plane + (long long)dy * dw + xq;
  if (PX == 4) {
    *reinterpret_cast<float4 *>(o) = make_float4(r[0], r[1], r[2], r[3]);
    *reinterpret_cast<float4 *>(o + plane) = make_float4(g[0], g[1], g[2], g[3]);
    *reinterpret_cast<float4 *>(o + 2 * plane) = make_float4(b[0], b[1], b[2], b[3]);
  } else {
    o[0] = r[0]; o[plane] = g[0]; o[2 * plane] = b[0];
  }
}

// NV12 (BT.601, cuda_preprocess.cu:207-253): one thread = two horizontally adjacent pixels sharing a UV pair
__global__ void __launch_bounds__(256) nv12_kernel(const uint8_t *__restrict__ y_plane, const uint8_t *__restrict__ uv_plane,
                                                   float *__restrict__ out, int width, int height, int y_pitch, int uv_pitch,
                                                   uyd_norm_params p) {
  const int x2 = blockIdx.x * blockDim.x + threadIdx.x, yc = blockIdx.y;
  if (x2 * 2 >= width) return;
  const long long uv_idx = (long long)(yc / 2) * uv_pitch + x2 * 2;
  const float U = uv_plane[uv_idx + 0] - 128.0f;
  const float V = uv_plane[uv_idx + 1] - 128.0f;
  const long long plane = (long long)width * height;
#pragma unroll
  for (int i = 0; i < 2; ++i) {
    const int x = x2 * 2 + i;
    if (x >= width) break;
    const float Y = y_plane[(long long)yc * y_pitch + x];
    float r = Y + 1.402f * V;
    float g = Y - 0.344136f * U - 0.714136f * V;
    float b = Y + 1.772f * U;
    r = fmaxf(0.0f, fminf(255.0f, r));
    g = fmaxf(0.0f, fminf(255.0f, g));
    b = fmaxf(0.0f, fminf(255.0f, b));
    float *o = out + (long long)yc * width + x;
    o[0] = norm1(r, p.mean_r, p.std_r);
    o[plane] = norm1(g, p.mean_g, p.std_g);
    o[2 * plane] = norm1(b, p.mean_b, p.std_b);
  }
}

}  // namespace
}  // namespace uyd

extern "C" uyd_norm_params uyd_norm_params_imagenet(void) {
  uyd_norm_params p = {0.485f, 0.456f, 0.406f, 0.229f, 0.224f, 0.225f};  // NormParams() default, cuda_preprocess.cu:64-66
  return p;
}

extern "C" uyd_norm_params uyd_norm_params_unit(void) {
  uyd_norm_params p = {0.f, 0.f, 0.f, 1.f, 1.f, 1.f};  // plain x / 255: what the Ultralytics predictor feeds the YAML model
  return p;
}

extern "C" int uyd_preprocess_bgra_batch(const uint8_t *d_input, float *d_output, int batch, long long frame_stride, int width,
                                         int height, int pitch, uyd_norm_params params, uyd_stream stream) {
  UYD_REQUIRE(d_input && d_output && batch > 0 && width > 0 && height > 0 && pitch >= width * 4, UYD_E_ARG,
              "uyd_preprocess_bgra: bad arguments");
  cudaStream_t s = (cudaStream_t)stream;
  const bool vec = width % 4 == 0 && pitch % 16 == 0 && frame_stride % 16 == 0 && (reinterpret_cast<uintptr_t>(d_input) & 15) == 0 &&
                   (reinterpret_cast<uintptr_t>(d_output) & 15) == 0;
  if (vec) {
    dim3 grid(uyd::ceil_div(width / 4, 256), height, batch);
    uyd::bgra_vec4_kernel<<<grid, 256, 0, s>>>(d_input, d_output, width, height, pitch, frame_stride, params);
  } else {
    dim3 grid(uyd::ceil_div(width, 256), height, batch);
    uyd::bgra_scalar_kernel<<<grid, 256, 0, s>>>(d_input, d_output, width, height, pitch, frame_stride, params);
  }
  return (int)cudaGetLastError();
}

extern "C" int uyd_preprocess_bgra(const uint8_t *d_input, float *d_output, int width, int height, int pitch,
                                   uyd_norm_params params, uyd_stream stream) {
  return uyd_preprocess_bgra_batch(d_input, d_output, 1, 0, width, height, pitch, params, stream);
}

extern "C" int uyd_preprocess_bgra_resize_batch(const uint8_t *d_input, float *d_output, int batch, long long frame_stride,
                                                int src_width, int src_height, int src_pitch, int dst_width, int dst_height,
                                                uyd_norm_params params, uyd_stream stream) {
  UYD_REQUIRE(d_input && d_output && batch > 0 && src_width > 0 && src_height > 0 && dst_width > 0 && dst_height > 0 &&
                  src_pitch >= src_width * 4, UYD_E_ARG, "uyd_preprocess_bgra_resize: bad arguments");
  UYD_REQUIRE(src_pitch % 4 == 0 && frame_stride % 4 == 0 && (reinterpret_cast<uintptr_t>(d_input) & 3) == 0, UYD_E_UNSUPPORTED,
              "uyd_preprocess_bgra_resize: BGRA pixels must be 4-byte aligned (pitch %% 4 == 0)");
  const bool vec = dst_width % 4 == 0 && (reinterpret_cast<uintptr_t>(d_output) & 15) == 0;
  if (vec) {
    dim3 grid(uyd::ceil_div(dst_width / 4, 128), dst_height, batch);
    uyd::bgra_resize_kernel<4><<<grid, 128, 0, (cudaStream_t)stream>>>(d_input, d_output, src_width, src_height, src_pitch,
                                                                       dst_width, dst_height, frame_stride, params);
  } else {
    dim3 grid(uyd::ceil_div(dst_width, 128), dst_height, batch);
    uyd::bgra_resize_kernel<1><<<grid, 128, 0, (cudaStream_t)stream>>>(d_input, d_output, src_width, src_height, src_pitch,
                                                                       dst_width, dst_height, frame_stride, params);
  }
  return (int)cudaGetLastError();
}

extern "C" int uyd_preprocess_bgra_resize(const uint8_t *d_input, float *d_output, int src_width, int src_height, int src_pitch,
                                          int dst_width, int dst_height, uyd_norm_params params, uyd_stream stream) {
  return uyd_preprocess_bgra_resize_batch(d_input, d_output, 1, 0, src_width, src_height, src_pitch, dst_width, dst_height, params,
                                          stream);
}

extern "C" int uyd_preprocess_nv12(const uint8_t *d_y_plane, const uint8_t *d_uv_plane, float *d_output, int width, int height,
                                   int y_pitch, int uv_pitch, uyd_norm_params params, uyd_stream stream) {
  UYD_REQUIRE(d_y_plane && d_uv_plane && d_output && width > 0 && height > 0 && y_pitch >= width && uv_pitch >= width, UYD_E_ARG,
              "uyd_preprocess_nv12: bad arguments");
  dim3 grid(uyd::ceil_div((width + 1) / 2, 256), height);
  uyd::nv12_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(d_y_plane, d_uv_plane, d_output, width, height, y_pitch, uv_pitch, params);
  return (int)cudaGetLastError();
}

// ---- letterboxed frames (UYD_CAM_BGRA_LETTERBOX): geometry and boxes back to frame pixels ----
namespace uyd {
namespace {

// torch's clamp_(lo, hi) on a CUDA float: NaN stays NaN, else min(max(v, lo), hi)
__device__ __forceinline__ float clamp_torch(float v, float hi) { return v != v ? v : fminf(fmaxf(v, 0.f), hi); }

// one thread per (image, row); rows past the image's count are left as they are.  The pad is subtracted and the
// quotient by the gain taken as a product with the fp32 reciprocal, as torch evaluates `boxes[..., :4] /= gain`
// (a CPU scalar divisor becomes a multiply by 1 / (float)gain); the _rn intrinsics keep the two steps unfused.
__global__ void __launch_bounds__(256) letterbox_boxes_kernel(float *__restrict__ det, const int *__restrict__ count, int batch,
                                                              int max_det, float left, float top, float inv_gain, float w0, float h0) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)batch * max_det) return;
  const int b = (int)(i / max_det), r = (int)(i - (long long)b * max_det);
  if (r >= count[b]) return;
  float *d = det + i * 6;
  d[0] = clamp_torch(__fmul_rn(__fsub_rn(d[0], left), inv_gain), w0);
  d[1] = clamp_torch(__fmul_rn(__fsub_rn(d[1], top), inv_gain), h0);
  d[2] = clamp_torch(__fmul_rn(__fsub_rn(d[2], left), inv_gain), w0);
  d[3] = clamp_torch(__fmul_rn(__fsub_rn(d[3], top), inv_gain), h0);
}

}  // namespace
}  // namespace uyd

extern "C" int uyd_letterbox_geometry(int src_w, int src_h, int dst_w, int dst_h, int *new_w, int *new_h, int *left, int *top,
                                      double *gain) {
  UYD_REQUIRE(src_w > 0 && src_h > 0 && dst_w > 0 && dst_h > 0 && new_w && new_h && left && top && gain, UYD_E_ARG,
              "uyd_letterbox_geometry: positive extents and non-NULL outputs required");
  const uyd::LetterboxGeom g = uyd::letterbox_geometry(src_w, src_h, dst_w, dst_h);
  *new_w = g.new_w; *new_h = g.new_h; *left = g.left; *top = g.top; *gain = g.gain;
  return UYD_OK;
}

extern "C" int uyd_letterbox_boxes(uyd_ctx *ctx, float *det, const int *count, int batch, int max_det, int src_w, int src_h, int dst_w,
                                   int dst_h, uyd_stream stream) {
  using namespace uyd;
  UYD_REQUIRE(det && count && (reinterpret_cast<uintptr_t>(det) & (alignof(float) - 1)) == 0, UYD_E_ARG,
              "uyd_letterbox_boxes: non-NULL det (float-aligned) and count required");
  UYD_REQUIRE(batch > 0 && max_det > 0 && src_w > 0 && src_h > 0 && dst_w > 0 && dst_h > 0, UYD_E_ARG,
              "uyd_letterbox_boxes: batch, max_det and extents must be positive");
  const LetterboxGeom g = letterbox_geometry(src_w, src_h, dst_w, dst_h);
  UYD_REQUIRE(g.new_w > 0 && g.new_h > 0, UYD_E_ARG, "uyd_letterbox_boxes: a %d x %d frame letterboxes to nothing in %d x %d", src_w,
              src_h, dst_w, dst_h);
  const long long rows = (long long)batch * max_det;
  UYD_REQUIRE(rows < (1ll << 31), UYD_E_ARG, "uyd_letterbox_boxes: fewer than 2^31 rows required");
  DeviceGuard guard(ctx_device(ctx));
  UYD_CUDA(guard.err);
  const float inv_gain = 1.0f / (float)g.gain;
  letterbox_boxes_kernel<<<ceil_div((int)rows, 256), 256, 0, (cudaStream_t)stream>>>(det, count, batch, max_det, (float)g.left, (float)g.top,
                                                                                     inv_gain, (float)src_w, (float)src_h);
  return (int)cudaGetLastError();
}
