// Shared host/device helpers for libuyd (sm_100a only).
#pragma once
#include <cuda.h>
#include <cuda_bf16.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/uyd.h"

namespace uyd {

void set_error(const char *fmt, ...);

#define UYD_CUDA(expr)                                                             \
  do {                                                                             \
    cudaError_t _e = (expr);                                                       \
    if (_e != cudaSuccess) {                                                       \
      uyd::set_error("%s:%d %s -> %s", __FILE__, __LINE__, #expr, cudaGetErrorString(_e)); \
      return (int)_e;                                                              \
    }                                                                              \
  } while (0)

#define UYD_REQUIRE(cond, code, ...)   \
  do {                                 \
    if (!(cond)) {                     \
      uyd::set_error(__VA_ARGS__);     \
      return (code);                   \
    }                                  \
  } while (0)

static inline int ceil_div(int a, int b) { return (a + b - 1) / b; }

// Opt-in to > 48 KB of dynamic shared memory, once per (kernel, device): cudaFuncSetAttribute applies to the
// CURRENT device only, so a process that drives several GPUs needs it on each of them (api.cu).
int smem_optin_impl(const void *kernel, int bytes);
template <class K>
inline int smem_optin(K *kernel, size_t bytes) { return smem_optin_impl(reinterpret_cast<const void *>(kernel), (int)bytes); }
int current_sm_count();  // SM count of the current device (cached per device)

// Makes `device` current for the lifetime of the guard and restores the caller's device afterwards: no entry
// point changes the caller's (or torch's) current device.
struct DeviceGuard {
  int prev = -1;
  cudaError_t err = cudaSuccess;
  explicit DeviceGuard(int device) {
    err = cudaGetDevice(&prev);
    if (err == cudaSuccess && prev != device) err = cudaSetDevice(device);
    else if (err == cudaSuccess) prev = -1;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};
int ctx_device(const uyd_ctx *ctx);  // the handle's device (the current device for a NULL handle)

#ifdef __CUDACC__
// Lets a successor launched with programmatic stream serialization (the tcgen05 kernels, tc_ptx.cuh) start its
// prologue while this kernel is still running; the successor still waits for this kernel's completion before
// it reads any activation.
// (lo, hi) -> max(x, 0) rounded to nearest-even bf16, packed: one F2FP.RELU
__device__ __forceinline__ uint32_t relu_pack_bf16x2(float lo, float hi) {
  uint32_t d;
  asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(d) : "f"(hi), "f"(lo));
  return d;
}
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
// Blocks until the predecessor kernel has completed and its writes are visible (no-op for plain launches).
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

// Launch with the programmatic-stream-serialization attribute (UYD_NO_PDL=1 launches plainly).
template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
  static const bool off = [] { const char *v = getenv("UYD_NO_PDL"); return v && *v == '1'; }();
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid;
  cfg.blockDim = block;
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr;
  cfg.numAttrs = off ? 0 : 1;
  return cudaLaunchKernelEx(&cfg, kernel, KArgs(args)...);
}
#endif

// ---------------------------------------------------------------------------------------
// Plan-level data structures shared by the kernel translation units.
// ---------------------------------------------------------------------------------------
struct Buffer {
  int h = 0, w = 0, c = 0, dtype = UYD_BF16;
  void *ptr = nullptr;
  size_t elem_bytes() const { return dtype == UYD_F32 ? 4 : (dtype == UYD_S8 ? 1 : 2); }
  size_t bytes_per_image() const { return (size_t)h * w * c * elem_bytes(); }
};

// Arguments every convolution kernel understands (device pointers already offset to the
// first image; pitches in elements).
struct ConvArgs {
  const void *in;       // NHWC bf16 slice base (or NCHW fp32 network input)
  void *out;            // NHWC slice base (bf16 or fp32)
  const void *res;      // residual slice base or nullptr (bf16)
  const void *w;        // packed weights (layout depends on kernel family)
  const float *bias;    // [cout]
  int n, ih, iw, oh, ow;
  int cin, cout;
  int in_pitch, out_pitch, res_pitch;
  int k, stride, relu, out_f32, in_nchw_f32;
};

struct ctx_impl;  // defined in api.cu

// ---- kernel family entry points (each in its own .cu) ----------------------------------
// conv_direct.cu
size_t direct_weight_bytes(const uyd_conv &d);
void direct_pack_weights(const uyd_conv &d, const float *w, void *dst_host);
int direct_conv_launch(const ConvArgs &a, bool depthwise, cudaStream_t s);
// Camera frames (camera.cuh) straight into model.py's stem: stem_camera_supported says which stems (Conv 3 -> 32, 3x3,
// stride 2, on conv_stem_mma_kernel) stem_camera_launch serves; any other returns UYD_E_UNSUPPORTED without a launch.
struct CamFrames;
bool stem_camera_supported(const ConvArgs &a);
int stem_camera_launch(const ConvArgs &a, const CamFrames &f, cudaStream_t s);

size_t direct_weight_bytes_s8(int cin, int cout, int k);
void direct_pack_weights_s8(int cin, int cout, int k, const int8_t *w, void *dst_host);
int direct_conv_s8_launch(const ConvArgs &a, const float *mult, float out_scale, int out_kind, cudaStream_t s);
void direct_pack_weights_s8_dw(int c, int k, const int8_t *w, void *dst_host);
int direct_conv_s8_dw_launch(const ConvArgs &a, const float *mult, float out_scale, int out_kind, cudaStream_t s);
int quantize_s8_launch(const __nv_bfloat16 *in, int in_pitch, int8_t *out, int out_pitch, long long npix, int c, float scale,
                       cudaStream_t s);
int absmax_launch(const __nv_bfloat16 *in, int in_pitch, long long npix, int c, unsigned int *out_bits, cudaStream_t s);
int abs_histogram_launch(const __nv_bfloat16 *in, int in_pitch, long long npix, int c, float inv_width, int nbins, unsigned int *hist,
                         cudaStream_t s);

// pool_upsample.cu
int sppf_pool_launch(__nv_bfloat16 *base, int n, int h, int w, int pitch, int c, cudaStream_t s);
int upsample2x_launch(const __nv_bfloat16 *in, int in_pitch, __nv_bfloat16 *out, int out_pitch, int n,
                      int ih, int iw, int c, cudaStream_t s);
int nhwc_to_nchw_f32_launch(const float *in, float *out, int n, int h, int w, int c, cudaStream_t s);

// decode.cu
int decode_dfl_launch(const float *head, int batch, int h, int w, int reg_max, int nc, float stride,
                      float *y, int a_total, int a_off, cudaStream_t s, float dfl_amax = 0.f);

}  // namespace uyd
