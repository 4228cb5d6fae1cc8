// Box decode kernels.
//  * DFL softmax-integral decode of the Ultralytics Detect head (SURVEY.md a-8:
//    Detect._inference, DFL.forward, make_anchors, dist2bbox) -- warp-shuffle kernel:
//    4 lanes per anchor, one box side (16 bins, 64 contiguous bytes) per lane.
//  * TLBR decode of the custom head (postprocess.hpp:94-145, gpu_postprocess.cu:102-199); the per-cell statement is
//    tlbr_cell (tlbr.cuh), shared with the batched decode + NMS of nms.cu.
#include "common.cuh"
#include "tlbr.cuh"

namespace uyd {
namespace {

constexpr int kThreads = 256;

__device__ __forceinline__ float sigmoidf_(float x) { return __fdividef(1.0f, 1.0f + __expf(-x)); }  // as in conv_chain.cu

// head: [batch, H, W, 4*16 + nc] fp32.  y: [batch, 4+nc, a_total].
template <int REG_MAX>
// q_scale > 0: the DFL projection conv is a QuantConv2d as well (every nn.Conv2d is wrapped, train.py:725):
// probabilities are quantised with scale q_scale = 127 / amax_p, the arange(16) weights with 127 / 15, and the
// expectation is the integer dot product times dq = (amax_p / 127) * (15 / 127).
__global__ void __launch_bounds__(kThreads) decode_dfl_kernel(const float *__restrict__ head, long long n_anchor_total,
                                                              int hw, int w, int nc, float stride,
                                                              float *__restrict__ y, int a_total, int a_off, float q_scale,
                                                              float dq) {
  const int no = 4 * REG_MAX + nc;
  const int lane = threadIdx.x & 31;
  const int side = lane & 3;
  const long long warp = ((long long)blockIdx.x * kThreads + threadIdx.x) >> 5;
  const long long a = warp * 8 + (lane >> 2);  // global anchor id over batch*hw
  const bool live = a < n_anchor_total;
  const long long aa = live ? a : 0;
  const float *p = head + aa * no;
  float v[REG_MAX];
#pragma unroll
  for (int i = 0; i < REG_MAX; i += 4) {
    const float4 q = *reinterpret_cast<const float4 *>(p + side * REG_MAX + i);
    v[i] = q.x; v[i + 1] = q.y; v[i + 2] = q.z; v[i + 3] = q.w;
  }
  float m = v[0];
#pragma unroll
  for (int i = 1; i < REG_MAX; ++i) m = fmaxf(m, v[i]);
  float s = 0.f, ws = 0.f;
#pragma unroll
  for (int i = 0; i < REG_MAX; ++i) {
    const float e = __expf(v[i] - m);  // ex2.approx (identical in conv_chain.cu's fused decode)
    s += e;
    ws = fmaf((float)i, e, ws);
  }
  float d = ws / s;  // expected distance of this side, in cells
  if (q_scale > 0.f) {
    int acc = 0;
#pragma unroll
    for (int i = 0; i < REG_MAX; ++i) {
      const int qp = max(-127, min(127, __float2int_rn(__fmul_rn(__fdiv_rn(__expf(v[i] - m), s), q_scale))));
      const int qw = __float2int_rn(__fmul_rn((float)i, __fdiv_rn(127.f, (float)(REG_MAX - 1))));
      acc += qp * qw;
    }
    d = __fmul_rn((float)acc, dq);
  }
  const unsigned full = 0xffffffffu;
  const int base = lane & ~3;
  const float dl = __shfl_sync(full, d, base + 0);
  const float dt = __shfl_sync(full, d, base + 1);
  const float dr = __shfl_sync(full, d, base + 2);
  const float db = __shfl_sync(full, d, base + 3);
  if (!live) return;
  const int b = (int)(aa / hw);
  const int i = (int)(aa % hw);
  float *yo = y + (long long)b * (4 + nc) * a_total + a_off + i;
  // lane `side` writes output channel `side` of the box (cx, cy, w, h)
  const float ax = (float)(i % w) + 0.5f, ay = (float)(i / w) + 0.5f;
  const float x1 = ax - dl, y1 = ay - dt, x2 = ax + dr, y2 = ay + db;
  float o;
  if (side == 0) o = (x1 + x2) * 0.5f;
  else if (side == 1) o = (y1 + y2) * 0.5f;
  else if (side == 2) o = x2 - x1;
  else o = y2 - y1;
  yo[(long long)side * a_total] = o * stride;
  for (int c = side; c < nc; c += 4) yo[(long long)(4 + c) * a_total] = sigmoidf_(p[4 * REG_MAX + c]);
}

// One thread per cell (tlbr_cell: explicit round-to-nearest box arithmetic, so that no FMA contraction can make it
// differ from the scalar CPU statement).
__global__ void __launch_bounds__(kThreads) decode_tlbr_kernel(const float *__restrict__ cls, const float *__restrict__ reg,
                                                               uyd_detection *dets, int *cell_idx, int *d_count, int cap,
                                                               int gw, int gh, int stride, int nc, float thr, float q,
                                                               int strict, int cell_base) {
  const int g = blockIdx.x * kThreads + threadIdx.x;
  const int hw = gw * gh;
  bool has = false;
  float mc = 0.f;
  int best = -1;
  float4 box = make_float4(0.f, 0.f, 0.f, 0.f);
  if (g < hw) has = tlbr_cell<true>(cls + g, reg + g, hw, nc, g % gw, g / gw, stride, thr, q, strict, mc, best, box);
  const unsigned ballot = __ballot_sync(0xffffffffu, has);
  if (!ballot) return;
  const int lane = threadIdx.x & 31;
  int basei = 0;
  if (lane == (__ffs(ballot) - 1)) basei = atomicAdd(d_count, __popc(ballot));
  basei = __shfl_sync(0xffffffffu, basei, __ffs(ballot) - 1);
  if (!has) return;
  const int slot = basei + __popc(ballot & ((1u << lane) - 1));
  if (slot >= cap) return;
  uyd_detection d;
  d.x1 = box.x; d.y1 = box.y; d.x2 = box.z; d.y2 = box.w; d.confidence = mc; d.class_id = best; d.valid = 1; d._pad = 0;
  dets[slot] = d;
  if (cell_idx) cell_idx[slot] = cell_base + g;
}

}  // namespace

int decode_dfl_launch(const float *head, int batch, int h, int w, int reg_max, int nc, float stride, float *y,
                      int a_total, int a_off, cudaStream_t s, float dfl_amax) {
  UYD_REQUIRE(reg_max == 16, UYD_E_UNSUPPORTED, "DFL decode is built for reg_max == 16 (got %d)", reg_max);
  UYD_REQUIRE(((4 * reg_max + nc) % 4) == 0 && (reinterpret_cast<uintptr_t>(head) & 15) == 0, UYD_E_UNSUPPORTED,
              "head rows must be 16-byte aligned (4*reg_max+nc multiple of 4)");
  const long long n = (long long)batch * h * w;
  const long long warps = (n + 7) / 8;
  const long long blocks = (warps * 32 + kThreads - 1) / kThreads;
  float q_scale = 0.f, dq = 0.f;
  if (dfl_amax > 0.f) {
    q_scale = 127.f / dfl_amax;
    dq = (dfl_amax / 127.f) * (15.f / 127.f);
  }
  decode_dfl_kernel<16><<<(unsigned)blocks, kThreads, 0, s>>>(head, n, h * w, w, nc, stride, y, a_total, a_off, q_scale, dq);
  return (int)cudaGetLastError();
}

}  // namespace uyd

extern "C" int uyd_decode_dfl(uyd_ctx *ctx, const float *head, int batch, int h, int w, int reg_max, int nc,
                              float stride, float *y, int a_total, int a_off, uyd_stream stream) {
  UYD_REQUIRE(head && y && batch > 0 && h > 0 && w > 0, UYD_E_ARG, "uyd_decode_dfl: bad arguments");
  uyd::DeviceGuard guard(uyd::ctx_device(ctx));
  return uyd::decode_dfl_launch(head, batch, h, w, reg_max, nc, stride, y, a_total, a_off, (cudaStream_t)stream, 0.f);
}

extern "C" int uyd_decode_tlbr(uyd_ctx *ctx, const float *d_cls, const float *d_reg, uyd_detection *dets, int *cell_idx,
                               int *d_count, int cap, int grid_w, int grid_h, int stride, int num_classes,
                               float conf_thr, float conformal_q, int strict, int cell_base, uyd_stream stream) {
  UYD_REQUIRE(d_cls && d_reg && dets && d_count && cap > 0 && grid_w > 0 && grid_h > 0, UYD_E_ARG,
              "uyd_decode_tlbr: bad arguments");
  uyd::DeviceGuard guard(uyd::ctx_device(ctx));
  const int hw = grid_w * grid_h;
  uyd::decode_tlbr_kernel<<<uyd::ceil_div(hw, uyd::kThreads), uyd::kThreads, 0, (cudaStream_t)stream>>>(
      d_cls, d_reg, dets, cell_idx, d_count, cap, grid_w, grid_h, stride, num_classes, conf_thr, conformal_q, strict, cell_base);
  return (int)cudaGetLastError();
}
