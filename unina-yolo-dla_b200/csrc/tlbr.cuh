// Per-cell arithmetic of the TLBR head (postprocess.hpp:94-145, gpu_postprocess.cu:102-199), shared by
// decode_tlbr_kernel (decode.cu, CHW planes per image) and the TLBR source of nms_records_kernel (nms.cu, the NHWC
// head buffers of the plan): both paths run this one statement, so their boxes, confidences and classes are
// bit-identical.
#pragma once
#include "common.cuh"

namespace uyd {

// The reference's device sigmoid, statement for statement (gpu_postprocess.cu:62-64): full-accuracy expf and an IEEE
// division, so the TLBR confidences are bit-identical to what decode_yolo_head_kernel produces on the same GPU.
__device__ __forceinline__ float sigmoid_ref(float x) { return __fdiv_rn(1.0f, __fadd_rn(1.0f, expf(-x))); }

// One cell: cls[c * cs] is the logit of class c, reg[k * cs] the k-th distance (left, top, right, bottom) in cells;
// (x, y) is the cell's column and row.  The best class is the first maximum of the SIGMOIDS (not of the logits:
// sigmoid saturates, so two different logits can give the same float).  The running maximum starts at 0, so a cell
// whose sigmoids all underflow keeps class -1 / confidence 0, which a threshold <= 0 (strict = 0) admits.
// Returns whether the cell passes the threshold (conf > thr for strict, conf >= thr otherwise); with BOX the box of
// an admitted cell is formed too, with explicit round-to-nearest intrinsics (no FMA contraction) and the conformal
// dilation by q of its width and height when q > 0.
template <bool BOX>
__device__ __forceinline__ bool tlbr_cell(const float *__restrict__ cls, const float *__restrict__ reg, long long cs, int nc,
                                          int x, int y, int stride, float thr, float q, int strict, float &conf, int &cls_id,
                                          float4 &box) {
  float mc = 0.f;
  int best = -1;
  for (int c = 0; c < nc; ++c) {
    const float pr = sigmoid_ref(cls[c * cs]);
    if (pr > mc) { mc = pr; best = c; }
  }
  conf = mc;
  cls_id = best;
  const bool has = strict ? (mc > thr) : (mc >= thr);
  if (BOX && has) {
    const float fs = (float)stride;
    const float xc = __fmul_rn(__fadd_rn((float)x, 0.5f), fs), yc = __fmul_rn(__fadd_rn((float)y, 0.5f), fs);
    float x1 = __fsub_rn(xc, __fmul_rn(reg[0], fs));
    float y1 = __fsub_rn(yc, __fmul_rn(reg[cs], fs));
    float x2 = __fadd_rn(xc, __fmul_rn(reg[2 * cs], fs));
    float y2 = __fadd_rn(yc, __fmul_rn(reg[3 * cs], fs));
    if (q > 0.f) {
      const float dw = __fmul_rn(__fsub_rn(x2, x1), q), dh = __fmul_rn(__fsub_rn(y2, y1), q);
      x1 = __fsub_rn(x1, dw); y1 = __fsub_rn(y1, dh); x2 = __fadd_rn(x2, dw); y2 = __fadd_rn(y2, dh);
    }
    box = make_float4(x1, y1, x2, y2);
  }
  return has;
}

}  // namespace uyd
