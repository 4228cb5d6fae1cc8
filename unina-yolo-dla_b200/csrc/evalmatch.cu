// Batched evaluation consumer of the [N, 6] detections (SURVEY.md section 8f row 2), the step right after
// the hot path and the reason its NCCL gather exists:
//   * small-object TP / FP / FN  -- UninaValidator.update_metrics, trainer.py:210-265 (pixel xyxy boxes,
//     "small" = width and height below size_thr, match = same class and Ultralytics box_iou > iou_thr;
//     TP = small ground truths hit by ANY prediction, FP = small predictions hitting no small ground truth)
//   * conformal nonconformity scores 1 - IoU of greedily matched pairs -- calibrate_conformal_prediction,
//     train.py:335-470 (predictions in confidence order, best unmatched same-class ground truth with
//     IoU >= match_thr, ties -> first ground truth).
// One CTA per image; detections arrive in confidence order (the NMS emits them that way).
#include "common.cuh"

namespace uyd {
namespace {

// Ultralytics metrics.box_iou: inter / (area1 + area2 - inter + eps), eps = 1e-7, fp32
__device__ __forceinline__ float iou_ultra(const float4 &a, const float4 &b) {
  const float w = fmaxf(__fsub_rn(fminf(a.z, b.z), fmaxf(a.x, b.x)), 0.f);
  const float h = fmaxf(__fsub_rn(fminf(a.w, b.w), fmaxf(a.y, b.y)), 0.f);
  const float inter = __fmul_rn(w, h);
  const float a1 = __fmul_rn(__fsub_rn(a.z, a.x), __fsub_rn(a.w, a.y)), a2 = __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y));
  return __fdiv_rn(inter, __fadd_rn(__fsub_rn(__fadd_rn(a1, a2), inter), 1e-7f));
}

// train.py:335-350: early-out on empty intersection, no epsilon
__device__ __forceinline__ float iou_plain(const float4 &a, const float4 &b) {
  const float x1 = fmaxf(a.x, b.x), y1 = fmaxf(a.y, b.y), x2 = fminf(a.z, b.z), y2 = fminf(a.w, b.w);
  if (x2 <= x1 || y2 <= y1) return 0.f;
  const float inter = __fmul_rn(__fsub_rn(x2, x1), __fsub_rn(y2, y1));
  const float uni = __fsub_rn(__fadd_rn(__fmul_rn(__fsub_rn(a.z, a.x), __fsub_rn(a.w, a.y)), __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y))), inter);
  return uni > 0.f ? __fdiv_rn(inter, uni) : 0.f;
}

constexpr int kThreads = 128, kMaxGt = 1024, kMaxDet = 1024;

__global__ void __launch_bounds__(kThreads) eval_update_kernel(const float *__restrict__ det, const int *__restrict__ cnt, int max_det,
                                                               const float *__restrict__ gt, const int *__restrict__ gt_cnt, int gmax,
                                                               float size_thr, float small_iou_thr, float match_iou_thr,
                                                               unsigned long long *__restrict__ counters, float *__restrict__ scores) {
  __shared__ float4 gbox[kMaxGt];
  __shared__ int gcls[kMaxGt];
  __shared__ unsigned char gsmall[kMaxGt], gused[kMaxGt];
  __shared__ int s_small_gt, s_tp, s_fp;
  __shared__ float w_iou[kThreads / 32];
  __shared__ int w_idx[kThreads / 32];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int n = min(cnt[b], max_det), g = min(gt_cnt[b], min(gmax, kMaxGt));
  const float *dimg = det + (long long)b * max_det * 6;
  if (tid == 0) s_small_gt = s_tp = s_fp = 0;
  __syncthreads();
  int local_small = 0;
  for (int j = tid; j < g; j += kThreads) {
    const float *q = gt + ((long long)b * gmax + j) * 5;
    gbox[j] = make_float4(q[1], q[2], q[3], q[4]);
    gcls[j] = (int)q[0];
    const bool sm = __fsub_rn(q[3], q[1]) < size_thr && __fsub_rn(q[4], q[2]) < size_thr;
    gsmall[j] = sm;
    gused[j] = 0;
    local_small += sm;
  }
  if (local_small) atomicAdd(&s_small_gt, local_small);
  __syncthreads();
  // ---- small-object counters (skipped entirely when the image has no small ground truth, trainer.py:231) ----
  if (s_small_gt > 0) {
    int tp = 0, fp = 0;
    for (int j = tid; j < g; j += kThreads) {
      if (!gsmall[j]) continue;
      bool hit = false;
      for (int i = 0; i < n && !hit; ++i) {
        const float *d = dimg + i * 6;
        hit = (int)d[5] == gcls[j] && iou_ultra(make_float4(d[0], d[1], d[2], d[3]), gbox[j]) > small_iou_thr;
      }
      tp += hit;
    }
    for (int i = tid; i < n; i += kThreads) {
      const float *d = dimg + i * 6;
      const float4 pb = make_float4(d[0], d[1], d[2], d[3]);
      if (!(__fsub_rn(pb.z, pb.x) < size_thr && __fsub_rn(pb.w, pb.y) < size_thr)) continue;
      bool hit = false;
      for (int j = 0; j < g && !hit; ++j) hit = gsmall[j] && (int)d[5] == gcls[j] && iou_ultra(pb, gbox[j]) > small_iou_thr;
      fp += !hit;
    }
    if (tp) atomicAdd(&s_tp, tp);
    if (fp) atomicAdd(&s_fp, fp);
  }
  __syncthreads();
  if (tid == 0 && s_small_gt > 0) {
    atomicAdd(&counters[0], (unsigned long long)s_tp);
    atomicAdd(&counters[1], (unsigned long long)s_fp);
    atomicAdd(&counters[2], (unsigned long long)(s_small_gt - s_tp));
  }
  // ---- conformal scores: greedy matching in confidence order ----
  if (!scores) return;
  for (int i = 0; i < max_det; ++i) {
    float best = 0.f;
    int best_j = 0x7fffffff;
    if (i < n) {
      const float *d = dimg + i * 6;
      const float4 pb = make_float4(d[0], d[1], d[2], d[3]);
      const int pc = (int)d[5];
      for (int j = tid; j < g; j += kThreads) {
        if (gused[j] || gcls[j] != pc) continue;
        const float v = iou_plain(pb, gbox[j]);
        if (v > best && v >= match_iou_thr) { best = v; best_j = j; }  // strict >: the first index wins a tie inside a thread
      }
    }
    // block argmax, ties -> lowest ground-truth index
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, best, o);
      const int oj = __shfl_xor_sync(0xffffffffu, best_j, o);
      if (ov > best || (ov == best && oj < best_j)) { best = ov; best_j = oj; }
    }
    if ((tid & 31) == 0) { w_iou[tid >> 5] = best; w_idx[tid >> 5] = best_j; }
    __syncthreads();
    if (tid == 0) {
      for (int w = 1; w < kThreads / 32; ++w)
        if (w_iou[w] > best || (w_iou[w] == best && w_idx[w] < best_j)) { best = w_iou[w]; best_j = w_idx[w]; }
      const bool ok = i < n && best_j != 0x7fffffff && best > 0.f;
      if (ok) gused[best_j] = 1;
      scores[(long long)b * max_det + i] = ok ? __fsub_rn(1.0f, best) : -1.0f;
    }
    __syncthreads();
  }
}


// ---- data_loader.SmallObjectMetric.update (data_loader.py:322-389), one CTA per image ------------------------
// Rows in the reference's own format: pred (x_c, y_c, w, h, conf, cls) and gt (cls, x_c, y_c, w, h), normalised to the
// image; predictions arrive in confidence order.  A "small" box has w * image_size and h * image_size below size_thr
// (double arithmetic, like the Python floats of _is_small).  Per prediction: the best IoU (> 0, strict: the first
// ground truth wins a tie) over the unmatched small ground truths of its class; IoU >= iou_thr -> TP and the ground
// truth is matched, else FP iff the prediction itself is small.  FN = small ground truths left unmatched.
__device__ __forceinline__ float iou_cxcywh(const float4 &a, const float4 &b) {  // data_loader.py:288-320, fp32 like the tensors
  const float ax1 = __fsub_rn(a.x, __fmul_rn(a.z, 0.5f)), ay1 = __fsub_rn(a.y, __fmul_rn(a.w, 0.5f));
  const float ax2 = __fadd_rn(a.x, __fmul_rn(a.z, 0.5f)), ay2 = __fadd_rn(a.y, __fmul_rn(a.w, 0.5f));
  const float bx1 = __fsub_rn(b.x, __fmul_rn(b.z, 0.5f)), by1 = __fsub_rn(b.y, __fmul_rn(b.w, 0.5f));
  const float bx2 = __fadd_rn(b.x, __fmul_rn(b.z, 0.5f)), by2 = __fadd_rn(b.y, __fmul_rn(b.w, 0.5f));
  const float iw = fmaxf(0.f, __fsub_rn(fminf(ax2, bx2), fmaxf(ax1, bx1))), ih = fmaxf(0.f, __fsub_rn(fminf(ay2, by2), fmaxf(ay1, by1)));
  const float inter = __fmul_rn(iw, ih);
  const float uni = __fsub_rn(__fadd_rn(__fmul_rn(__fsub_rn(ax2, ax1), __fsub_rn(ay2, ay1)), __fmul_rn(__fsub_rn(bx2, bx1), __fsub_rn(by2, by1))), inter);
  return uni <= 0.f ? 0.f : __fdiv_rn(inter, uni);
}

__global__ void __launch_bounds__(kThreads) small_object_metric_kernel(const float *__restrict__ pred, const int *__restrict__ cnt,
                                                                       int max_det, const float *__restrict__ gt,
                                                                       const int *__restrict__ gt_cnt, int gmax, double size_thr,
                                                                       double iou_thr, double image_size,
                                                                       unsigned long long *__restrict__ counters) {
  __shared__ float4 gbox[kMaxGt];
  __shared__ int gcls[kMaxGt];
  __shared__ unsigned char gused[kMaxGt];
  __shared__ int s_n;
  __shared__ float w_iou[kThreads / 32];
  __shared__ int w_idx[kThreads / 32];
  const int b = blockIdx.x, tid = threadIdx.x;
  const int n = min(cnt[b], max_det), g = min(gt_cnt[b], min(gmax, kMaxGt));
  if (tid == 0) {  // ordered compaction of the small ground truths (the order decides IoU ties)
    int k = 0;
    for (int j = 0; j < g; ++j) {
      const float *q = gt + ((long long)b * gmax + j) * 5;
      if ((double)q[3] * image_size < size_thr && (double)q[4] * image_size < size_thr) {
        gbox[k] = make_float4(q[1], q[2], q[3], q[4]);
        gcls[k] = (int)q[0];
        gused[k] = 0;
        ++k;
      }
    }
    s_n = k;
  }
  __syncthreads();
  const int ns = s_n;
  if (ns == 0) return;  // no small objects in this image (data_loader.py:337-338)
  int tp = 0, fp = 0;
  for (int i = 0; i < n; ++i) {
    const float *d = pred + ((long long)b * max_det + i) * 6;
    const float4 pb = make_float4(d[0], d[1], d[2], d[3]);
    const int pc = (int)d[5];
    float best = 0.f;
    int best_j = 0x7fffffff;
    for (int j = tid; j < ns; j += kThreads) {
      if (gused[j] || gcls[j] != pc) continue;
      const float v = iou_cxcywh(pb, gbox[j]);
      if (v > best) { best = v; best_j = j; }
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      const float ov = __shfl_xor_sync(0xffffffffu, best, o);
      const int oj = __shfl_xor_sync(0xffffffffu, best_j, o);
      if (ov > best || (ov == best && oj < best_j)) { best = ov; best_j = oj; }
    }
    if ((tid & 31) == 0) { w_iou[tid >> 5] = best; w_idx[tid >> 5] = best_j; }
    __syncthreads();
    if (tid == 0) {
      for (int w = 1; w < kThreads / 32; ++w)
        if (w_iou[w] > best || (w_iou[w] == best && w_idx[w] < best_j)) { best = w_iou[w]; best_j = w_idx[w]; }
      if ((double)best >= iou_thr) {
        ++tp;
        if (best_j != 0x7fffffff) gused[best_j] = 1;   // (iou_thr <= 0 with no candidate: the reference adds index -1)
      } else if ((double)pb.z * image_size < size_thr && (double)pb.w * image_size < size_thr) {
        ++fp;
      }
    }
    __syncthreads();
  }
  if (tid == 0) {
    int matched = 0;
    for (int j = 0; j < ns; ++j) matched += gused[j];
    atomicAdd(&counters[0], (unsigned long long)tp);
    atomicAdd(&counters[1], (unsigned long long)fp);
    atomicAdd(&counters[2], (unsigned long long)(ns - matched));
  }
}

// ---- mAP50 / mAP50-95: Ultralytics DetectionValidator.match_predictions + metrics.ap_per_class (oracle/evalref.py) --
// map_match_kernel, one CTA per image.  match_predictions keeps, per detection, its best ground truth among the pairs
// with IoU >= t, then, per ground truth, the lowest detection index.  The best pair over IoU >= t is the detection's
// best same-class ground truth j*(p) (the highest index among equal IoUs) whenever its IoU v*(p) >= t, so one pass
// serves every threshold: first[j][t] = the lowest p with j*(p) = j and v*(p) >= t is the TP of (j, t).  Per row the
// kernel writes the TP mask (bit t) and the sort key class << 32 | descending confidence; rows past the count and
// rows whose class is not an integer in [0, nc) or whose confidence is NaN get kMapPadKey, which sorts behind every
// class.  Ground truths and detections that cannot be indexed are counted in *dropped instead.
constexpr int kMapMaxT = 16, kMapThreads = 256, kMapMaxGt = 1024, kMapMaxDet = 1024, kMapMaxClasses = 1 << 20;
constexpr long long kMapPadKey = 0x7fffffffffffffffLL;

struct MapThresholds {
  float t[kMapMaxT];
};

__device__ __forceinline__ bool class_index(float c, int nc, int &out) {
  if (!(c >= 0.f && c < (float)nc && c == truncf(c))) return false;   // NaN fails every comparison
  out = (int)c;
  return true;
}

// ascending key for descending confidence; -0 ranks as +0 (numpy compares them equal, the stable sort keeps order)
__device__ __forceinline__ unsigned int conf_desc_bits(float c) {
  unsigned int u = __float_as_uint(c == 0.f ? 0.f : c);
  u = (u & 0x80000000u) ? ~u : (u | 0x80000000u);
  return ~u;
}

__device__ __forceinline__ float conf_from_key(long long k) {
  unsigned int u = ~(unsigned int)k;
  u = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
  return __uint_as_float(u);
}

__global__ void __launch_bounds__(kMapThreads) map_match_kernel(const float *__restrict__ det, const int *__restrict__ cnt, int max_det,
                                                                 const float *__restrict__ gt, const int *__restrict__ gt_cnt, int gmax,
                                                                 int nc, MapThresholds thr, int nthr, unsigned short *__restrict__ tp_mask,
                                                                 long long *__restrict__ key, unsigned long long *__restrict__ n_labels,
                                                                 unsigned long long *__restrict__ dropped) {
  extern __shared__ __align__(16) unsigned char map_smem[];
  float4 *gbox = reinterpret_cast<float4 *>(map_smem);                    // [gmax]
  unsigned int *first = reinterpret_cast<unsigned int *>(gbox + gmax);    // [gmax][nthr]
  int *gcls = reinterpret_cast<int *>(first + gmax * nthr);               // [gmax], -1: not indexable
  int *dj = gcls + gmax;                                                  // [max_det] j*(p); -1 none, -2 dropped
  __shared__ int s_drop;
  const int b = blockIdx.x, tid = threadIdx.x;
  const int n = max(0, min(cnt[b], max_det)), g = max(0, min(gt_cnt[b], gmax));
  const float *dimg = det + (long long)b * max_det * 6;
  if (tid == 0) s_drop = 0;
  int drop = 0;
  for (int j = tid; j < g; j += kMapThreads) {
    const float *q = gt + ((long long)b * gmax + j) * 5;
    gbox[j] = make_float4(q[1], q[2], q[3], q[4]);
    int c;
    if (class_index(q[0], nc, c)) {
      atomicAdd(&n_labels[c], 1ull);
    } else {
      c = -1;
      ++drop;
    }
    gcls[j] = c;
  }
  for (int k = tid; k < g * nthr; k += kMapThreads) first[k] = 0xffffffffu;
  __syncthreads();
  for (int i = tid; i < n; i += kMapThreads) {
    const float *d = dimg + i * 6;
    int pc, bj = -1;
    if (class_index(d[5], nc, pc) && !isnan(d[4])) {
      const float4 pb = make_float4(d[0], d[1], d[2], d[3]);
      float best = 0.f;
      for (int j = 0; j < g; ++j) {
        if (gcls[j] != pc) continue;
        const float v = iou_ultra(pb, gbox[j]);
        if (v >= best) { best = v; bj = j; }   // >=: the higher index wins a tie; NaN never enters
      }
      if (bj >= 0)
        for (int t = 0; t < nthr; ++t)
          if (best >= thr.t[t]) atomicMin(&first[bj * nthr + t], (unsigned int)i);
    } else {
      bj = -2;
      ++drop;
    }
    dj[i] = bj;
  }
  if (drop) atomicAdd(&s_drop, drop);
  __syncthreads();
  unsigned short *mrow = tp_mask + (long long)b * max_det;
  long long *krow = key + (long long)b * max_det;
  for (int i = tid; i < max_det; i += kMapThreads) {
    unsigned int m = 0;
    long long k = kMapPadKey;
    if (i < n && dj[i] != -2) {
      const int j = dj[i];
      if (j >= 0)
        for (int t = 0; t < nthr; ++t) m |= (unsigned int)(first[j * nthr + t] == (unsigned int)i) << t;
      k = ((long long)(int)dimg[i * 6 + 5] << 32) | conf_desc_bits(dimg[i * 6 + 4]);
    }
    mrow[i] = (unsigned short)m;
    krow[i] = k;
  }
  if (tid == 0 && s_drop) atomicAdd(dropped, (unsigned long long)s_drop);
}

// ap_per_class_kernel, one CTA per class c over that class's records [s, e) of the key-sorted order (confidence
// descending, ties in record order).  Everything is fp64 with explicit round-to-nearest operations, so the result is
// numpy's: tpc / fpc are int64 prefix counts, recall = tpc / (n_l + 1e-16), precision = tpc / (tpc + fpc).
// compute_ap works on the positions j = 0 .. n + 1 of mrec = [0, recall, 1] / mpre = [1, precision, 0]; mpre becomes
// its suffix maximum (the envelope).  np.interp(x, mrec, mpre) at x_i = i * 0.01 (x_100 = 1) takes the last j with
// mrec[j] <= x_i: mpre[j] when j = n + 1 or mrec[j] == x_i, else slope * (x_i - mrec[j]) + mpre[j] with
// slope = (mpre[j+1] - mpre[j]) / (mrec[j+1] - mrec[j]).  So each j owns the grid points in [mrec[j], mrec[j+1]).
// The positions are walked backwards in chunks of kApChunk: a block suffix sum of the TP counts gives each thread
// its tpc, a block suffix max of the precisions its envelope, then each thread walks its kApPer positions down.
// The 1000-point p / r curves at threshold 0 are np.interp(-x, -conf, ., left) the same way, owned by records.
constexpr int kApThreads = 256, kApPer = 16, kApChunk = kApThreads * kApPer, kApWarps = kApThreads / 32;

__device__ __forceinline__ double grid101(int i) { return i >= 100 ? 1.0 : __dmul_rn((double)i, 0.01); }      // np.linspace(0, 1, 101)
__device__ __forceinline__ double grid1000(int q) { return q >= 999 ? 1.0 : __dmul_rn((double)q, 1.0 / 999.0); }  // np.linspace(0, 1, 1000)

__device__ __forceinline__ int first_ge101(double r) {   // lowest i in [0, 101] with grid101(i) >= r
  int i = (int)fmin(fmax(ceil(r * 100.0) - 1.0, 0.0), 101.0);
  while (i < 101 && grid101(i) < r) ++i;
  while (i > 0 && grid101(i - 1) >= r) --i;
  return i;
}

__device__ __forceinline__ int first_gt1000(double c) {  // lowest q in [0, 1000] with grid1000(q) > c
  int q = (int)fmin(fmax(floor(c * 999.0) - 1.0, 0.0), 1000.0);
  while (q < 1000 && grid1000(q) <= c) ++q;
  while (q > 0 && grid1000(q - 1) > c) --q;
  return q;
}

// np.interp between (xa, ya) and (xb, yb), xa < x < xb: slope * (x - xa) + ya, unfused
__device__ __forceinline__ double interp_np(double x, double xa, double xb, double ya, double yb) {
  const double slope = __ddiv_rn(__dsub_rn(yb, ya), __dsub_rn(xb, xa));
  return __dadd_rn(__dmul_rn(slope, __dsub_rn(x, xa)), ya);
}

__global__ void __launch_bounds__(kApThreads) ap_per_class_kernel(const long long *__restrict__ skey, const long long *__restrict__ order,
                                                                  const unsigned short *__restrict__ tp_mask, long long nrec,
                                                                  const long long *__restrict__ n_labels, int nthr,
                                                                  double *__restrict__ ap, double *__restrict__ p_curve,
                                                                  double *__restrict__ r_curve) {
  __shared__ double s_y[kMapMaxT][101];                     // np.interp(x, mrec, mpre) at the 101 grid points
  __shared__ unsigned short s_mask[kApPer][kApThreads];     // the chunk's TP masks, [r][thread]
  __shared__ float s_conf[kApPer][kApThreads];
  __shared__ long long s_wsum[kApWarps][kMapMaxT], s_tpc_after[kMapMaxT], s_tot[kMapMaxT];
  __shared__ double s_wmax[kApWarps][kMapMaxT], s_env_after[kMapMaxT];
  __shared__ long long s_seg[2];
  const int c = blockIdx.x, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  if (tid < 2) {   // [s, e): lower bounds of c << 32 and (c + 1) << 32
    const long long want = (long long)(c + tid) << 32;
    long long lo = 0, hi = nrec;
    while (lo < hi) {
      const long long mid = (lo + hi) >> 1;
      if (skey[mid] < want) lo = mid + 1; else hi = mid;
    }
    s_seg[tid] = lo;
  }
  if (tid < kMapMaxT) { s_tpc_after[tid] = 0; s_env_after[tid] = 0.0; }
  __syncthreads();
  const long long s = s_seg[0], n = s_seg[1] - s, nl = n_labels[c];
  double *pc = p_curve + (long long)c * 1000, *rc = r_curve + (long long)c * 1000;
  if (n == 0 || nl == 0) {   // no prediction (or no label: the host does not report the class): zeros
    for (int q = tid; q < 1000; q += kApThreads) pc[q] = rc[q] = 0.0;
    if (tid < nthr) ap[(long long)c * nthr + tid] = 0.0;
    return;
  }
  const double nld = __dadd_rn((double)nl, 1e-16);
  const long long M = n + 2;   // positions of mrec / mpre

  {  // the TP totals per threshold
    long long tot[kMapMaxT];
#pragma unroll
    for (int t = 0; t < kMapMaxT; ++t) tot[t] = 0;
    for (long long k = tid; k < n; k += kApThreads) {
      const unsigned int m = tp_mask[order[s + k]];
#pragma unroll
      for (int t = 0; t < kMapMaxT; ++t) tot[t] += (m >> t) & 1u;
    }
#pragma unroll
    for (int t = 0; t < kMapMaxT; ++t) {
      if (t >= nthr) break;
      long long x = tot[t];
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
      if (lane == 0) s_wsum[warp][t] = x;
    }
    __syncthreads();
    if (tid < nthr) {
      long long x = 0;
      for (int w = 0; w < kApWarps; ++w) x += s_wsum[w][tid];
      s_tot[tid] = x;
    }
    __syncthreads();
  }

  for (long long base = ((M - 1) / kApChunk) * kApChunk; base >= 0; base -= kApChunk) {
    const long long p0 = base + (long long)tid * kApPer, phi = p0 + kApPer - 1;
    // stage the chunk's masks and confidences (position j >= 1 is record j - 1)
    long long cnt[kMapMaxT];
#pragma unroll
    for (int t = 0; t < kMapMaxT; ++t) cnt[t] = 0;
    for (int r = 0; r < kApPer; ++r) {
      const long long j = p0 + r;
      unsigned int m = 0;
      float cf = 0.f;
      if (j >= 1 && j <= n) {
        m = tp_mask[order[s + j - 1]];
        cf = conf_from_key(skey[s + j - 1]);
      }
      s_mask[r][tid] = (unsigned short)m;
      s_conf[r][tid] = cf;
#pragma unroll
      for (int t = 0; t < kMapMaxT; ++t) cnt[t] += (m >> t) & 1u;
    }
    // block suffix sum: TPs at positions above this thread's run
    long long after[kMapMaxT];
#pragma unroll
    for (int t = 0; t < kMapMaxT; ++t) {
      if (t >= nthr) break;
      long long x = cnt[t];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const long long y = __shfl_down_sync(0xffffffffu, x, o);
        if (lane + o < 32) x += y;
      }
      if (lane == 0) s_wsum[warp][t] = x;
      after[t] = x - cnt[t];
    }
    __syncthreads();
    long long tpc[kMapMaxT];
#pragma unroll
    for (int t = 0; t < kMapMaxT; ++t) tpc[t] = 0;
#pragma unroll
    for (int t = 0; t < kMapMaxT; ++t) {
      if (t >= nthr) break;
      long long a = after[t] + s_tpc_after[t];
      for (int w = warp + 1; w < kApWarps; ++w) a += s_wsum[w][t];
      tpc[t] = s_tot[t] - a;   // tpc at position phi
    }
    // run maximum of the precision, then the block suffix max: the envelope above this thread's run
    double emax[kMapMaxT];
#pragma unroll
    for (int t = 0; t < kMapMaxT; ++t) {
      if (t >= nthr) break;
      long long k = tpc[t];
      double mx = 0.0;
      for (int r = kApPer - 1; r >= 0; --r) {
        const long long j = p0 + r;
        if (j < M) mx = fmax(mx, j == 0 ? 1.0 : j == M - 1 ? 0.0 : __ddiv_rn((double)k, (double)j));
        k -= (s_mask[r][tid] >> t) & 1u;
      }
      double x = mx;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const double y = __shfl_down_sync(0xffffffffu, x, o);
        if (lane + o < 32) x = fmax(x, y);
      }
      if (lane == 0) s_wmax[warp][t] = x;
      const double y = __shfl_down_sync(0xffffffffu, x, 1);
      emax[t] = lane < 31 ? y : 0.0;   // max over the later lanes of this warp
    }
    __syncthreads();
    // the record right above the run (the next thread's first, or the next chunk's)
    unsigned int nmask = 0;
    double nconf = 0.0;
    if (phi + 1 <= n) {
      nmask = tp_mask[order[s + phi]];
      nconf = (double)conf_from_key(skey[s + phi]);
    }
    double next_rec[kMapMaxT], next_env[kMapMaxT], next_p0 = 0.0;
#pragma unroll
    for (int t = 0; t < kMapMaxT; ++t) {
      if (t >= nthr) break;
      double e = fmax(emax[t], s_env_after[t]);
      for (int w = warp + 1; w < kApWarps; ++w) e = fmax(e, s_wmax[w][t]);
      next_env[t] = e;
      const long long jn = phi + 1, kn = tpc[t] + ((nmask >> t) & 1u);
      next_rec[t] = jn >= M - 1 ? 1.0 : __ddiv_rn((double)kn, nld);
      if (t == 0 && jn <= n) next_p0 = __ddiv_rn((double)kn, (double)jn);
    }
    int next_q = first_gt1000(nconf);
    // the walk down the run
    for (int r = kApPer - 1; r >= 0; --r) {
      const long long j = p0 + r;
      const unsigned int m = s_mask[r][tid];
      if (j < M) {
        const bool last = j == M - 1;
#pragma unroll
        for (int t = 0; t < kMapMaxT; ++t) {
          if (t >= nthr) break;
          const double rec = j == 0 ? 0.0 : last ? 1.0 : __ddiv_rn((double)tpc[t], nld);
          const double pre = j == 0 ? 1.0 : last ? 0.0 : __ddiv_rn((double)tpc[t], (double)j);
          const double env = fmax(pre, next_env[t]);
          if (last || rec < next_rec[t]) {   // equal recalls own no grid point
            const int i1 = last ? 101 : first_ge101(next_rec[t]);
            for (int i = first_ge101(rec); i < i1; ++i) {
              const double x = grid101(i);
              s_y[t][i] = (last || x == rec) ? env : interp_np(x, rec, next_rec[t], env, next_env[t]);
            }
          }
          if (t == 0 && j >= 1 && j <= n) {   // the curves: xp = -conf, this record owns -conf[j] <= -x < -conf[j + 1]
            const double cf = (double)s_conf[r][tid];
            const int q0 = j == n ? 0 : next_q, q1 = first_gt1000(cf);
            for (int q = q0; q < q1; ++q) {
              const double x = grid1000(q);
              if (j == n || x == cf) {
                rc[q] = rec;
                pc[q] = pre;
              } else {
                rc[q] = interp_np(-x, -cf, -nconf, rec, next_rec[0]);
                pc[q] = interp_np(-x, -cf, -nconf, pre, next_p0);
              }
            }
            if (j == 1)
              for (int q = q1; q < 1000; ++q) { rc[q] = 0.0; pc[q] = 1.0; }   // left of the first sample
            next_q = q1;
            nconf = cf;
            next_p0 = pre;
          }
          next_rec[t] = rec;
          next_env[t] = env;
        }
      }
#pragma unroll
      for (int t = 0; t < kMapMaxT; ++t)
        if (t < nthr) tpc[t] -= (m >> t) & 1u;
    }
    __syncthreads();
    if (tid == 0) {   // carry into the chunk below
#pragma unroll
      for (int t = 0; t < kMapMaxT; ++t) {
        if (t >= nthr) break;
        long long a = 0;
        double e = 0.0;
        for (int w = 0; w < kApWarps; ++w) { a += s_wsum[w][t]; e = fmax(e, s_wmax[w][t]); }
        s_tpc_after[t] += a;
        s_env_after[t] = fmax(s_env_after[t], e);
      }
    }
    __syncthreads();
  }
  // np.trapezoid over the 100 intervals: numpy's pairwise sum of fewer than 128 terms is eight strided
  // accumulators over terms 0..95, combined pairwise, then terms 96..99 in order
  if (tid < nthr) {
    const double *y = s_y[tid];
    auto term = [y](int i) {
      return __ddiv_rn(__dmul_rn(__dsub_rn(grid101(i + 1), grid101(i)), __dadd_rn(y[i + 1], y[i])), 2.0);
    };
    double acc[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) acc[k] = term(k);
    for (int i = 8; i < 96; i += 8)
#pragma unroll
      for (int k = 0; k < 8; ++k) acc[k] = __dadd_rn(acc[k], term(i + k));
    double res = __dadd_rn(__dadd_rn(__dadd_rn(acc[0], acc[1]), __dadd_rn(acc[2], acc[3])),
                           __dadd_rn(__dadd_rn(acc[4], acc[5]), __dadd_rn(acc[6], acc[7])));
    for (int i = 96; i < 100; ++i) res = __dadd_rn(res, term(i));
    ap[(long long)c * nthr + tid] = res;
  }
}

}  // namespace
}  // namespace uyd

extern "C" int uyd_small_object_metric_update(uyd_ctx *ctx, const float *pred, const int *count, int batch, int max_det, const float *gt,
                                              const int *gt_count, int gt_max, double size_thr, double iou_thr, double image_size,
                                              unsigned long long *counters, uyd_stream stream) {
  UYD_REQUIRE(pred && count && gt && gt_count && counters && batch > 0 && max_det > 0 && gt_max > 0, UYD_E_ARG,
              "uyd_small_object_metric_update: bad arguments");
  uyd::DeviceGuard guard(uyd::ctx_device(ctx));
  UYD_REQUIRE(gt_max <= uyd::kMaxGt, UYD_E_UNSUPPORTED, "uyd_small_object_metric_update: at most %d ground truths per image", uyd::kMaxGt);
  uyd::small_object_metric_kernel<<<batch, uyd::kThreads, 0, (cudaStream_t)stream>>>(pred, count, max_det, gt, gt_count, gt_max, size_thr,
                                                                                      iou_thr, image_size, counters);
  return (int)cudaGetLastError();
}

extern "C" int uyd_eval_update(uyd_ctx *ctx, const float *det, const int *count, int batch, int max_det, const float *gt,
                               const int *gt_count, int gt_max, float size_thr, float small_iou_thr, float match_iou_thr,
                               unsigned long long *counters, float *scores, uyd_stream stream) {
  UYD_REQUIRE(det && count && gt && gt_count && counters && batch > 0 && max_det > 0 && gt_max > 0, UYD_E_ARG,
              "uyd_eval_update: bad arguments");
  uyd::DeviceGuard guard(uyd::ctx_device(ctx));
  UYD_REQUIRE(gt_max <= uyd::kMaxGt && max_det <= uyd::kMaxDet, UYD_E_UNSUPPORTED, "uyd_eval_update: at most %d ground truths / %d detections per image",
              uyd::kMaxGt, uyd::kMaxDet);
  uyd::eval_update_kernel<<<batch, uyd::kThreads, 0, (cudaStream_t)stream>>>(det, count, max_det, gt, gt_count, gt_max, size_thr,
                                                                              small_iou_thr, match_iou_thr, counters, scores);
  return (int)cudaGetLastError();
}

extern "C" int uyd_eval_match(uyd_ctx *ctx, const float *det, const int *count, int batch, int max_det, const float *gt,
                              const int *gt_count, int gt_max, int nc, const float *iou_thresholds, int n_thresholds,
                              unsigned short *tp_mask, long long *sort_key, long long *n_labels, long long *dropped,
                              uyd_stream stream) {
  UYD_REQUIRE(det && count && gt && gt_count && iou_thresholds && tp_mask && sort_key && n_labels && dropped && batch > 0 &&
                  max_det > 0 && gt_max > 0 && nc > 0 && n_thresholds >= 1 && n_thresholds <= uyd::kMapMaxT,
              UYD_E_ARG, "uyd_eval_match: bad arguments");
  uyd::MapThresholds thr{};
  for (int t = 0; t < n_thresholds; ++t) {
    UYD_REQUIRE(iou_thresholds[t] > 0.f, UYD_E_ARG, "uyd_eval_match: IoU threshold %d is not positive", t);
    thr.t[t] = iou_thresholds[t];
  }
  UYD_REQUIRE(nc <= uyd::kMapMaxClasses && gt_max <= uyd::kMapMaxGt && max_det <= uyd::kMapMaxDet, UYD_E_UNSUPPORTED,
              "uyd_eval_match: at most %d classes, %d ground truths and %d detections per image", uyd::kMapMaxClasses,
              uyd::kMapMaxGt, uyd::kMapMaxDet);
  uyd::DeviceGuard guard(uyd::ctx_device(ctx));
  const size_t smem = (size_t)gt_max * (sizeof(float4) + sizeof(int) * (n_thresholds + 1)) + (size_t)max_det * sizeof(int);
  if (smem > 48 * 1024) {
    const cudaError_t e = cudaFuncSetAttribute(uyd::map_match_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return (int)e;
  }
  uyd::map_match_kernel<<<batch, uyd::kMapThreads, smem, (cudaStream_t)stream>>>(
      det, count, max_det, gt, gt_count, gt_max, nc, thr, n_thresholds, tp_mask, sort_key, (unsigned long long *)n_labels,
      (unsigned long long *)dropped);
  return (int)cudaGetLastError();
}

extern "C" int uyd_eval_ap(uyd_ctx *ctx, const long long *sorted_key, const long long *order, const unsigned short *tp_mask,
                           long long n_records, const long long *n_labels, int nc, int n_thresholds, double *ap, double *p_curve,
                           double *r_curve, uyd_stream stream) {
  UYD_REQUIRE(sorted_key && order && tp_mask && n_labels && ap && p_curve && r_curve && n_records > 0 && nc > 0 &&
                  n_thresholds >= 1 && n_thresholds <= uyd::kMapMaxT,
              UYD_E_ARG, "uyd_eval_ap: bad arguments");
  UYD_REQUIRE(nc <= uyd::kMapMaxClasses, UYD_E_UNSUPPORTED, "uyd_eval_ap: at most %d classes", uyd::kMapMaxClasses);
  uyd::DeviceGuard guard(uyd::ctx_device(ctx));
  uyd::ap_per_class_kernel<<<nc, uyd::kApThreads, 0, (cudaStream_t)stream>>>(sorted_key, order, tp_mask, n_records, n_labels,
                                                                             n_thresholds, ap, p_curve, r_curve);
  return (int)cudaGetLastError();
}
