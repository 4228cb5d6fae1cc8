// Class-aware NMS, bit-exact with the CPU statement.
//
// uyd_nms (Ultralytics non_max_suppression + torchvision.ops.nms, SURVEY.md A.3/A.4; reference call sites
// train.py:396-405, eval.py:32) runs as ONE launch, nms_image_kernel below; uyd_nms_detections (the custom head's
// postprocess.hpp:44-67 NMS over detection records) as ONE launch, nms_records_kernel; uyd_nms_tlbr (TLBR decode of
// the custom head + the same NMS, a whole batch) as ONE launch of nms_records_kernel reading the head levels.  No
// library sort: all sort in shared memory.
// All IoU arithmetic uses explicit round-to-nearest fp32 intrinsics in the operand order of
// the CPU code it mirrors.  Two IoU policies:
//   TV  : torchvision nms_kernel_impl on class-offset boxes; the fp32 IoU is compared against
//         the largest float <= the double threshold (== torchvision's float-vs-double compare).
//   HPP : the reference's own postprocess.hpp:28-67 (same class only, early-out on empty
//         intersection, float threshold).
#include <climits>
#include <cmath>
#include <cstdlib>

#include "common.cuh"
#include "tlbr.cuh"

namespace uyd {
namespace {

constexpr int kMaxDetCap = 1024;   // kept-list capacity (the reference's MAX_DETECTIONS, gpu_postprocess.h:24)
constexpr int kAnchorBits = 22;

__device__ __forceinline__ float box_area(const float4 &b) { return __fmul_rn(__fsub_rn(b.z, b.x), __fsub_rn(b.w, b.y)); }

template <bool HPP>
__device__ __forceinline__ bool suppresses(const float4 &a, float aa, int ca, const float4 &b, float ab, int cb, float thr) {
  if (HPP) {  // postprocess.hpp:28-39,58-62
    if (ca != cb) return false;
    const float ix1 = fmaxf(a.x, b.x), iy1 = fmaxf(a.y, b.y), ix2 = fminf(a.z, b.z), iy2 = fminf(a.w, b.w);
    if (ix1 >= ix2 || iy1 >= iy2) return 0.0f > thr;
    const float inter = __fmul_rn(__fsub_rn(ix2, ix1), __fsub_rn(iy2, iy1));
    return __fdiv_rn(inter, __fsub_rn(__fadd_rn(aa, ab), inter)) > thr;
  }
  // torchvision nms_kernel_impl operand order
  const float xx1 = fmaxf(a.x, b.x), yy1 = fmaxf(a.y, b.y), xx2 = fminf(a.z, b.z), yy2 = fminf(a.w, b.w);
  const float w = fmaxf(0.f, __fsub_rn(xx2, xx1)), h = fmaxf(0.f, __fsub_rn(yy2, yy1));
  const float inter = __fmul_rn(w, h);
  // inter == 0 gives 0/x = 0 or 0/0 = NaN: never > thr for thr >= 0, so the division is skipped
  if (inter == 0.f && thr >= 0.f) return false;
  return __fdiv_rn(inter, __fsub_rn(__fadd_rn(aa, ab), inter)) > thr;
}

// =================================================================================================
// Fused per-image NMS (uyd_nms / uyd_nms_ex): ONE launch, one 1024-thread CTA per image.
//   1. scan   : best class / score per anchor (MULTI: every (anchor, class) pair), conf filter, class filter
//               (FILTER: after the best class is chosen, or per pair), 64-bit key (score code | anchor | class); the keys
//               of the current slab are captured in shared memory.  A slab is a key range holding at most
//               kFCap candidates: normally the whole image (<= kFCap candidates: one pass over the scores);
//               dense scenes are cut into consecutive ranges with a 2048-bin histogram of the key space
//               (three passes per slab; the ranges are processed best-first, so the loop usually ends after
//               the first slab because max_det boxes are kept).
//   2. sort   : bitonic sort of the slab in shared memory (keys are unique: ties in score resolve to the lower
//               anchor, exactly the stable descending sort of the reference).
//   3. greedy : as nms_greedy_kernel (chunks of 128, kept-list test by 8 threads per candidate, ballot
//               compaction, IoU bitmask among survivors, one warp resolves), boxes formed on the fly from y.
//   4. emit   : rows / anchor indices / count written by the same CTA.
// Replaces key kernel + 5 radix passes over batch x anchors + gather + greedy + emit (365 -> ~150 us at
// batch 64 x 33 600 anchors) and is what batch-1 latency needs (one dependent launch instead of eleven).
// =================================================================================================
constexpr int kFThreads = 1024, kFCap = 4096, kFChunk = 128, kFSplit = kFThreads / kFChunk, kFBins = 2048;
constexpr int kKeyAnchorShift = 8, kKeyCodeShift = 30;  // key = code << 30 | anchor << 8 | class

__device__ __forceinline__ uint64_t fused_key(float best, int j, int a, bool pos) {
  const uint32_t bits = __float_as_uint(best);
  uint32_t code;
  if (pos) code = 0x7FFFFFFFu - bits;
  else code = ~((bits & 0x80000000u) ? ~bits : (bits | 0x80000000u));
  return ((uint64_t)code << kKeyCodeShift) | ((uint64_t)a << kKeyAnchorShift) | (uint64_t)j;
}
__device__ __forceinline__ float fused_key_score(uint64_t key, bool pos) {
  const uint32_t code = (uint32_t)(key >> kKeyCodeShift);
  if (pos) return __uint_as_float(0x7FFFFFFFu - code);
  const uint32_t asc = ~code;
  return __uint_as_float((asc & 0x80000000u) ? (asc & 0x7FFFFFFFu) : ~asc);
}

struct FusedSmem {
  unsigned long long keys[kFCap];
  unsigned int hist[kFBins];
  float4 kbox[kMaxDetCap], kraw[kMaxDetCap];
  float karea[kMaxDetCap], kconf[kMaxDetCap];
  int kcls[kMaxDetCap], kanchor[kMaxDetCap];
  float4 abox[kFChunk], araw[kFChunk];
  float aarea[kFChunk], aconf[kFChunk];
  int acls[kFChunk], aanchor[kFChunk];
  __align__(16) unsigned mask[kFChunk][kFChunk / 32];
  int klist[kFChunk];
  int warp_cnt[kFThreads / 32];
  unsigned long long kmin, kmax, cut;
  int count, kept, alive;
  unsigned cmask[8];  // FILTER: bit c set = class c is kept
};

struct ClassMask {  // the class filter of uyd_nms_options as 256 bits (nc <= 256)
  unsigned w[8];
};

// MULTI: one candidate per (anchor, class) with score > conf_thr (Ultralytics multi_label=True); otherwise one per anchor,
// its best class.  FILTER: only the classes set in cmask become candidates.  The default call is <false, false>.
template <bool MULTI, bool FILTER>
__device__ __forceinline__ void nms_image(const float *__restrict__ y, int nc, int A, float conf_thr, float iou_thr, int max_nms,
                                          int max_det, float max_wh, int pos, float *__restrict__ out_det,
                                          int *__restrict__ out_idx, int *__restrict__ out_count, const ClassMask &cmask) {
  extern __shared__ __align__(16) unsigned char fused_raw[];
  FusedSmem &S = *reinterpret_cast<FusedSmem *>(fused_raw);
  const int b = blockIdx.x, tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const float *yb = y + (long long)b * (4 + nc) * A;
  if (tid == 0) {
    S.kept = 0;
    if (FILTER) {
#pragma unroll
      for (int i = 0; i < 8; ++i) S.cmask[i] = cmask.w[i];
    }
  }
  unsigned long long lo = 0ull;   // keys below lo have been consumed
  int processed = 0;
  __syncthreads();
  auto kept_class = [&](int c) { return !FILTER || ((S.cmask[c >> 5] >> (c & 31)) & 1u) != 0u; };

  // mode 0: count keys in [lo, hi), track min / max, capture the first kFCap;  mode 1: histogram over (key - kmin) >> shift
  auto scan = [&](unsigned long long hi, int mode, int shift) {
    constexpr int U = 4;  // anchors per thread and round: U independent loads in flight per class plane
    unsigned long long mn = ~0ull, mx = 0ull;  // per-thread key range, reduced once after the loop
    // every lane of the warp calls this for each of its keys (in = false for none)
    auto offer = [&](bool in, unsigned long long key) {
      if (mode == 0) {
        const unsigned bal = __ballot_sync(0xffffffffu, in);
        if (bal) {
          int base = 0;
          if (lane == 0) base = atomicAdd(&S.count, __popc(bal));
          base = __shfl_sync(0xffffffffu, base, 0);
          if (in) {
            const int slot = base + __popc(bal & ((1u << lane) - 1));
            if (slot < kFCap) S.keys[slot] = key;
            mn = key < mn ? key : mn;
            mx = key > mx ? key : mx;
          }
        }
      } else if (in) {
        atomicAdd(&S.hist[(unsigned)((key - S.kmin) >> shift)], 1u);
      }
    };
    for (int a0 = 0; a0 < A; a0 += U * kFThreads) {
      if constexpr (MULTI) {
        // class planes in order; a plane the filter drops is not read at all (c is uniform across the CTA)
        for (int c = 0; c < nc; ++c) {
          if (!kept_class(c)) continue;
          const float *pc = yb + (4ll + c) * A;
          float v[U];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int a = a0 + u * kFThreads + tid;
            v[u] = a < A ? pc[a] : -INFINITY;
          }
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int a = a0 + u * kFThreads + tid;
            bool in = false;
            unsigned long long key = 0ull;
            if (a < A && v[u] > conf_thr) {
              key = fused_key(v[u], c, a, pos != 0);
              in = key >= lo && key < hi;
            }
            offer(in, key);
          }
        }
      } else {
        float best[U];
        int bj[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int a = a0 + u * kFThreads + tid;
          best[u] = a < A ? yb[4ll * A + a] : -INFINITY;
          bj[u] = 0;
        }
        for (int c = 1; c < nc; ++c) {
          const float *pc = yb + (4ll + c) * A;
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int a = a0 + u * kFThreads + tid;
            const float v = a < A ? pc[a] : -INFINITY;
            if (v > best[u]) { best[u] = v; bj[u] = c; }   // first maximum wins
          }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int a = a0 + u * kFThreads + tid;
          bool in = false;
          unsigned long long key = 0ull;
          // the filter applies to the chosen class: an anchor whose best class is dropped does not fall back to another
          if (a < A && best[u] > conf_thr && kept_class(bj[u])) {
            key = fused_key(best[u], bj[u], a, pos != 0);
            in = key >= lo && key < hi;
          }
          offer(in, key);
        }
      }
    }
    if (mode == 0) {  // one pair of atomics per warp
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long omn = __shfl_xor_sync(0xffffffffu, mn, o), omx = __shfl_xor_sync(0xffffffffu, mx, o);
        mn = omn < mn ? omn : mn;
        mx = omx > mx ? omx : mx;
      }
      if (lane == 0 && mn <= mx) { atomicMin(&S.kmin, mn); atomicMax(&S.kmax, mx); }
    }
  };

  while (true) {
    // ---- 1. the next slab: keys in [lo, hi) with at most kFCap members ----
    unsigned long long hi = ~0ull;
    int n_slab = 0;
    while (true) {
      if (tid == 0) { S.count = 0; S.kmin = ~0ull; S.kmax = 0ull; }
      __syncthreads();
      scan(hi, 0, 0);
      __syncthreads();
      n_slab = S.count;
      if (n_slab <= kFCap) break;
      // too many: histogram the occupied key range and cut it where the cumulative count would exceed the capacity
      const unsigned long long kmin = S.kmin, span = S.kmax - S.kmin;
      int shift = 0;
      while ((span >> shift) >= (unsigned long long)kFBins) ++shift;
      for (int i = tid; i < kFBins; i += kFThreads) S.hist[i] = 0u;
      __syncthreads();
      scan(hi, 1, shift);
      __syncthreads();
      if (tid == 0) {
        unsigned cum = 0;
        int nb = 0;
        while (nb < kFBins && cum + S.hist[nb] <= (unsigned)kFCap) cum += S.hist[nb++];
        if (nb == 0) nb = 1;  // a single bin overflows: narrow the range to it (keys are unique, so this terminates)
        S.cut = kmin + ((unsigned long long)nb << shift);
      }
      __syncthreads();
      hi = S.cut;
      __syncthreads();
    }
    if (n_slab == 0) break;
    // ---- 2. bitonic sort of the slab (ascending key = descending score, ties -> lower anchor) ----
    int P = 32;
    while (P < n_slab) P <<= 1;
    for (int i = n_slab + tid; i < P; i += kFThreads) S.keys[i] = ~0ull;
    __syncthreads();
    // One compare-exchange per thread and step: pair p -> elements i = p with a zero inserted at bit log2(j), i | j.
    // For j <= 32 the 32 pairs of a warp live in its own 64 consecutive elements: those steps only need __syncwarp.
    for (int k = 2; k <= P; k <<= 1) {
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int pr = tid; pr < (P >> 1); pr += kFThreads) {
          const int i = ((pr & ~(j - 1)) << 1) | (pr & (j - 1)), q = i | j;
          const unsigned long long x = S.keys[i], z = S.keys[q];
          if ((x > z) == ((i & k) == 0)) { S.keys[i] = z; S.keys[q] = x; }
        }
        if (j > 32 || j == 1 || P > 2 * kFThreads) __syncthreads();
        else __syncwarp();
      }
    }
    // ---- 3. greedy NMS over the slab, in order, at most max_nms candidates per image in total ----
    const int take = min(n_slab, max_nms - processed);
    for (int c0 = 0; c0 < take; c0 += kFChunk) {
      const int kept = S.kept;
      if (kept >= max_det) break;
      const int i = c0 + tid / kFSplit, slice = tid % kFSplit;
      const bool valid = i < take;
      float4 bo = make_float4(0.f, 0.f, 0.f, 0.f), bx = bo;
      float ar = 0.f, sc = 0.f;
      int cl = 0, an = 0;
      bool sup = false;
      if (valid) {
        const unsigned long long key = S.keys[i];
        an = (int)((key >> kKeyAnchorShift) & ((1u << kAnchorBits) - 1));
        cl = (int)(key & 0xFF);
        sc = fused_key_score(key, pos != 0);
        const float *p = yb + an;
        const float cx = p[0], cy = p[A], w = p[2ll * A], h = p[3ll * A];
        const float hw = __fmul_rn(w, 0.5f), hh = __fmul_rn(h, 0.5f);
        bx.x = __fsub_rn(cx, hw); bx.y = __fsub_rn(cy, hh); bx.z = __fadd_rn(cx, hw); bx.w = __fadd_rn(cy, hh);
        const float off = __fmul_rn((float)cl, max_wh);
        bo.x = __fadd_rn(bx.x, off); bo.y = __fadd_rn(bx.y, off); bo.z = __fadd_rn(bx.z, off); bo.w = __fadd_rn(bx.w, off);
        ar = box_area(bo);
        for (int k = slice; k < kept; k += kFSplit)
          if (suppresses<false>(S.kbox[k], S.karea[k], S.kcls[k], bo, ar, cl, iou_thr)) { sup = true; break; }
      }
#pragma unroll
      for (int o = 1; o < kFSplit; o <<= 1) sup |= __shfl_xor_sync(0xffffffffu, sup ? 1 : 0, o) != 0;
      const bool alive = valid && !sup && slice == 0;
      const unsigned bal = __ballot_sync(0xffffffffu, alive);
      if (lane == 0) S.warp_cnt[wid] = __popc(bal);
      __syncthreads();
      int base = 0;
      for (int w2 = 0; w2 < wid; ++w2) base += S.warp_cnt[w2];
      if (tid == kFThreads - 1) S.alive = base + __popc(bal);
      if (alive) {
        const int slot = base + __popc(bal & ((1u << lane) - 1));
        S.abox[slot] = bo; S.araw[slot] = bx; S.aarea[slot] = ar; S.acls[slot] = cl; S.aconf[slot] = sc; S.aanchor[slot] = an;
      }
      __syncthreads();
      const int m = S.alive;
      const int words = (m + 31) >> 5;
      // (c) suppression bitmask among survivors (upper triangle), one item = 16 pairs so that all 1024 threads work
      for (int item = tid; item < m * words * 2; item += kFThreads) {
        const int r = item / (words * 2), cw = (item >> 1) % words, half = item & 1;
        unsigned bits = 0;
        const int j0 = cw * 32 + half * 16;
        if (j0 + 15 > r) {
          const float4 rb = S.abox[r];
          const float ra = S.aarea[r];
          const int rc = S.acls[r];
#pragma unroll 4
          for (int jj = 0; jj < 16; ++jj) {
            const int j = j0 + jj;
            if (j > r && j < m && suppresses<false>(rb, ra, rc, S.abox[j], S.aarea[j], S.acls[j], iou_thr)) bits |= 1u << jj;
          }
        }
        reinterpret_cast<unsigned short *>(&S.mask[r][cw])[half] = (unsigned short)bits;
      }
      __syncthreads();
      // (d) serial resolution by ONE thread with the removal mask in registers (the chain per kept box is
      // ffs -> one 16-byte row load -> or); the kept-list entries are copied by all threads afterwards
      if (tid == 0) {
        unsigned rem[kFChunk / 32] = {0u, 0u, 0u, 0u};
        int k = kept;
#pragma unroll
        for (int w = 0; w < kFChunk / 32; ++w) {
          if (w >= words) break;
          const unsigned in_range = (w * 32 + 32 <= m) ? ~0u : ((1u << (m - w * 32)) - 1u);
          unsigned alive_bits = ~rem[w] & in_range;
          while (alive_bits && k < max_det) {
            const int bit = __ffs(alive_bits) - 1, r = w * 32 + bit;
            S.klist[k - kept] = r;
            ++k;
            const uint4 row = *reinterpret_cast<const uint4 *>(S.mask[r]);
            rem[0] |= row.x; rem[1] |= row.y; rem[2] |= row.z; rem[3] |= row.w;
            alive_bits = ~rem[w] & in_range & ~((2u << bit) - 1u);
          }
        }
        S.kept = k;
      }
      __syncthreads();
      const int k_new = S.kept - kept;
      if (tid < k_new) {
        const int r = S.klist[tid], k = kept + tid;
        S.kbox[k] = S.abox[r]; S.kraw[k] = S.araw[r]; S.karea[k] = S.aarea[r]; S.kcls[k] = S.acls[r];
        S.kconf[k] = S.aconf[r]; S.kanchor[k] = S.aanchor[r];
      }
      __syncthreads();
    }
    processed += take;
    if (hi == ~0ull || S.kept >= max_det || processed >= max_nms) break;
    lo = hi;
    __syncthreads();
  }
  // ---- 4. emit ----
  __syncthreads();
  const int kept = S.kept;
  for (int k = tid; k < max_det; k += kFThreads) {  // every row is defined: zeros / index -1 past the count
    float *o = out_det + ((long long)b * max_det + k) * 6;
    if (k < kept) {
      const float4 r = S.kraw[k];
      o[0] = r.x; o[1] = r.y; o[2] = r.z; o[3] = r.w; o[4] = S.kconf[k]; o[5] = (float)S.kcls[k];
    } else {
      o[0] = o[1] = o[2] = o[3] = o[4] = o[5] = 0.f;
    }
    if (out_idx) out_idx[(long long)b * max_det + k] = k < kept ? S.kanchor[k] : -1;
  }
  if (tid == 0) out_count[b] = kept;
}

// One entry point for the four instances (bit 1 of mode: MULTI, bit 0: FILTER), so the library keeps a single NMS
// kernel symbol; the mode is uniform over the launch and each CTA runs exactly one inlined instance.
__global__ void __launch_bounds__(kFThreads, 1) nms_image_kernel(const float *__restrict__ y, int nc, int A, float conf_thr,
                                                                 float iou_thr, int max_nms, int max_det, float max_wh, int pos,
                                                                 float *__restrict__ out_det, int *__restrict__ out_idx,
                                                                 int *__restrict__ out_count, int mode, ClassMask cmask) {
  switch (mode) {
    case 0: nms_image<false, false>(y, nc, A, conf_thr, iou_thr, max_nms, max_det, max_wh, pos, out_det, out_idx, out_count, cmask); break;
    case 1: nms_image<false, true>(y, nc, A, conf_thr, iou_thr, max_nms, max_det, max_wh, pos, out_det, out_idx, out_count, cmask); break;
    case 2: nms_image<true, false>(y, nc, A, conf_thr, iou_thr, max_nms, max_det, max_wh, pos, out_det, out_idx, out_count, cmask); break;
    default: nms_image<true, true>(y, nc, A, conf_thr, iou_thr, max_nms, max_det, max_wh, pos, out_det, out_idx, out_count, cmask); break;
  }
}

// =================================================================================================
// Candidate-list variant (custom head, postprocess.hpp:44-67 semantics): ONE launch, one 1024-thread CTA per image.
// Where the candidates come from is the template's source (RecordSource, TlbrSource below):
//   1. slab   : 64-bit key (descending-confidence code | tie) of every candidate, the keys of the current slab and
//               their slots captured in shared memory; more than kRCap candidates are cut into consecutive key
//               ranges with a histogram (as in nms_image_kernel) and consumed best-first.
//   2. sort   : bitonic sort of the (key, slot) pairs in shared memory.  Ties in confidence resolve to the lower
//               cell index (or slot), which freezes the order the header's std::sort leaves unspecified.
//   3. greedy : the max_nms best candidates in chunks of 128 (kept-list test by 8 threads per candidate, ballot
//               compaction, IoU bitmask among survivors, serial resolution), same class only, IoU > thr; the box and
//               class of a slot come from the source.
//   4. emit   : by the source -- records: survivors compacted in kept order (out), or, INPLACE, the first n records
//               of `dets` rewritten in sorted order with valid = 1 / 0, which is what run_gpu_nms leaves behind
//               (gpu_postprocess.cu:366-387); TLBR: [max_det, 6] rows of the image plus its count.
// =================================================================================================
constexpr int kRThreads = 1024, kRCap = 4096, kRChunk = 128, kRSplit = kRThreads / kRChunk, kRBins = 2048;

struct RecSmem {
  unsigned long long keys[kRCap];
  int slot[kRCap];
  unsigned int hist[kRBins];
  float4 kbox[kMaxDetCap];
  float karea[kMaxDetCap];
  int kcls[kMaxDetCap], kslot[kMaxDetCap];
  float4 abox[kRChunk];
  float aarea[kRChunk];
  int acls[kRChunk], aslot[kRChunk];
  __align__(16) unsigned mask[kRChunk][kRChunk / 32];
  int klist[kRChunk];
  int warp_cnt[kRThreads / 32];
  unsigned long long kmin, kmax, cut;
  int count, kept, alive;
};

__device__ __forceinline__ unsigned long long record_key(float conf, unsigned tie) {
  const uint32_t bits = __float_as_uint(conf);
  const uint32_t asc = (bits & 0x80000000u) ? ~bits : (bits | 0x80000000u);
  return ((unsigned long long)(~asc) << 32) | tie;
}

// Records (uyd_nms_detections, uyd_nms_detections_inplace): the first min(*d_count or n_host, cap) uyd_detection
// records of `dets`, tie = cell_idx[i] (or the slot i when NULL); one CTA.
template <bool INPLACE>
struct RecordSource {
  static constexpr bool kInplace = INPLACE;
  uyd_detection *dets;
  const int *cell_idx, *d_count;
  int n_host, cap;
  uyd_detection *out;
  int *d_out_count;

  __device__ int count() const { return min(d_count ? *d_count : n_host, cap); }
  __device__ bool key(int i, unsigned long long &k) const {
    k = record_key(dets[i].confidence, cell_idx ? (unsigned)cell_idx[i] : (unsigned)i);
    return true;
  }
  __device__ void candidate(int slot, float4 &bx, int &cl, float &conf) const {
    const uyd_detection d = dets[slot];
    bx = make_float4(d.x1, d.y1, d.x2, d.y2);
    cl = d.class_id;
    conf = d.confidence;
  }
  __device__ void emit(const int *kslot, int kept, int tid) const {
    for (int k = tid; k < kept; k += kRThreads) {
      if (INPLACE) {
        dets[kslot[k]].valid = 1;
      } else {
        uyd_detection d = dets[kslot[k]];
        d.valid = 1;
        out[k] = d;
      }
    }
    if (tid == 0 && d_out_count) *d_out_count = kept;
  }
};

// TLBR head levels (uyd_nms_tlbr): image blockIdx.x of heads[l] = [batch, grid_h[l], grid_w[l], nc + 4] fp32 (class
// logits, then l, t, r, b).  Slot = cell = base[l] + row-major cell index of level l, which is also the tie; the box,
// confidence and class of a slot are recomputed from the head by tlbr_cell (the statement of decode_tlbr_kernel)
// wherever they are needed, so no record buffer exists.
constexpr int kMaxLevels = 8;

struct TlbrSource {
  static constexpr bool kInplace = false;
  const float *head[kMaxLevels];
  int gw[kMaxLevels], stride[kMaxLevels];
  int base[kMaxLevels + 1];  // base[nl] = cells per image
  int nl, nc, strict, max_det;
  float thr, q;
  float *out_det;
  int *out_count;

  __device__ int count() const { return base[nl]; }
  // level of cell i selected with static indices only (no local-memory copy of the parameter arrays)
  template <bool BOX>
  __device__ bool cell(int i, float &conf, int &cl, float4 &bx) const {
    const float *h = head[0];
    int b0 = 0, w = gw[0], st = stride[0], n = base[1];
#pragma unroll
    for (int j = 1; j < kMaxLevels; ++j)
      if (j < nl && i >= base[j]) { h = head[j]; b0 = base[j]; w = gw[j]; st = stride[j]; n = base[j + 1] - base[j]; }
    const int g = i - b0;
    const float *row = h + ((long long)blockIdx.x * n + g) * (nc + 4);
    return tlbr_cell<BOX>(row, row + nc, 1, nc, g % w, g / w, st, thr, q, strict, conf, cl, bx);
  }
  __device__ bool key(int i, unsigned long long &k) const {
    float conf;
    int cl;
    float4 bx;
    if (!cell<false>(i, conf, cl, bx)) return false;
    k = record_key(conf, (unsigned)i);
    return true;
  }
  __device__ void candidate(int slot, float4 &bx, int &cl, float &conf) const { cell<true>(slot, conf, cl, bx); }
  __device__ void emit(const int *kslot, int kept, int tid) const {
    for (int k = tid; k < max_det; k += kRThreads) {  // every row is defined: zeros past the count
      float *o = out_det + ((long long)blockIdx.x * max_det + k) * 6;
      if (k < kept) {
        float4 bx;
        int cl;
        float conf;
        candidate(kslot[k], bx, cl, conf);
        o[0] = bx.x; o[1] = bx.y; o[2] = bx.z; o[3] = bx.w; o[4] = conf; o[5] = (float)cl;
      } else {
        o[0] = o[1] = o[2] = o[3] = o[4] = o[5] = 0.f;
      }
    }
    if (tid == 0) out_count[blockIdx.x] = kept;
  }
};

template <class Src>
__global__ void __launch_bounds__(kRThreads, 1) nms_records_kernel(const Src src, float iou_thr, int max_nms, int max_keep) {
  constexpr bool INPLACE = Src::kInplace;
  extern __shared__ __align__(16) unsigned char rec_raw[];
  RecSmem &S = *reinterpret_cast<RecSmem *>(rec_raw);
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  const int n = src.count();
  if (tid == 0) S.kept = 0;
  unsigned long long lo = 0ull;
  int processed = 0;
  __syncthreads();

  auto scan = [&](unsigned long long hi, int mode, int shift) {
    unsigned long long mn = ~0ull, mx = 0ull;
    for (int i0 = 0; i0 < n; i0 += kRThreads) {
      const int i = i0 + tid;
      bool in = false;
      unsigned long long key = 0ull;
      if (i < n && src.key(i, key)) in = key >= lo && key < hi;
      if (mode == 0) {
        const unsigned bal = __ballot_sync(0xffffffffu, in);
        if (bal) {
          int base = 0;
          if (lane == 0) base = atomicAdd(&S.count, __popc(bal));
          base = __shfl_sync(0xffffffffu, base, 0);
          if (in) {
            const int s = base + __popc(bal & ((1u << lane) - 1));
            if (s < kRCap) { S.keys[s] = key; S.slot[s] = i; }
            mn = key < mn ? key : mn;
            mx = key > mx ? key : mx;
          }
        }
      } else if (in) {
        atomicAdd(&S.hist[(unsigned)((key - S.kmin) >> shift)], 1u);
      }
    }
    if (mode == 0) {
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long omn = __shfl_xor_sync(0xffffffffu, mn, o), omx = __shfl_xor_sync(0xffffffffu, mx, o);
        mn = omn < mn ? omn : mn;
        mx = omx > mx ? omx : mx;
      }
      if (lane == 0 && mn <= mx) { atomicMin(&S.kmin, mn); atomicMax(&S.kmax, mx); }
    }
  };

  while (true) {
    // ---- 1. the next slab ----
    unsigned long long hi = ~0ull;
    int n_slab = 0;
    while (true) {
      if (tid == 0) { S.count = 0; S.kmin = ~0ull; S.kmax = 0ull; }
      __syncthreads();
      scan(hi, 0, 0);
      __syncthreads();
      n_slab = S.count;
      if (n_slab <= kRCap) break;
      const unsigned long long kmin = S.kmin, span = S.kmax - S.kmin;
      int shift = 0;
      while ((span >> shift) >= (unsigned long long)kRBins) ++shift;
      for (int i = tid; i < kRBins; i += kRThreads) S.hist[i] = 0u;
      __syncthreads();
      scan(hi, 1, shift);
      __syncthreads();
      if (tid == 0) {
        unsigned cum = 0;
        int nb = 0;
        while (nb < kRBins && cum + S.hist[nb] <= (unsigned)kRCap) cum += S.hist[nb++];
        if (nb == 0) nb = 1;  // keys are unique (tie bits), so narrowing to one bin terminates
        S.cut = kmin + ((unsigned long long)nb << shift);
      }
      __syncthreads();
      hi = S.cut;
      __syncthreads();
    }
    if (n_slab == 0) break;
    // ---- 2. bitonic sort of the (key, slot) pairs ----
    int P = 32;
    while (P < n_slab) P <<= 1;
    for (int i = n_slab + tid; i < P; i += kRThreads) { S.keys[i] = ~0ull; S.slot[i] = -1; }
    __syncthreads();
    for (int k = 2; k <= P; k <<= 1) {
      for (int j = k >> 1; j > 0; j >>= 1) {
        for (int pr = tid; pr < (P >> 1); pr += kRThreads) {
          const int i = ((pr & ~(j - 1)) << 1) | (pr & (j - 1)), q = i | j;
          const unsigned long long x = S.keys[i], z = S.keys[q];
          if ((x > z) == ((i & k) == 0)) {
            S.keys[i] = z; S.keys[q] = x;
            const int sx = S.slot[i];
            S.slot[i] = S.slot[q]; S.slot[q] = sx;
          }
        }
        if (j > 32 || j == 1 || P > 2 * kRThreads) __syncthreads();
        else __syncwarp();
      }
    }
    if constexpr (INPLACE) {  // n <= kRThreads: one record per thread, rewritten in sorted order (valid decided in step 4)
      uyd_detection rec;
      if (tid < n_slab) rec = src.dets[S.slot[tid]];
      __syncthreads();
      if (tid < n_slab) {
        S.keys[tid] = rec.valid ? 1ull : 0ull;  // records that arrive invalid neither suppress nor survive
        rec.valid = 0;
        src.dets[tid] = rec;
        S.slot[tid] = tid;
      }
      __syncthreads();
    }
    // ---- 3. greedy over the slab, in order, at most max_nms candidates per image in total ----
    const int take = min(n_slab, max_nms - processed);
    for (int c0 = 0; c0 < take; c0 += kRChunk) {
      const int kept = S.kept;
      if (kept >= max_keep) break;
      const int i = c0 + tid / kRSplit, slice = tid % kRSplit;
      bool valid = i < take;
      float4 bx = make_float4(0.f, 0.f, 0.f, 0.f);
      float ar = 0.f, conf;
      int cl = 0, sl = 0;
      bool sup = false;
      if (valid) {
        sl = S.slot[i];
        src.candidate(sl, bx, cl, conf);
        if (INPLACE && S.keys[i] == 0ull) valid = false;
        ar = box_area(bx);
        if (valid)
          for (int k = slice; k < kept; k += kRSplit)
            if (suppresses<true>(S.kbox[k], S.karea[k], S.kcls[k], bx, ar, cl, iou_thr)) { sup = true; break; }
      }
#pragma unroll
      for (int o = 1; o < kRSplit; o <<= 1) sup |= __shfl_xor_sync(0xffffffffu, sup ? 1 : 0, o) != 0;
      const bool alive = valid && !sup && slice == 0;
      const unsigned bal = __ballot_sync(0xffffffffu, alive);
      if (lane == 0) S.warp_cnt[wid] = __popc(bal);
      __syncthreads();
      int base = 0;
      for (int w2 = 0; w2 < wid; ++w2) base += S.warp_cnt[w2];
      if (tid == kRThreads - 1) S.alive = base + __popc(bal);
      if (alive) {
        const int s = base + __popc(bal & ((1u << lane) - 1));
        S.abox[s] = bx; S.aarea[s] = ar; S.acls[s] = cl; S.aslot[s] = sl;
      }
      __syncthreads();
      const int m = S.alive;
      const int words = (m + 31) >> 5;
      for (int item = tid; item < m * words * 2; item += kRThreads) {
        const int r = item / (words * 2), cw = (item >> 1) % words, half = item & 1;
        unsigned bits = 0;
        const int j0 = cw * 32 + half * 16;
        if (j0 + 15 > r) {
          const float4 rb = S.abox[r];
          const float ra = S.aarea[r];
          const int rc = S.acls[r];
#pragma unroll 4
          for (int jj = 0; jj < 16; ++jj) {
            const int j = j0 + jj;
            if (j > r && j < m && suppresses<true>(rb, ra, rc, S.abox[j], S.aarea[j], S.acls[j], iou_thr)) bits |= 1u << jj;
          }
        }
        reinterpret_cast<unsigned short *>(&S.mask[r][cw])[half] = (unsigned short)bits;
      }
      __syncthreads();
      if (tid == 0) {
        unsigned rem[kRChunk / 32] = {0u, 0u, 0u, 0u};
        int k = kept;
#pragma unroll
        for (int w = 0; w < kRChunk / 32; ++w) {
          if (w >= words) break;
          const unsigned in_range = (w * 32 + 32 <= m) ? ~0u : ((1u << (m - w * 32)) - 1u);
          unsigned alive_bits = ~rem[w] & in_range;
          while (alive_bits && k < max_keep) {
            const int bit = __ffs(alive_bits) - 1, r = w * 32 + bit;
            S.klist[k - kept] = r;
            ++k;
            const uint4 row = *reinterpret_cast<const uint4 *>(S.mask[r]);
            rem[0] |= row.x; rem[1] |= row.y; rem[2] |= row.z; rem[3] |= row.w;
            alive_bits = ~rem[w] & in_range & ~((2u << bit) - 1u);
          }
        }
        S.kept = k;
      }
      __syncthreads();
      const int k_new = S.kept - kept;
      if (tid < k_new) {
        const int r = S.klist[tid], k = kept + tid;
        S.kbox[k] = S.abox[r]; S.karea[k] = S.aarea[r]; S.kcls[k] = S.acls[r]; S.kslot[k] = S.aslot[r];
      }
      __syncthreads();
    }
    processed += take;
    if (INPLACE || hi == ~0ull || S.kept >= max_keep || processed >= max_nms) break;
    lo = hi;
    __syncthreads();
  }
  // ---- 4. emit ----
  __syncthreads();
  src.emit(S.kslot, S.kept, tid);
}

// Ordered stream compaction of the valid records (copy_valid_detections_to_host's cub::DeviceSelect::If,
// gpu_postprocess.cu:412-416) for n <= 1024: one CTA, ballot + warp prefix.
__global__ void __launch_bounds__(kRThreads) compact_valid_kernel(const uyd_detection *dets, int n, uyd_detection *out, int *d_out_count) {
  __shared__ int warp_cnt[kRThreads / 32];
  const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
  uyd_detection d;
  bool v = false;
  if (tid < n) { d = dets[tid]; v = d.valid != 0; }
  const unsigned bal = __ballot_sync(0xffffffffu, v);
  if (lane == 0) warp_cnt[wid] = __popc(bal);
  __syncthreads();
  int base = 0;
  for (int w = 0; w < wid; ++w) base += warp_cnt[w];
  if (v) out[base + __popc(bal & ((1u << lane) - 1))] = d;
  if (tid == kRThreads - 1) *d_out_count = base + __popc(bal);
}

template <class Src>
int launch_candidates(const Src &src, int grid, float iou_thr, int max_nms, int max_keep, cudaStream_t s) {
  if (int e = smem_optin(nms_records_kernel<Src>, sizeof(RecSmem))) return e;
  nms_records_kernel<Src><<<grid, kRThreads, sizeof(RecSmem), s>>>(src, iou_thr, max_nms, max_keep);
  return (int)cudaGetLastError();
}

}  // namespace
}  // namespace uyd

extern "C" size_t uyd_nms_workspace_bytes(int batch, int anchors) {  // kept for ABI stability: the kernel needs none
  return (batch > 0 && anchors > 0) ? 256 : 0;
}

extern "C" int uyd_nms_ex(uyd_ctx *ctx, const float *y, int batch, int nc, int anchors, float conf_thr, double iou_thr,
                          int max_nms, int max_det, float max_wh, const uyd_nms_options *opt, float *out_det, int *out_idx,
                          int *out_count, uyd_stream stream) {
  using namespace uyd;
  UYD_REQUIRE(y && out_det && out_count && batch > 0 && nc > 0 && anchors > 0, UYD_E_ARG, "uyd_nms: bad arguments");
  UYD_REQUIRE(!opt || (opt->num_filter_classes >= 0 && (opt->num_filter_classes == 0 || opt->filter_classes)), UYD_E_ARG,
              "uyd_nms_ex: num_filter_classes must be >= 0, and > 0 only with a filter_classes array");
  DeviceGuard guard(ctx_device(ctx));
  UYD_REQUIRE(nc <= 256 && anchors < (1 << kAnchorBits), UYD_E_UNSUPPORTED, "uyd_nms: nc <= 256 and anchors < 4M per image");
  UYD_REQUIRE(max_det > 0 && max_det <= kMaxDetCap, UYD_E_UNSUPPORTED, "uyd_nms: max_det <= %d", kMaxDetCap);
  const bool multi = opt && opt->multi_label && nc > 1;  // Ultralytics: multi_label &= nc > 1
  const bool filter = opt && opt->filter_classes;
  const long long cands = multi ? (long long)anchors * nc : anchors;  // at most this many candidates per image
  if (max_nms > cands) max_nms = (int)cands;
  UYD_REQUIRE(max_nms > 0, UYD_E_ARG, "uyd_nms: max_nms must be positive");
  ClassMask cm{};
  if (filter)  // ids outside [0, nc) match no class
    for (int i = 0; i < opt->num_filter_classes; ++i) {
      const int c = opt->filter_classes[i];
      if (c >= 0 && c < nc) cm.w[c >> 5] |= 1u << (c & 31);
    }
  float thr_f = (float)iou_thr;  // largest float <= the double threshold
  if ((double)thr_f > iou_thr) thr_f = nextafterf(thr_f, -INFINITY);
  if (int e = smem_optin(nms_image_kernel, sizeof(FusedSmem))) return e;
  nms_image_kernel<<<batch, kFThreads, sizeof(FusedSmem), (cudaStream_t)stream>>>(
      y, nc, anchors, conf_thr, thr_f, max_nms, max_det, max_wh, conf_thr >= 0.f ? 1 : 0, out_det, out_idx, out_count,
      (multi ? 2 : 0) | (filter ? 1 : 0), cm);
  UYD_CUDA(cudaGetLastError());
  return UYD_OK;
}

extern "C" int uyd_nms(uyd_ctx *ctx, const float *y, int batch, int nc, int anchors, float conf_thr, double iou_thr,
                       int max_nms, int max_det, float max_wh, void *workspace, size_t workspace_bytes, float *out_det,
                       int *out_idx, int *out_count, uyd_stream stream) {
  (void)workspace; (void)workspace_bytes;
  return uyd_nms_ex(ctx, y, batch, nc, anchors, conf_thr, iou_thr, max_nms, max_det, max_wh, nullptr, out_det, out_idx,
                    out_count, stream);
}

extern "C" size_t uyd_nms_detections_workspace_bytes(int cap) { return cap > 0 ? 256 : 0; }  // kept for ABI stability: unused

extern "C" int uyd_nms_detections(uyd_ctx *ctx, const uyd_detection *dets, const int *cell_idx, const int *d_count, int cap,
                                  float iou_thr, void *workspace, size_t workspace_bytes, uyd_detection *out,
                                  int *d_out_count, uyd_stream stream) {
  using namespace uyd;
  (void)workspace; (void)workspace_bytes;
  UYD_REQUIRE(dets && d_count && out && d_out_count && cap > 0, UYD_E_ARG, "uyd_nms_detections: bad arguments");
  DeviceGuard guard(ctx_device(ctx));
  UYD_REQUIRE(out != dets, UYD_E_ARG, "uyd_nms_detections: out must not alias dets (use uyd_nms_detections_inplace)");
  const RecordSource<false> src{const_cast<uyd_detection *>(dets), cell_idx, d_count, 0, cap, out, d_out_count};
  return launch_candidates(src, 1, iou_thr, INT_MAX, kMaxDetCap, (cudaStream_t)stream);
}

extern "C" int uyd_nms_detections_inplace(uyd_ctx *ctx, uyd_detection *dets, const int *cell_idx, int n, float iou_thr,
                                          int *d_out_count, uyd_stream stream) {
  using namespace uyd;
  UYD_REQUIRE(dets && n >= 0 && n <= kMaxDetCap, UYD_E_ARG, "uyd_nms_detections_inplace: 0 <= n <= %d", kMaxDetCap);
  DeviceGuard guard(ctx_device(ctx));
  if (n == 0) return UYD_OK;
  const RecordSource<true> src{dets, cell_idx, nullptr, n, n, nullptr, d_out_count};
  return launch_candidates(src, 1, iou_thr, INT_MAX, kMaxDetCap, (cudaStream_t)stream);
}

extern "C" int uyd_nms_tlbr(uyd_ctx *ctx, const float *const *heads, const int *grid_h, const int *grid_w, const int *strides,
                            int nl, int batch, int num_classes, float conf_thr, float conformal_q, int strict, float iou_thr,
                            int max_nms, int max_det, float *out_det, int *out_count, uyd_stream stream) {
  using namespace uyd;
  UYD_REQUIRE(nl >= 1 && heads && grid_h && grid_w && strides && out_det && out_count, UYD_E_ARG,
              "uyd_nms_tlbr: at least one level and non-NULL pointers required");
  UYD_REQUIRE(nl <= kMaxLevels, UYD_E_UNSUPPORTED, "uyd_nms_tlbr: at most %d levels (got %d)", kMaxLevels, nl);
  UYD_REQUIRE(batch > 0 && num_classes > 0 && max_nms >= 0, UYD_E_ARG, "uyd_nms_tlbr: batch, num_classes > 0, max_nms >= 0");
  UYD_REQUIRE(max_det >= 1 && max_det <= kMaxDetCap, UYD_E_UNSUPPORTED, "uyd_nms_tlbr: 1 <= max_det <= %d (got %d)", kMaxDetCap,
              max_det);
  TlbrSource src{};
  long long cells = 0;
  for (int l = 0; l < nl; ++l) {
    UYD_REQUIRE(heads[l] && grid_h[l] > 0 && grid_w[l] > 0 && strides[l] > 0, UYD_E_ARG,
                "uyd_nms_tlbr: level %d: NULL head or non-positive grid / stride", l);
    UYD_REQUIRE((reinterpret_cast<uintptr_t>(heads[l]) & (alignof(float) - 1)) == 0, UYD_E_ARG,
                "uyd_nms_tlbr: level %d: head rows must start on a float boundary", l);
    src.head[l] = heads[l];
    src.gw[l] = grid_w[l];
    src.stride[l] = strides[l];
    src.base[l] = (int)cells;
    cells += (long long)grid_h[l] * grid_w[l];
    UYD_REQUIRE(cells < (1ll << 31), UYD_E_UNSUPPORTED, "uyd_nms_tlbr: fewer than 2^31 cells per image");
  }
  src.base[nl] = (int)cells;
  src.nl = nl; src.nc = num_classes; src.strict = strict ? 1 : 0; src.max_det = max_det;
  src.thr = conf_thr; src.q = conformal_q; src.out_det = out_det; src.out_count = out_count;
  DeviceGuard guard(ctx_device(ctx));
  return launch_candidates(src, batch, iou_thr, max_nms > 0 ? max_nms : INT_MAX, max_det, (cudaStream_t)stream);
}

extern "C" int uyd_compact_valid(uyd_ctx *ctx, const uyd_detection *dets, int n, uyd_detection *out, int *d_out_count,
                                 uyd_stream stream) {
  using namespace uyd;
  UYD_REQUIRE(dets && out && d_out_count && n >= 0 && n <= kMaxDetCap, UYD_E_ARG, "uyd_compact_valid: 0 <= n <= %d", kMaxDetCap);
  DeviceGuard guard(ctx_device(ctx));
  compact_valid_kernel<<<1, kRThreads, 0, (cudaStream_t)stream>>>(dets, n, out, d_out_count);
  return (int)cudaGetLastError();
}
