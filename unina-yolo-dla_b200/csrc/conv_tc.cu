// Implicit-GEMM convolution on tcgen05 tensor cores (sm_100a), NHWC bf16, fp32 accumulate in
// TMEM, TMA-staged activation and weight tiles.  Replaces the Conv+BN(folded)+ReLU layers the
// reference runs through TensorRT / cuDNN (ConvBlock.forward model.py:49-50, Ultralytics Conv).
//
// GEMM view: D[M = 128 output pixels, N = Cout] += A[M, K] * B[N, K]^T, K = taps * Cin.
// Both operands are K-major in shared memory in the canonical UMMA swizzled layout whose row
// width equals one channel block (CB channels = 32/64/128 bytes -> SWIZZLE_32B/64B/128B).
//
// Three ways of forming A (all im2col-free, the activation tensor is only ever read by TMA):
//   FLAT   (1x1)        : a tile is 128 consecutive pixels of the flattened [N*H*W, C] view;
//                         one 2-D TMA box per channel block.
//   HALO   (3x3, s = 1) : a tile is 16 rows x 8 columns of output pixels.  The (16+2) x (8+2)
//                         input halo of one channel block is loaded ONCE (18 row TMAs, each row
//                         padded to a 16-pixel pitch so every 8-pixel group stays inside one
//                         swizzle atom); the nine filter taps are nine UMMA descriptors that
//                         start at (r * pitch + s) pixels into that halo.  Activation bytes
//                         cross L2->SMEM 1.4x instead of 9x.
//   PERTAP (3x3, any s) : one TMA box per (channel block, tap); stride 2 uses the TMA
//                         traversal stride.  Always swizzle-atom aligned; also the fallback
//                         for HALO.
//
// Warp roles (576 threads, one persistent CTA per SM): warp 0 = TMA producer, warp 1 = TMEM
// allocator + single-thread tcgen05.mma issuer (elect.sync), warps 2..17 = four epilogue warpgroups
// taking tiles round-robin (tcgen05.ld -> bias -> ReLU -> residual -> bf16/fp32 -> staged, row-coalesced
// global stores).  Three mbarrier pipelines: smem full/empty, TMEM full/empty (four accumulators),
// weights-resident.
#include "common.cuh"
#include "tc_ptx.cuh"

namespace uyd {

// PAIRS (3x3 stride 2, Cin = 32): ncu of PERTAP showed nothing saturated but the TMA unit -- nine boxes with traversal
// stride 2 are 1152 separate 64-byte segments per tile (~6 cycles each).  Here ONE contiguous box [34 rows][9 pixel
// pairs][2 x 32 channels] is loaded per tile (the dense NHWC input viewed as [n][h][w/2][2 c]): an A row is a PAIR of pixels =
// 128 bytes (SWIZZLE_128B), the even / odd pixel of the pair is a 64-byte offset inside the row (like a k-step),
// the previous pair a 128-byte row shift (like a HALO tap), and the vertical stride 2 is the descriptor's stride
// between 8-row groups (2 box rows).  Same 18 MMAs per tile, every input byte fetched once.
enum { TC_FLAT = 0, TC_HALO = 1, TC_PERTAP = 2, TC_PAIRS = 3 };
constexpr int kPairRows = 34, kPairCols = 9;  // box of a 16 x 8 output tile: input rows 2 y0 - 1 .., pixel pairs x0 - 1 ..

struct TcParams {
  int mode;
  int H, W;              // output extent
  int n0, nb;            // image range handled by this launch
  int ncb, cb_bytes;     // channel blocks, bytes per block row (32/64/128)
  int taps;              // 1 or 9
  int stride;            // conv stride (PERTAP)
  int N;                 // UMMA N (cout padded to a multiple of 16)
  int cout;
  int tiles_x, tiles_y;  // HALO / PERTAP tiling of one image
  long long total_tiles;
  int stages;
  int nacc;              // TMEM accumulator stages (nacc * N columns)
  int dual;              // 1: two MMA-issuing warps take alternate tiles (stages is a multiple of 2 x blocks per tile, so a
                         // ring slot always belongs to the same issuer and each issuer runs the ordinary parity protocol)
  int ngroups;           // active epilogue warpgroups (1, 2 or 4: as many as the staging tiles leave room for)
  int halo_pitch;        // HALO: pixels per halo row in shared memory (10 = dense single TMA box, 16 = padded rows)
  int stage_pitch;       // bytes per row of the epilogue staging tile (0 = direct stores)
  int i8;                // 1: int8 operands, int32 accumulate (kind::i8), requant epilogue
  int out_kind;          // i8 path: 0 = bf16, 1 = fp32, 2 = int8 (re-quantised with out_scale), 3 = int8 of the bf16-rounded value
  float out_scale;
  const float *mult;     // i8 path: per-channel fp32 multiplier m_c
  uint32_t blk_bytes;    // one A block in shared memory
  uint32_t tx_bytes;     // bytes TMA delivers per A block
  uint32_t w_bytes;      // resident weights
  uint32_t sbo_a;        // stride between 8-row groups of A
  uint32_t idesc;
  uint32_t layout_type;  // UMMA smem-descriptor swizzle code
  int base_offset_mode;  // HALO: 1 = descriptor base_offset = (addr >> 7) & 7, 0 = always 0
  void *out;
  int out_pitch, out_f32;
  const __nv_bfloat16 *res;
  int res_pitch;
  const float *bias;
  int relu;
  const float *pre;      // fp32 [n, H/2, W/2, cout] partial sums added (nearest x2 upsampled) before the activation, or null
  // ---- BIG variant (conv_tc_big_kernel: weights streamed, two M-tiles per CTA) ----
  int big;               // 1: weights do not fit shared memory
  int wstages;           // weight pipeline stages
  uint32_t wblk_bytes;   // one weight block (N x 128 B) in shared memory
  uint32_t tile_off;     // byte offset of the second M-tile inside an A block
  int pairs_x;           // 16 x 16 pixel regions per image row (HALO / PERTAP)
  unsigned tpi, m_tpi, m_tx;  // tiles (pairs) per image and the fastdiv magics of tiles-per-image / tiles per row
};

namespace {

constexpr int kEpiGroups = 4;                   // epilogue warpgroups taking tiles round-robin (latency hiding: the epilogue
                                                // of a tile is a long dependent chain: TMEM load -> math -> staging -> stores)
constexpr int kThreads = 64 + 128 * kEpiGroups + 32;  // TMA warp + MMA warp + kEpiGroups x 4 epilogue warps + second MMA warp
constexpr int kIssuer2 = kThreads / 32 - 1;           // ncu (profiles/r03_issue.md): the single issuing warp executed ~230
                                                      // instructions per 18-MMA tile and WAS the tile period (2135 cycles vs 864
                                                      // of tensor time); two issuers take alternate tiles (different accumulators)
constexpr uint32_t kTailFixed = 1536 + 8 * 128 * kEpiGroups;  // barriers + bias + mult | row -> pixel map
constexpr int kHaloRows = 18, kTileH = 16, kTileW = 8;
constexpr int kMaxAcc = 4;  // TMEM accumulator stages

// One 16-column chunk of one accumulator row: bias -> ReLU -> residual -> store.
__device__ __forceinline__ void epilogue_chunk(const uint32_t (&raw)[16], const float *bias_s, int c0, long long pix,
                                               const TcParams &p, long long ppix) {
  float v[16];
#pragma unroll
  for (int i = 0; i < 4; ++i) {  // 16-byte broadcast loads of the bias vector
    const float4 q = reinterpret_cast<const float4 *>(bias_s + c0)[i];
    v[4 * i] = q.x; v[4 * i + 1] = q.y; v[4 * i + 2] = q.z; v[4 * i + 3] = q.w;
  }
  if (ppix >= 0) {  // partial sums of the low-resolution half (cout % 16 == 0, checked on the host)
    const float4 *pp = reinterpret_cast<const float4 *>(p.pre + ppix * p.cout + c0);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 q = pp[i];
      v[4 * i] += q.x; v[4 * i + 1] += q.y; v[4 * i + 2] += q.z; v[4 * i + 3] += q.w;
    }
  }
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const float x = __uint_as_float(raw[i]) + v[i];
    v[i] = p.relu ? fmaxf(x, 0.f) : x;
  }
  const int nvalid = p.cout - c0;
  if (nvalid >= 16) {
    if (p.res) {
      const __nv_bfloat16 *rp = p.res + pix * p.res_pitch + c0;
      const uint4 r0 = *reinterpret_cast<const uint4 *>(rp), r1 = *reinterpret_cast<const uint4 *>(rp + 8);
      const __nv_bfloat162 *h0 = reinterpret_cast<const __nv_bfloat162 *>(&r0);
      const __nv_bfloat162 *h1 = reinterpret_cast<const __nv_bfloat162 *>(&r1);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 f0 = __bfloat1622float2(h0[i]), f1 = __bfloat1622float2(h1[i]);
        v[2 * i] += f0.x; v[2 * i + 1] += f0.y; v[8 + 2 * i] += f1.x; v[8 + 2 * i + 1] += f1.y;
      }
    }
    if (p.out_f32) {
      float *op = reinterpret_cast<float *>(p.out) + pix * p.out_pitch + c0;
#pragma unroll
      for (int i = 0; i < 16; i += 4) *reinterpret_cast<float4 *>(op + i) = make_float4(v[i], v[i + 1], v[i + 2], v[i + 3]);
    } else {
      __nv_bfloat16 *op = reinterpret_cast<__nv_bfloat16 *>(p.out) + pix * p.out_pitch + c0;
      uint4 o0, o1;
      uint32_t *w0 = reinterpret_cast<uint32_t *>(&o0), *w1 = reinterpret_cast<uint32_t *>(&o1);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        __nv_bfloat162 a = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
        __nv_bfloat162 b = __floats2bfloat162_rn(v[8 + 2 * i], v[8 + 2 * i + 1]);
        w0[i] = *reinterpret_cast<uint32_t *>(&a);
        w1[i] = *reinterpret_cast<uint32_t *>(&b);
      }
      *reinterpret_cast<uint4 *>(op) = o0;
      *reinterpret_cast<uint4 *>(op + 8) = o1;
    }
  } else {  // ragged tail (Cout not a multiple of 16): predicated scalar stores, static indices
#pragma unroll
    for (int i = 0; i < 16; ++i) {
      if (i < nvalid) {
        float x = v[i];
        if (p.res) x += __bfloat162float(p.res[pix * p.res_pitch + c0 + i]);
        if (p.out_f32) reinterpret_cast<float *>(p.out)[pix * p.out_pitch + c0 + i] = x;
        else reinterpret_cast<__nv_bfloat16 *>(p.out)[pix * p.out_pitch + c0 + i] = __float2bfloat16_rn(x);
      }
    }
  }
}

// Same arithmetic, but the 16 results go to this thread's row of the per-warp staging tile in
// shared memory; the warp then copies whole rows out with 16-byte lanes laid along the row, so
// one store instruction touches 32*16/row_bytes rows instead of 32 different 128-byte lines.
__device__ __forceinline__ void epilogue_chunk_staged(const uint32_t (&raw)[16], const float *bias_s, int c0, long long pix,
                                                      const TcParams &p, unsigned char *srow, long long ppix) {
  float v[16];
#pragma unroll
  for (int i = 0; i < 4; ++i) {  // 16-byte broadcast loads of the bias vector
    const float4 q = reinterpret_cast<const float4 *>(bias_s + c0)[i];
    v[4 * i] = q.x; v[4 * i + 1] = q.y; v[4 * i + 2] = q.z; v[4 * i + 3] = q.w;
  }
  if (ppix >= 0) {  // partial sums of the low-resolution half of an upsample + concat + 1x1 conv (staged rows: cout % 16 == 0)
    const float4 *pp = reinterpret_cast<const float4 *>(p.pre + ppix * p.cout + c0);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 q = pp[i];
      v[4 * i] += q.x; v[4 * i + 1] += q.y; v[4 * i + 2] += q.z; v[4 * i + 3] += q.w;
    }
  }
  if (p.relu && !p.res && !p.out_f32) {  // the common case (Conv + BN + ReLU -> bf16): ReLU rides on the conversion
    uint4 o0, o1;
    uint32_t *w0 = reinterpret_cast<uint32_t *>(&o0), *w1 = reinterpret_cast<uint32_t *>(&o1);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      w0[i] = relu_pack_bf16x2(__uint_as_float(raw[2 * i]) + v[2 * i], __uint_as_float(raw[2 * i + 1]) + v[2 * i + 1]);
      w1[i] = relu_pack_bf16x2(__uint_as_float(raw[8 + 2 * i]) + v[8 + 2 * i], __uint_as_float(raw[8 + 2 * i + 1]) + v[8 + 2 * i + 1]);
    }
    uint4 *sp = reinterpret_cast<uint4 *>(srow + c0 * 2);
    sp[0] = o0;
    sp[1] = o1;
    return;
  }
#pragma unroll
  for (int i = 0; i < 16; ++i) {
    const float x = __uint_as_float(raw[i]) + v[i];
    v[i] = p.relu ? fmaxf(x, 0.f) : x;
  }
  if (p.res && pix >= 0) {  // residual convs have Cout % 16 == 0 (checked on the host)
    const __nv_bfloat16 *rp = p.res + pix * p.res_pitch + c0;
    const uint4 r0 = *reinterpret_cast<const uint4 *>(rp), r1 = *reinterpret_cast<const uint4 *>(rp + 8);
    const __nv_bfloat162 *h0 = reinterpret_cast<const __nv_bfloat162 *>(&r0);
    const __nv_bfloat162 *h1 = reinterpret_cast<const __nv_bfloat162 *>(&r1);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float2 f0 = __bfloat1622float2(h0[i]), f1 = __bfloat1622float2(h1[i]);
      v[2 * i] += f0.x; v[2 * i + 1] += f0.y; v[8 + 2 * i] += f1.x; v[8 + 2 * i + 1] += f1.y;
    }
  }
  if (p.out_f32) {
    float4 *sp = reinterpret_cast<float4 *>(srow + c0 * 4);
#pragma unroll
    for (int i = 0; i < 4; ++i) sp[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
  } else {
    uint4 o0, o1;
    uint32_t *w0 = reinterpret_cast<uint32_t *>(&o0), *w1 = reinterpret_cast<uint32_t *>(&o1);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 a = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
      __nv_bfloat162 b = __floats2bfloat162_rn(v[8 + 2 * i], v[8 + 2 * i + 1]);
      w0[i] = *reinterpret_cast<uint32_t *>(&a);
      w1[i] = *reinterpret_cast<uint32_t *>(&b);
    }
    uint4 *sp = reinterpret_cast<uint4 *>(srow + c0 * 2);
    sp[0] = o0;
    sp[1] = o1;
  }
}

// INT8 path: y = float(acc) * m_c + b_c with separate round-to-nearest multiply and add (the
// oracle's integer reference, oracle/quant.py), ReLU, then bf16 / fp32 / re-quantised int8, written at byte c0 * esize of
// `srow`: this thread's row of the staging tile (conv_tc_kernel) or its output pixel's row in global memory
// (conv_tc_big_kernel, whose rows are 16-byte aligned: checked on the host).
__device__ __forceinline__ void epilogue_chunk_i8(const uint32_t (&raw)[16], const float *bias_s, const float *mult_s,
                                                  int c0, long long pix, const TcParams &p, unsigned char *srow, long long ppix) {
  float v[16], mv[16], bv[16];
#pragma unroll
  for (int i = 0; i < 4; ++i) {  // 16-byte broadcast loads of the multiplier / bias vectors
    const float4 m4 = reinterpret_cast<const float4 *>(mult_s + c0)[i], b4 = reinterpret_cast<const float4 *>(bias_s + c0)[i];
    mv[4 * i] = m4.x; mv[4 * i + 1] = m4.y; mv[4 * i + 2] = m4.z; mv[4 * i + 3] = m4.w;
    bv[4 * i] = b4.x; bv[4 * i + 1] = b4.y; bv[4 * i + 2] = b4.z; bv[4 * i + 3] = b4.w;
  }
  if (ppix >= 0) {  // integer partial sums of the low-resolution half (fp32 holds them exactly): acc = acc_skip + up(acc_low)
    const float4 *pp = reinterpret_cast<const float4 *>(p.pre + ppix * p.cout + c0);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const float4 q = pp[i];
      v[4 * i] = q.x; v[4 * i + 1] = q.y; v[4 * i + 2] = q.z; v[4 * i + 3] = q.w;
    }
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __fadd_rn(__fmul_rn(__fadd_rn(__int2float_rn((int)raw[i]), v[i]), mv[i]), bv[i]);
  } else {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __fadd_rn(__fmul_rn(__int2float_rn((int)raw[i]), mv[i]), bv[i]);
  }
  if (p.relu && !p.res && p.out_kind == 0) {  // the common case: ReLU rides on the bf16 conversion
    uint4 o0, o1;
    uint32_t *w0 = reinterpret_cast<uint32_t *>(&o0), *w1 = reinterpret_cast<uint32_t *>(&o1);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      w0[i] = relu_pack_bf16x2(v[2 * i], v[2 * i + 1]);
      w1[i] = relu_pack_bf16x2(v[8 + 2 * i], v[8 + 2 * i + 1]);
    }
    uint4 *sp = reinterpret_cast<uint4 *>(srow + c0 * 2);
    sp[0] = o0;
    sp[1] = o1;
    return;
  }
  if (p.relu && !p.res && p.out_kind == 3) {
    // the consumer's int8 input straight from the accumulator: ReLU + bf16 rounding on one cvt per pair (the activation
    // the graph defines), times the consumer's scale, F2I.S8 (round to nearest even, saturating: the values are >= 0,
    // so [0, 127] is the narrow range), four results packed with three PRMT
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const uint32_t p01 = relu_pack_bf16x2(v[4 * i], v[4 * i + 1]), p23 = relu_pack_bf16x2(v[4 * i + 2], v[4 * i + 3]);
      int q[4];
      const float f[4] = {__uint_as_float(p01 << 16), __uint_as_float(p01 & 0xffff0000u), __uint_as_float(p23 << 16),
                          __uint_as_float(p23 & 0xffff0000u)};
#pragma unroll
      for (int j = 0; j < 4; ++j) asm("cvt.rni.sat.s8.f32 %0, %1;" : "=r"(q[j]) : "f"(__fmul_rn(f[j], p.out_scale)));
      w[i] = __byte_perm(__byte_perm(q[0], q[1], 0x0040), __byte_perm(q[2], q[3], 0x0040), 0x5410);
    }
    *reinterpret_cast<uint4 *>(srow + c0) = make_uint4(w[0], w[1], w[2], w[3]);
    return;
  }
  if (p.relu) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], 0.f);
  }
  if (p.res && pix >= 0) {  // residual (bf16) added in fp32 after the activation
    const __nv_bfloat16 *rp = p.res + pix * p.res_pitch + c0;
    if (p.cout - c0 >= 16 && ((p.res_pitch | (int)(reinterpret_cast<uintptr_t>(p.res) >> 1)) & 7) == 0) {
      const uint4 r0 = *reinterpret_cast<const uint4 *>(rp), r1 = *reinterpret_cast<const uint4 *>(rp + 8);
      const __nv_bfloat162 *h0 = reinterpret_cast<const __nv_bfloat162 *>(&r0);
      const __nv_bfloat162 *h1 = reinterpret_cast<const __nv_bfloat162 *>(&r1);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 f0 = __bfloat1622float2(h0[i]), f1 = __bfloat1622float2(h1[i]);
        v[2 * i] = __fadd_rn(v[2 * i], f0.x); v[2 * i + 1] = __fadd_rn(v[2 * i + 1], f0.y);
        v[8 + 2 * i] = __fadd_rn(v[8 + 2 * i], f1.x); v[8 + 2 * i + 1] = __fadd_rn(v[8 + 2 * i + 1], f1.y);
      }
    } else {  // narrow or unaligned slices (Cout = 8 bottlenecks): guarded scalar loads
#pragma unroll
      for (int i = 0; i < 16; ++i)
        if (c0 + i < p.cout) v[i] = __fadd_rn(v[i], __bfloat162float(rp[i]));
    }
  }
  if (p.out_kind >= 2) {
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      uint32_t pk = 0;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float yv = p.out_kind == 3 ? __bfloat162float(__float2bfloat16_rn(v[4 * i + j])) : v[4 * i + j];
        int q = __float2int_rn(__fmul_rn(yv, p.out_scale));
        q = max(-127, min(127, q));
        pk |= (uint32_t)(q & 0xFF) << (8 * j);
      }
      w[i] = pk;
    }
    *reinterpret_cast<uint4 *>(srow + c0) = make_uint4(w[0], w[1], w[2], w[3]);
  } else if (p.out_kind == 1) {
    float4 *sp = reinterpret_cast<float4 *>(srow + c0 * 4);
#pragma unroll
    for (int i = 0; i < 4; ++i) sp[i] = make_float4(v[4 * i], v[4 * i + 1], v[4 * i + 2], v[4 * i + 3]);
  } else {
    uint4 o0, o1;
    uint32_t *w0 = reinterpret_cast<uint32_t *>(&o0), *w1 = reinterpret_cast<uint32_t *>(&o1);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      __nv_bfloat162 a = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
      __nv_bfloat162 b = __floats2bfloat162_rn(v[8 + 2 * i], v[8 + 2 * i + 1]);
      w0[i] = *reinterpret_cast<uint32_t *>(&a);
      w1[i] = *reinterpret_cast<uint32_t *>(&b);
    }
    uint4 *sp = reinterpret_cast<uint4 *>(srow + c0 * 2);
    sp[0] = o0;
    sp[1] = o1;
  }
}

template <bool I8, int KSTEPS>  // KSTEPS = 32-byte k-steps per channel block (cb_bytes / 32)
__global__ void __launch_bounds__(kThreads, 1) conv_tc_kernel(const __grid_constant__ CUtensorMap tm_in,
                                                              const __grid_constant__ CUtensorMap tm_w, const TcParams p) {
  extern __shared__ unsigned char smem_dyn[];
  const uint32_t raw = smem_u32(smem_dyn);
  const uint32_t base = (raw + 1023u) & ~1023u;  // swizzle atoms need 1024-byte alignment
  const uint32_t w_s = base;
  const uint32_t a_s = base + ((p.w_bytes + 1023u) & ~1023u);
  const uint32_t bar0 = a_s + (uint32_t)p.stages * p.blk_bytes;
  // barrier map: full[stages] | empty[stages] | wfull | tfull[4] | tempty[4] | tmem slot | bias[N]
  const uint32_t full0 = bar0, empty0 = bar0 + 8u * p.stages;
  const uint32_t wfull = empty0 + 8u * p.stages;
  const uint32_t tfull0 = wfull + 8, tempty0 = tfull0 + 8u * kMaxAcc, slot = tempty0 + 8u * kMaxAcc;
  uint32_t *slot_ptr = reinterpret_cast<uint32_t *>(smem_dyn + (slot - raw));
  float *bias_s = reinterpret_cast<float *>(smem_dyn + (bar0 + 512u - raw));
  float *mult_s = reinterpret_cast<float *>(smem_dyn + (bar0 + 1024u - raw));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nacc = p.nacc;
  uint32_t tmem_cols = 32;
  while (tmem_cols < (uint32_t)nacc * p.N) tmem_cols <<= 1;

  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) {
      mbar_init(full0 + 8u * s, 1);
      mbar_init(empty0 + 8u * s, 1);
    }
    mbar_init(wfull, 1);
    for (int a = 0; a < nacc; ++a) {
      mbar_init(tfull0 + 8u * a, 1);
      mbar_init(tempty0 + 8u * a, 128);
    }
    fence_barrier_init();
    // the weights do not depend on the previous kernel: their TMA is part of the prologue that overlaps its tail
    mbar_expect_tx(wfull, p.w_bytes);
    const int nblk = p.ncb * p.taps;
    for (int i = 0; i < nblk; ++i) tma_load_2d(w_s + (uint32_t)i * p.N * p.cb_bytes, &tm_w, wfull, 0, i * p.N);
  }
  griddep_trigger();
  for (int i = threadIdx.x; i < p.N; i += kThreads) {
    bias_s[i] = i < p.cout ? p.bias[i] : 0.f;
    mult_s[i] = (I8 && i < p.cout) ? p.mult[i] : 0.f;
  }
  if (warp == 1) tmem_alloc(slot, tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *slot_ptr;
  griddep_wait();  // from here on the activations written by the previous kernel are read

  const int blocks_per_tile = p.mode == TC_PERTAP ? p.ncb * p.taps : p.ncb;  // HALO / PAIRS: all taps from one block
  const int cb_elems = I8 ? p.cb_bytes : p.cb_bytes / 2;
  const int stages = p.stages;
  const uint32_t blk_bytes = p.blk_bytes, cb_bytes = p.cb_bytes;

  if (warp == 0) {
    // ================= TMA producer =================
    int stage = 0;
    uint32_t phase = 0;
    for (long long tile = blockIdx.x; tile < p.total_tiles; tile += gridDim.x) {
      int n = 0, x0 = 0, y0 = 0;
      if (p.mode != TC_FLAT) {
        const unsigned ut = (unsigned)tile, img = fastdiv(ut, p.tpi, p.m_tpi), t = ut - img * p.tpi;
        const unsigned ty = fastdiv(t, (unsigned)p.tiles_x, p.m_tx);
        n = p.n0 + (int)img;
        y0 = (int)ty * kTileH;
        x0 = (int)(t - ty * (unsigned)p.tiles_x) * kTileW;
      }
      for (int j = 0; j < blocks_per_tile; ++j) {
        mbar_wait(empty0 + 8u * stage, phase ^ 1u);
        const uint32_t dst = a_s + (uint32_t)stage * blk_bytes;
        const uint32_t fb = full0 + 8u * stage;
        if (lane == 0) mbar_expect_tx(fb, p.tx_bytes);
        __syncwarp();
        if (p.mode == TC_FLAT) {
          if (lane == 0) {
            const long long row0 = ((long long)p.n0 * p.H * p.W) + tile * 128;
            tma_load_2d(dst, &tm_in, fb, j * cb_elems, (int)row0);
          }
        } else if (p.mode == TC_HALO) {
          if (p.halo_pitch == kTileW + 2) {  // one dense [18][10][CB] box: the 8-row groups are not 1024-byte
            if (lane == 0)                   // aligned, which is fine because the swizzle is a function of the address
              tma_load_4d(dst, &tm_in, fb, j * cb_elems, x0 - 1, y0 - 1, n);
          } else if (lane < kHaloRows) {
            tma_load_4d(dst + (uint32_t)lane * p.halo_pitch * cb_bytes, &tm_in, fb, j * cb_elems, x0 - 1, y0 - 1 + lane, n);
          }
        } else if (p.mode == TC_PAIRS) {
          if (lane == 0) tma_load_4d(dst, &tm_in, fb, 0, x0 - 1, 2 * y0 - 1, n);
        } else {
          if (lane == 0) {
            const int cb = j / p.taps, tap = j % p.taps;
            const int r = tap / 3, s = tap % 3;
            tma_load_4d(dst, &tm_in, fb, cb * cb_elems, x0 * p.stride + s - 1, y0 * p.stride + r - 1, n);
          }
        }
        if (++stage == stages) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1 || warp == kIssuer2) {
    // ================= MMA issuers: warp 1 takes the even tiles of this CTA's sequence, warp kIssuer2 the odd ones =================
    mbar_wait(wfull, 0);
    const int me = warp == 1 ? 0 : 1;
    int stage = 0;
    uint32_t phase = 0;
    // the other issuer's tile occupies the next blocks_per_tile slots of the ring
    auto skip_tile = [&]() {
      stage += blocks_per_tile;
      while (stage >= stages) { stage -= stages; phase ^= 1u; }
    };
    const int step = p.dual ? 2 : 1;
    if (me) skip_tile();
    const int nacc_mask = nacc - 1, nacc_shift = nacc == 4 ? 2 : 1;
    int it = me;
    const bool pairs = p.mode == TC_PAIRS;
    const uint64_t adesc0 = make_desc_base(p.sbo_a, pairs ? 2u : p.layout_type);  // PAIRS: 128-byte A rows, SWIZZLE_128B
    const uint64_t bdesc0 = make_desc_base(8u * cb_bytes, p.layout_type);
    const uint32_t wblk_bytes = (uint32_t)p.N * cb_bytes;
    const uint32_t idesc = p.idesc;
    const bool halo = p.mode == TC_HALO;
    const uint32_t px_units = cb_bytes >> 4, row_units = (uint32_t)p.halo_pitch * px_units, wblk_units = wblk_bytes >> 4;
    for (long long tile = (me && !p.dual) ? p.total_tiles : blockIdx.x + (long long)me * gridDim.x; tile < p.total_tiles;
         tile += (long long)step * gridDim.x, it += step) {
      const int acc = it & nacc_mask;
      const uint32_t acc_phase = (uint32_t)(it >> nacc_shift) & 1u;
      mbar_wait(tempty0 + 8u * acc, acc_phase ^ 1u);
      tc_fence_after();
      const uint32_t d_tmem = tmem_base + (uint32_t)acc * p.N;
      for (int j = 0; j < blocks_per_tile; ++j) {
        mbar_wait(full0 + 8u * stage, phase);
        tc_fence_after();
        if (elect_one()) {
          // The issue loop runs in ONE thread (elect.sync on the converged warp, see tc_ptx.cuh): every instruction here sits on the critical path of the
          // tensor pipe, so descriptors are advanced by precomputed 16-byte-unit increments and both
          // loops are fully unrolled (KSTEPS is a template parameter).
          const uint64_t ablk_d = adesc0 + (uint64_t)(((a_s + (uint32_t)stage * blk_bytes) & 0x3FFFFu) >> 4);
          uint64_t wd = bdesc0 + (uint64_t)(((w_s + (uint32_t)((halo || pairs) ? j * 9 : j) * wblk_bytes) & 0x3FFFFu) >> 4);
          uint32_t accum = j != 0;
          if (pairs) {
#pragma unroll
            for (int t = 0; t < 9; ++t) {
              // box row t / 3 (+ 2 per output row through SBO); kx = 0: odd pixel of pair 0, 1: even pixel of pair 1, 2: its odd pixel
              const uint64_t ad = ablk_d + (uint64_t)(((t / 3) * kPairCols * 128 + 64 + (t % 3) * 64) >> 4);
#pragma unroll
              for (int k = 0; k < KSTEPS; ++k) {
                umma_bf16(d_tmem, ad + 2 * k, wd + 2 * k, idesc, accum);
                accum = 1;
              }
              wd += wblk_units;
            }
          } else if (halo) {
#pragma unroll
            for (int t = 0; t < 9; ++t) {
              const uint64_t ad = ablk_d + (uint64_t)((t / 3) * row_units + (t % 3) * px_units);
#pragma unroll
              for (int k = 0; k < KSTEPS; ++k) {
                if (I8) umma_i8(d_tmem, ad + 2 * k, wd + 2 * k, idesc, accum);
                else umma_bf16(d_tmem, ad + 2 * k, wd + 2 * k, idesc, accum);
                accum = 1;
              }
              wd += wblk_units;
            }
          } else {
#pragma unroll
            for (int k = 0; k < KSTEPS; ++k) {
              if (I8) umma_i8(d_tmem, ablk_d + 2 * k, wd + 2 * k, idesc, accum);
              else umma_bf16(d_tmem, ablk_d + 2 * k, wd + 2 * k, idesc, accum);
              accum = 1;
            }
          }
          umma_commit(empty0 + 8u * stage);  // smem slot is free once these MMAs retire
          if (j == blocks_per_tile - 1) umma_commit(tfull0 + 8u * acc);
        }
        __syncwarp();
        if (++stage == stages) { stage = 0; phase ^= 1u; }
      }
      if (p.dual) skip_tile();
    }
  } else {
    // ================= epilogue =================
    const int q = warp & 3;  // TMEM lane quarter this warp may touch
    const int m = q * 32 + lane;
    const int nchunks = p.N >> 4;
    const bool staged = p.stage_pitch != 0;
    const int esize = I8 ? (p.out_kind >= 2 ? 1 : (p.out_kind == 1 ? 4 : 2)) : (p.out_f32 ? 4 : 2);
    const int lpr = staged ? (p.cout * esize) / 16 : 1;  // 16-byte lanes per output row
    const int lpr_shift = 31 - __clz(lpr);  // lpr is a power of two (host check)
    const int rows_per_it = 32 >> lpr_shift, sub = lane >> lpr_shift, chunk = lane & (lpr - 1);
    const long long out_row_pitch = (long long)p.out_pitch * esize;
    unsigned char *gout_lane = reinterpret_cast<unsigned char *>(p.out) + (long long)sub * out_row_pitch + chunk * 16;
    const long long gstep = (long long)rows_per_it * out_row_pitch;
    const int sstep = rows_per_it * p.stage_pitch;
    long long *spix = reinterpret_cast<long long *>(smem_dyn + (bar0 + 1536u - raw)) + (warp - 2) * 32;
    unsigned char *swarp = smem_dyn + (bar0 + kTailFixed - raw) + (size_t)(warp - 2) * 32 * p.stage_pitch;
    const int group = (warp - 2) >> 2;  // the epilogue warpgroups take tiles round-robin
    unsigned char *srow = swarp + (size_t)lane * p.stage_pitch;
    // Group g takes tiles g, g + ngroups, ... of this CTA's sequence (groups >= ngroups idle).  ngroups and nacc are
    // powers of two (nacc a multiple of ngroups: an accumulator always belongs to the same group) and every tile /
    // pixel index of a launch fits 32 bits (checked on the host): no runtime division on the per-tile path except
    // the one 32-bit tile -> (image, tile row, tile column) split.
    const int nacc_mask = nacc - 1, nacc_shift = nacc == 4 ? 2 : 1;
    const unsigned hw = (unsigned)p.H * (unsigned)p.W;
    int it = group;
    for (long long tile = blockIdx.x + (long long)group * gridDim.x; group < p.ngroups && tile < p.total_tiles;
         tile += (long long)p.ngroups * gridDim.x, it += p.ngroups) {
      const int acc = it & nacc_mask;
      const uint32_t acc_phase = (uint32_t)(it >> nacc_shift) & 1u;
      long long pix;        // flattened output pixel (n, oy, ox) or -1
      long long ppix = -1;  // pixel of the half-resolution partial-sum tensor this output pixel adds, or -1
      if (p.mode == TC_FLAT) {
        const unsigned row = (unsigned)tile * 128u + (unsigned)m;
        pix = row < (unsigned)p.nb * hw ? (long long)((unsigned)p.n0 * hw + row) : -1;
        if (p.pre && pix >= 0) {
          const unsigned upix = (unsigned)pix, t = upix / (unsigned)p.W, ox = upix - t * (unsigned)p.W;
          const unsigned img = t / (unsigned)p.H, oy = t - img * (unsigned)p.H;
          ppix = (long long)((img * (unsigned)(p.H >> 1) + (oy >> 1)) * (unsigned)(p.W >> 1) + (ox >> 1));
        }
      } else {
        const unsigned ut = (unsigned)tile, img = fastdiv(ut, p.tpi, p.m_tpi), t = ut - img * p.tpi;
        const unsigned ty = fastdiv(t, (unsigned)p.tiles_x, p.m_tx), tx = t - ty * (unsigned)p.tiles_x;
        const int n = p.n0 + (int)img;
        const int oy = (int)ty * kTileH + (m >> 3), ox = (int)tx * kTileW + (m & 7);
        pix = (oy < p.H && ox < p.W) ? ((long long)n * p.H + oy) * p.W + ox : -1;
        if (p.pre && pix >= 0) ppix = ((long long)n * (p.H >> 1) + (oy >> 1)) * (p.W >> 1) + (ox >> 1);
      }
      mbar_wait(tfull0 + 8u * acc, acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)acc * p.N;
      uint32_t cur[16], nxt[16];
      tmem_ld16_issue(taddr, cur);
      tmem_ld_wait();
      if (staged) spix[lane] = pix;
      for (int c = 0; c < nchunks; ++c) {
        const bool more = c + 1 < nchunks;
        if (more) {
          tmem_ld16_issue(taddr + 16u * (c + 1), nxt);  // in flight while this chunk is processed
        } else {
          tc_fence_before();
          mbar_arrive(tempty0 + 8u * acc);  // every TMEM read of this accumulator has completed
        }
        if (staged) {
          if (c * 16 < p.cout) {
            if (I8) epilogue_chunk_i8(cur, bias_s, mult_s, c * 16, pix, p, srow, ppix);
            else epilogue_chunk_staged(cur, bias_s, c * 16, pix, p, srow, ppix);
          }
        } else if (pix >= 0 && c * 16 < p.cout) {
          epilogue_chunk(cur, bias_s, c * 16, pix, p, ppix);
        }
        if (more) {
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i) cur[i] = nxt[i];
        }
      }
      if (staged) {  // coalesced copy-out of this warp's 32 rows: 16-byte lanes laid along the rows
        __syncwarp();
        const unsigned char *sp = swarp + sub * p.stage_pitch + chunk * 16;
        if (p.mode == TC_FLAT) {  // the rows of a tile are consecutive pixels: no row -> pixel map
          const unsigned row0 = (unsigned)tile * 128u + (unsigned)(q * 32), nrows = (unsigned)p.nb * hw;
          unsigned char *gp = gout_lane + (long long)((unsigned)p.n0 * hw + row0) * out_row_pitch;
          for (int r = sub; r < 32; r += rows_per_it, gp += gstep, sp += sstep)
            if (row0 + (unsigned)r < nrows) *reinterpret_cast<uint4 *>(gp) = *reinterpret_cast<const uint4 *>(sp);
        } else {
          for (int r = sub; r < 32; r += rows_per_it, sp += sstep) {
            const long long pr = spix[r];
            if (pr >= 0) *reinterpret_cast<uint4 *>(gout_lane + pr * out_row_pitch - (long long)sub * out_row_pitch) = *reinterpret_cast<const uint4 *>(sp);
          }
        }
        __syncwarp();
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, tmem_cols);
}


// =================================================================================================
// BIG variant: convolutions whose weights do not fit shared memory (Cin * k * k * Cout * 2 B > 150 KB: the
// 128 / 256 / 512-channel layers of the model.py network, model.py:274-303,308-365).
//   * a CTA owns a PAIR of M-tiles (a 16 x 16 pixel region, or 256 consecutive pixels of a 1x1 conv) with
//     two TMEM accumulators of N <= 256 columns: every weight block that crosses L2 -> SMEM feeds 2 x 128 rows;
//   * weights stream through their own TMA pipeline, one (channel block, tap) block of N x 128 bytes per stage;
//   * activations: HALO (3x3 s1: one [18][18][128 B] box per channel block, nine tap-shifted descriptors per tile),
//     PERTAP (3x3 s2: one strided [16][16][128 B] box per block and tap) or FLAT (1x1: [256][128 B]).
// A 128-byte row is 64 bf16 channels (kind::f16, K = 16 per MMA) or, with I8, 128 int8 channels (kind::i8, K = 32,
// S32 accumulators, the requant epilogue of the resident int8 kernel): the byte geometry is the same.
// Warps: 0 = activation TMA, 1 = TMEM allocator + MMA issuer, 2 = weight TMA, 4..11 = two epilogue groups
// (group g drains M-tile g).  When 4 N <= 512 the accumulator pairs are double-buffered.
// =================================================================================================
constexpr int kBigThreads = 128 + 256;
constexpr int kBigHalo = 18;

template <bool I8>
__global__ void __launch_bounds__(kBigThreads, 1) conv_tc_big_kernel(const __grid_constant__ CUtensorMap tm_in,
                                                                     const __grid_constant__ CUtensorMap tm_w, const TcParams p) {
  extern __shared__ unsigned char smem_dyn[];
  const uint32_t raw = smem_u32(smem_dyn);
  const uint32_t base = (raw + 1023u) & ~1023u;
  const uint32_t a_s = base;
  const uint32_t w_s = a_s + (uint32_t)p.stages * p.blk_bytes;
  const uint32_t bar0 = w_s + (uint32_t)p.wstages * p.wblk_bytes;
  // barrier map: afull[4] aempty[4] wfull[8] wempty[8] tfull[2] tempty[2] | slot | bias[256] | mult[256] (I8)
  const uint32_t afull = bar0, aempty = bar0 + 32, wfull = bar0 + 64, wempty = bar0 + 128, tfull = bar0 + 192, tempty = bar0 + 208;
  const uint32_t slot = bar0 + 224;
  uint32_t *slot_ptr = reinterpret_cast<uint32_t *>(smem_dyn + (slot - raw));
  float *bias_s = reinterpret_cast<float *>(smem_dyn + (bar0 + 256u - raw));
  float *mult_s = reinterpret_cast<float *>(smem_dyn + (bar0 + 1280u - raw));

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nacc = p.nacc;  // accumulator PAIRS
  const uint32_t tmem_cols = 512;
  if (threadIdx.x == 0) {
    for (int s = 0; s < p.stages; ++s) { mbar_init(afull + 8u * s, 1); mbar_init(aempty + 8u * s, 1); }
    for (int s = 0; s < p.wstages; ++s) { mbar_init(wfull + 8u * s, 1); mbar_init(wempty + 8u * s, 1); }
    for (int a = 0; a < nacc; ++a) { mbar_init(tfull + 8u * a, 1); mbar_init(tempty + 8u * a, 256); }
    fence_barrier_init();
  }
  griddep_trigger();
  for (int i = threadIdx.x; i < 256; i += kBigThreads) bias_s[i] = i < p.cout ? p.bias[i] : 0.f;
  if (I8)
    for (int i = threadIdx.x; i < 256; i += kBigThreads) mult_s[i] = i < p.cout ? p.mult[i] : 0.f;
  if (warp == 1) tmem_alloc(slot, tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *slot_ptr;
  griddep_wait();

  const int kblocks = p.ncb * p.taps;                                   // weight blocks per pair
  const bool a_per_tap = p.mode == TC_PERTAP;                           // else one A block per channel block
  const long long total = p.total_tiles;                                // pairs of this launch
  constexpr int cb_elems = I8 ? 128 : 64;                               // channels per 128-byte row

  if (warp == 0) {
    // ================= activation TMA =================
    int stage = 0;
    uint32_t phase = 0;
    for (long long pair = blockIdx.x; pair < total; pair += gridDim.x) {
      int n = 0, x0 = 0, y0 = 0;
      if (p.mode != TC_FLAT) {
        const unsigned up = (unsigned)pair, img = fastdiv(up, p.tpi, p.m_tpi), t = up - img * p.tpi;
        const unsigned ty = fastdiv(t, (unsigned)p.pairs_x, p.m_tx);
        n = p.n0 + (int)img;
        y0 = (int)ty * 16;
        x0 = (int)(t - ty * (unsigned)p.pairs_x) * 16;
      }
      const int nblk = a_per_tap ? kblocks : p.ncb;
      for (int j = 0; j < nblk; ++j) {
        mbar_wait(aempty + 8u * stage, phase ^ 1u);
        if (lane == 0) {
          const uint32_t dst = a_s + (uint32_t)stage * p.blk_bytes, fb = afull + 8u * stage;
          mbar_expect_tx(fb, p.tx_bytes);
          if (p.mode == TC_FLAT) {
            tma_load_2d(dst, &tm_in, fb, j * cb_elems, (int)((long long)p.n0 * p.H * p.W + pair * 256));
          } else if (p.mode == TC_HALO) {
            tma_load_4d(dst, &tm_in, fb, j * cb_elems, x0 - 1, y0 - 1, n);
          } else {
            const int cb = j / 9, tap = j % 9;
            tma_load_4d(dst, &tm_in, fb, cb * cb_elems, x0 * p.stride + tap % 3 - 1, y0 * p.stride + tap / 3 - 1, n);
          }
        }
        __syncwarp();
        if (++stage == p.stages) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 2) {
    // ================= weight TMA =================
    int stage = 0;
    uint32_t phase = 0;
    for (long long pair = blockIdx.x; pair < total; pair += gridDim.x) {
      for (int j = 0; j < kblocks; ++j) {
        mbar_wait(wempty + 8u * stage, phase ^ 1u);
        if (lane == 0) {
          const uint32_t fb = wfull + 8u * stage;
          mbar_expect_tx(fb, (uint32_t)p.N * 128u);
          tma_load_2d(w_s + (uint32_t)stage * p.wblk_bytes, &tm_w, fb, 0, j * p.N);
        }
        __syncwarp();
        if (++stage == p.wstages) { stage = 0; phase ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // ================= MMA issuer =================
    int astage = 0, wstage = 0, acc = 0;
    uint32_t aphase = 0, wphase = 0, acc_phase = 0;
    const uint64_t adesc0 = make_desc_base(p.sbo_a, 2u);   // 128-byte rows, SWIZZLE_128B
    const uint64_t bdesc0 = make_desc_base(1024u, 2u);
    const bool halo = p.mode == TC_HALO;
    const uint32_t tile_units = p.tile_off >> 4;
    for (long long pair = blockIdx.x; pair < total; pair += gridDim.x) {
      mbar_wait(tempty + 8u * acc, acc_phase ^ 1u);
      tc_fence_after();
      const uint32_t d0 = tmem_base + (uint32_t)acc * 2u * p.N;
      for (int j = 0; j < kblocks; ++j) {
        const int tap = halo ? j % 9 : 0;
        if (!halo || tap == 0) {
          mbar_wait(afull + 8u * astage, aphase);
        }
        mbar_wait(wfull + 8u * wstage, wphase);
        tc_fence_after();
        if (elect_one()) {
          uint64_t ad = adesc0 + (uint64_t)(((a_s + (uint32_t)astage * p.blk_bytes) & 0x3FFFFu) >> 4);
          if (halo) ad += (uint64_t)(((tap / 3) * kBigHalo + (tap % 3)) * 8);   // (r * pitch + s) pixels of 128 bytes
          const uint64_t wd = bdesc0 + (uint64_t)(((w_s + (uint32_t)wstage * p.wblk_bytes) & 0x3FFFFu) >> 4);
          const uint32_t accum = j != 0;
#pragma unroll
          for (int t = 0; t < 2; ++t) {
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              if (I8) umma_i8(d0 + (uint32_t)t * p.N, ad + (uint64_t)t * tile_units + 2 * k, wd + 2 * k, p.idesc, (accum | (uint32_t)k) ? 1u : 0u);
              else umma_bf16(d0 + (uint32_t)t * p.N, ad + (uint64_t)t * tile_units + 2 * k, wd + 2 * k, p.idesc, (accum | (uint32_t)k) ? 1u : 0u);
            }
          }
          umma_commit(wempty + 8u * wstage);
          if (!halo || tap == 8) umma_commit(aempty + 8u * astage);
          if (j == kblocks - 1) umma_commit(tfull + 8u * acc);
        }
        __syncwarp();
        if (++wstage == p.wstages) { wstage = 0; wphase ^= 1u; }
        if (!halo || tap == 8) {
          if (++astage == p.stages) { astage = 0; aphase ^= 1u; }
        }
      }
      if (++acc == nacc) { acc = 0; acc_phase ^= 1u; }
    }
  } else if (warp >= 4) {
    // ================= epilogue: group g drains M-tile g of every pair =================
    const int q = warp & 3, g = (warp - 4) >> 2;
    const int m = q * 32 + lane;
    const int nchunks = p.N >> 4;
    const unsigned hw = (unsigned)p.H * (unsigned)p.W;
    unsigned char *out_row = reinterpret_cast<unsigned char *>(p.out);  // I8: rows of out_pitch * esize bytes
    const long long out_row_pitch = (long long)p.out_pitch * (p.out_kind >= 2 ? 1 : (p.out_kind == 1 ? 4 : 2));
    int it = 0;
    for (long long pair = blockIdx.x; pair < total; pair += gridDim.x, ++it) {
      const int acc = nacc == 2 ? (it & 1) : 0;
      const uint32_t acc_phase = (uint32_t)(nacc == 2 ? (it >> 1) : it) & 1u;
      long long pix;
      if (p.mode == TC_FLAT) {
        const unsigned row = (unsigned)pair * 256u + (unsigned)g * 128u + (unsigned)m;
        pix = row < (unsigned)p.nb * hw ? (long long)((unsigned)p.n0 * hw + row) : -1;
      } else {
        const unsigned up = (unsigned)pair, img = fastdiv(up, p.tpi, p.m_tpi), t = up - img * p.tpi;
        const unsigned ty = fastdiv(t, (unsigned)p.pairs_x, p.m_tx), tx = t - ty * (unsigned)p.pairs_x;
        const int oy = (int)ty * 16 + (m >> 3), ox = (int)tx * 16 + g * 8 + (m & 7);
        pix = (oy < p.H && ox < p.W) ? ((long long)(p.n0 + (int)img) * p.H + oy) * p.W + ox : -1;
      }
      mbar_wait(tfull + 8u * acc, acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)acc * 2u * p.N + (uint32_t)g * p.N;
      uint32_t cur[16], nxt[16];
      tmem_ld16_issue(taddr, cur);
      tmem_ld_wait();
      for (int c = 0; c < nchunks; ++c) {
        const bool more = c + 1 < nchunks;
        if (more) {
          tmem_ld16_issue(taddr + 16u * (c + 1), nxt);
        } else {
          tc_fence_before();
          mbar_arrive(tempty + 8u * acc);
        }
        if (pix >= 0 && c * 16 < p.cout) {
          if (I8) epilogue_chunk_i8(cur, bias_s, mult_s, c * 16, pix, p, out_row + pix * out_row_pitch, -1);
          else epilogue_chunk(cur, bias_s, c * 16, pix, p, -1);
        }
        if (more) {
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i) cur[i] = nxt[i];
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) tmem_dealloc(tmem_base, tmem_cols);
}

}  // namespace

// ---- host side -----------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void *p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<EncodeTiledFn>(p);
  }
  return fn;
}

static CUtensorMapSwizzle swizzle_of(int cb_bytes) {
  return cb_bytes == 128 ? CU_TENSOR_MAP_SWIZZLE_128B : cb_bytes == 64 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B;
}

static int encode(CUtensorMap *tm, void *base, int rank, const cuuint64_t *dims, const cuuint64_t *strides_bytes,
                  const cuuint32_t *box, const cuuint32_t *estr, int cb_bytes, bool u8 = false) {
  EncodeTiledFn fn = get_encode();
  UYD_REQUIRE(fn, UYD_E_NOGPU, "cuTensorMapEncodeTiled is not available (no CUDA driver)");
  CUresult r = fn(tm, u8 ? CU_TENSOR_MAP_DATA_TYPE_UINT8 : CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, base, dims, strides_bytes, box, estr,
                  CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle_of(cb_bytes), CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                  CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  UYD_REQUIRE(r == CUDA_SUCCESS, UYD_E_ARG, "cuTensorMapEncodeTiled failed with CUresult %d (rank %d)", (int)r, rank);
  return UYD_OK;
}

struct TcConv {  // everything a launch needs, prepared once at plan finalize
  CUtensorMap tm_in, tm_w;
  TcParams p;
  size_t smem;
  void *w_dev = nullptr;
};

static int pick_cb(int cin) { return cin % 64 == 0 ? 64 : (cin % 32 == 0 ? 32 : (cin % 16 == 0 ? 16 : 0)); }
// int8: channels (= bytes) per block
static int pick_cb_s8(int cin) { return cin % 128 == 0 ? 128 : (cin % 64 == 0 ? 64 : (cin % 32 == 0 ? 32 : 0)); }

// BIG variant (streamed weights): 64-channel blocks, Cout <= 256 in 16-column chunks, no partial sums
static bool tc_big_supported(const uyd_conv &d) {
  return d.cin % 64 == 0 && d.cout % 16 == 0 && d.cout <= 256 && !d.pre_buf_p1;
}

bool tc_supported(const uyd_conv &d, int in_pitch, int in_coff, int out_pitch, int out_coff, bool in_is_network_input) {
  if (in_is_network_input || d.depthwise) return false;
  if (!(d.k == 1 || d.k == 3) || !(d.stride == 1 || d.stride == 2)) return false;
  if (d.k == 1 && d.stride != 1) return false;
  if (pick_cb(d.cin) == 0 || d.cout < 4) return false;
  if (in_pitch % 8 || in_coff % 8 || out_pitch % 4 || out_coff % 4) return false;
  const int N = (d.cout + 15) / 16 * 16;
  if (d.cout > 128 || (size_t)d.cin * d.k * d.k * N * 2 > 150 * 1024) return tc_big_supported(d);
  return true;
}

size_t tc_weight_bytes(const uyd_conv &d) {
  const int N = (d.cout + 15) / 16 * 16;
  return (size_t)d.cin * d.k * d.k * N * 2;
}

// PyTorch [cout][cin][k][k] fp32 -> bf16 [cb][tap][n (padded to N)][CB]
void tc_pack_weights(const uyd_conv &d, const float *w, void *dst_host) {
  const int CB = pick_cb(d.cin), ncb = d.cin / CB, taps = d.k * d.k, N = (d.cout + 15) / 16 * 16;
  __nv_bfloat16 *o = reinterpret_cast<__nv_bfloat16 *>(dst_host);
  for (int cb = 0; cb < ncb; ++cb)
    for (int t = 0; t < taps; ++t)
      for (int n = 0; n < N; ++n)
        for (int c = 0; c < CB; ++c) {
          const float v = n < d.cout ? w[((size_t)n * d.cin + cb * CB + c) * taps + t] : 0.f;
          o[(((size_t)cb * taps + t) * N + n) * CB + c] = __float2bfloat16_rn(v);
        }
}

// int8 on the resident-weight kernel: Cout <= 128, output rows a power-of-two number of 16-byte lanes (staging tile),
// resident weights + two 128-row stages + one staging group within 227 KB
static bool tc_resident_fits_s8(int cin, int cout, int k, int out_esize) {
  if (pick_cb_s8(cin) == 0 || cout > 128) return false;
  const int rb = cout * out_esize;
  if (rb < 16 || rb > 512 || (rb & (rb - 1))) return false;
  const int N = (cout + 15) / 16 * 16;
  const size_t need = (((size_t)cin * k * k * N + 1023) & ~(size_t)1023) + 2 * (size_t)128 * pick_cb_s8(cin) + kTailFixed +
                      (size_t)128 * 1 * (N * out_esize + 16) + 1024;  // at least one staging group
  return need <= 227 * 1024;
}

// int8 on the streamed-weight kernel, taken only where the resident one cannot run: 128-channel blocks,
// Cout <= 256 in 16-column chunks, direct 16-byte row stores, no partial sums
static bool tc_big_s8(int cin, int cout, int k, int out_esize, bool pre) {
  return !tc_resident_fits_s8(cin, cout, k, out_esize) && cin % 128 == 0 && cout % 16 == 0 && cout <= 256 && !pre;
}

bool tc_supported_s8(int cin, int cout, int k, int stride, int in_pitch, int in_coff, int out_pitch, int out_coff, int out_esize,
                     bool pre) {
  if (!(k == 1 || k == 3) || !(stride == 1 || stride == 2) || (k == 1 && stride != 1)) return false;
  if (pick_cb_s8(cin) == 0 || cout < 4) return false;
  if (in_pitch % 16 || in_coff % 16) return false;
  if ((out_pitch * out_esize) % 16 || (out_coff * out_esize) % 16) return false;
  return tc_resident_fits_s8(cin, cout, k, out_esize) || tc_big_s8(cin, cout, k, out_esize, pre);
}

size_t tc_weight_bytes_s8(int cin, int cout, int k) { return (size_t)cin * k * k * ((cout + 15) / 16 * 16); }

// [cout][cin][k][k] int8 -> int8 [cb][tap][n (padded to N)][CB]
void tc_pack_weights_s8(int cin, int cout, int k, const int8_t *w, void *dst_host) {
  const int CB = pick_cb_s8(cin), ncb = cin / CB, taps = k * k, N = (cout + 15) / 16 * 16;
  int8_t *o = reinterpret_cast<int8_t *>(dst_host);
  for (int cb = 0; cb < ncb; ++cb)
    for (int t = 0; t < taps; ++t)
      for (int n = 0; n < N; ++n)
        for (int c = 0; c < CB; ++c)
          o[(((size_t)cb * taps + t) * N + n) * CB + c] = n < cout ? w[((size_t)n * cin + cb * CB + c) * taps + t] : (int8_t)0;
}


// i8: int8 operands (128 channels per row), requant epilogue with mult_dev / out_scale / out_kind as in tc_prepare
static int tc_prepare_big(TcConv *tc, const uyd_conv &d, void *in_base, int in_pitch, int ih, int iw, int max_batch, void *out_base,
                          int out_pitch, int out_f32, const void *res_base, int res_pitch, void *w_dev, const float *bias_dev,
                          int i8 = 0, const float *mult_dev = nullptr, float out_scale = 0.f, int out_kind = 0) {
  TcParams &p = tc->p;
  const int es = i8 ? 1 : 2, ce = 128 / es;  // bytes per element, channels per 128-byte row
  UYD_REQUIRE(i8 ? (d.cin % 128 == 0 && d.cout % 16 == 0 && d.cout <= 256 && !d.pre_buf_p1) : tc_big_supported(d), UYD_E_UNSUPPORTED,
              "conv_tc big: cin %% %d, cout %% 16, cout <= 256, no partial sums", ce);
  UYD_REQUIRE(!res_base || ((res_pitch % 8) == 0 && (reinterpret_cast<uintptr_t>(res_base) & 15) == 0), UYD_E_UNSUPPORTED,
              "conv_tc big: residual slice must be 16-byte aligned");
  if (i8) {
    const int esize = out_kind >= 2 ? 1 : (out_kind == 1 ? 4 : 2);
    UYD_REQUIRE((out_pitch * esize) % 16 == 0 && (reinterpret_cast<uintptr_t>(out_base) & 15) == 0, UYD_E_UNSUPPORTED,
                "conv_tc big int8: output rows must be 16-byte aligned");
    p.i8 = 1;
    p.mult = mult_dev;
    p.out_scale = out_scale;
    p.out_kind = out_kind;
    out_f32 = out_kind == 1;
  }
  p.big = 1;
  p.cb_bytes = 128;
  p.ncb = d.cin / ce;
  p.taps = d.k * d.k;
  p.stride = d.stride;
  p.N = d.cout;
  p.cout = d.cout;
  p.H = d.k == 1 ? ih : (ih + 2 - 3) / d.stride + 1;
  p.W = d.k == 1 ? iw : (iw + 2 - 3) / d.stride + 1;
  p.mode = d.k == 1 ? TC_FLAT : (d.stride == 1 ? TC_HALO : TC_PERTAP);
  p.layout_type = 2u;
  p.idesc = ((i8 ? 2u : 1u) << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  p.pairs_x = ceil_div(p.W, 16);
  p.tiles_y = ceil_div(p.H, 16);
  p.tiles_x = p.pairs_x;
  if (p.mode == TC_HALO) {
    p.tx_bytes = (uint32_t)kBigHalo * kBigHalo * 128u;
    p.sbo_a = (uint32_t)kBigHalo * 128u;
    p.tile_off = 8u * 128u;
  } else if (p.mode == TC_PERTAP) {
    p.tx_bytes = 256u * 128u;
    p.sbo_a = 16u * 128u;
    p.tile_off = 8u * 128u;
  } else {
    p.tx_bytes = 256u * 128u;
    p.sbo_a = 1024u;
    p.tile_off = 128u * 128u;
  }
  p.blk_bytes = (p.tx_bytes + 1023u) & ~1023u;
  p.wblk_bytes = (uint32_t)p.N * 128u;   // N % 16 == 0 and >= 144: a multiple of 1024 whenever N % 8 == 0
  p.wblk_bytes = (p.wblk_bytes + 1023u) & ~1023u;
  const size_t tail = 256 + 1024 + 1024;  // barriers + bias + mult
  const size_t budget = 227 * 1024 - 1024 - tail;
  int stages = p.mode == TC_HALO ? 2 : 3;
  int wstages = (int)((budget - (size_t)stages * p.blk_bytes) / p.wblk_bytes);
  if (wstages > 8) wstages = 8;
  while (wstages < 3 && stages > 2) { --stages; wstages = (int)((budget - (size_t)stages * p.blk_bytes) / p.wblk_bytes); }
  UYD_REQUIRE(wstages >= 2, UYD_E_UNSUPPORTED, "conv_tc big: no room for two weight stages (N = %d)", p.N);
  // the space left after 3+ weight stages goes to activation stages
  if (wstages > 4) {
    const int extra = (int)((budget - (size_t)stages * p.blk_bytes - (size_t)4 * p.wblk_bytes) / p.blk_bytes);
    if (extra > 0) { stages += extra > 2 ? 2 : extra; wstages = (int)((budget - (size_t)stages * p.blk_bytes) / p.wblk_bytes); if (wstages > 8) wstages = 8; }
  }
  if (stages > 4) stages = 4;
  p.stages = stages;
  p.wstages = wstages;
  p.nacc = 4 * p.N <= 512 ? 2 : 1;
  tc->smem = 1024 + (size_t)stages * p.blk_bytes + (size_t)wstages * p.wblk_bytes + tail;
  p.out = out_base; p.out_pitch = out_pitch; p.out_f32 = out_f32;
  p.res = reinterpret_cast<const __nv_bfloat16 *>(res_base); p.res_pitch = res_pitch;
  p.bias = bias_dev; p.relu = d.relu;
  tc->w_dev = w_dev;
  const cuuint32_t one4[4] = {1, 1, 1, 1};
  {  // weights [rows = ncb * taps * N][128 bytes]: one box = one (channel block, tap) block
    const cuuint64_t dims[2] = {(cuuint64_t)ce, (cuuint64_t)p.ncb * p.taps * p.N};
    const cuuint64_t str[1] = {128};
    const cuuint32_t box[2] = {(cuuint32_t)ce, (cuuint32_t)p.N};
    if (int e = encode(&tc->tm_w, w_dev, 2, dims, str, box, one4, 128, i8)) return e;
  }
  if (p.mode == TC_FLAT) {
    const cuuint64_t dims[2] = {(cuuint64_t)d.cin, (cuuint64_t)max_batch * ih * iw};
    const cuuint64_t str[1] = {(cuuint64_t)in_pitch * es};
    const cuuint32_t box[2] = {(cuuint32_t)ce, 256};
    if (int e = encode(&tc->tm_in, in_base, 2, dims, str, box, one4, 128, i8)) return e;
  } else {
    const cuuint64_t dims[4] = {(cuuint64_t)d.cin, (cuuint64_t)iw, (cuuint64_t)ih, (cuuint64_t)max_batch};
    const cuuint64_t str[3] = {(cuuint64_t)in_pitch * es, (cuuint64_t)iw * in_pitch * es, (cuuint64_t)ih * iw * in_pitch * es};
    if (p.mode == TC_HALO) {
      const cuuint32_t box[4] = {(cuuint32_t)ce, (cuuint32_t)kBigHalo, (cuuint32_t)kBigHalo, 1};
      if (int e = encode(&tc->tm_in, in_base, 4, dims, str, box, one4, 128, i8)) return e;
    } else {
      const cuuint32_t sd = (cuuint32_t)d.stride;
      const cuuint32_t box[4] = {(cuuint32_t)ce, 16 * sd, 16 * sd, 1};
      const cuuint32_t estr[4] = {1, sd, sd, 1};
      if (int e = encode(&tc->tm_in, in_base, 4, dims, str, box, estr, 128, i8)) return e;
    }
  }
  return i8 ? smem_optin(conv_tc_big_kernel<true>, 227 * 1024) : smem_optin(conv_tc_big_kernel<false>, 227 * 1024);
}

// mode_override: -1 auto, else TC_*.  in_base/out_base/res_base: slice bases of image 0.
// i8 != 0: int8 operands (weights already quantised), per-channel multiplier mult_dev,
// out_kind 0/1/2 = bf16 / fp32 / int8 re-quantised with out_scale.
int tc_prepare(TcConv *tc, const uyd_conv &d, void *in_base, int in_pitch, int ih, int iw, int max_batch, void *out_base,
               int out_pitch, int out_f32, const void *res_base, int res_pitch, void *w_dev, const float *bias_dev,
               int mode_override, int base_offset_mode, int stages_override, int i8 = 0, const float *mult_dev = nullptr,
               float out_scale = 0.f, int out_kind = 0, int halo_pitch = 10) {
  TcParams &p = tc->p;
  memset(&p, 0, sizeof(p));
  {
    const int Np = (d.cout + 15) / 16 * 16;
    if (!i8 && (d.cout > 128 || (size_t)d.cin * d.k * d.k * Np * 2 > 150 * 1024))
      return tc_prepare_big(tc, d, in_base, in_pitch, ih, iw, max_batch, out_base, out_pitch, out_f32, res_base, res_pitch, w_dev, bias_dev);
    const int out_esize = out_kind >= 2 ? 1 : (out_kind == 1 ? 4 : 2);
    if (i8 && tc_big_s8(d.cin, d.cout, d.k, out_esize, d.pre_buf_p1 != 0))
      return tc_prepare_big(tc, d, in_base, in_pitch, ih, iw, max_batch, out_base, out_pitch, out_f32, res_base, res_pitch, w_dev, bias_dev,
                            1, mult_dev, out_scale, out_kind);
  }
  const int es = i8 ? 1 : 2;
  const int CB = i8 ? pick_cb_s8(d.cin) : pick_cb(d.cin);
  UYD_REQUIRE(CB, UYD_E_UNSUPPORTED, "conv_tc: cin %d is not a multiple of %d", d.cin, i8 ? 32 : 16);
  p.i8 = i8;
  p.mult = mult_dev;
  p.out_scale = out_scale;
  p.out_kind = out_kind;
  if (i8) out_f32 = out_kind == 1;
  p.cb_bytes = CB * es;
  p.ncb = d.cin / CB;
  p.taps = d.k * d.k;
  p.stride = d.stride;
  p.N = (d.cout + 15) / 16 * 16;
  p.cout = d.cout;
  p.H = d.k == 1 ? ih : (ih + 2 * 1 - 3) / d.stride + 1;
  p.W = d.k == 1 ? iw : (iw + 2 * 1 - 3) / d.stride + 1;
  p.mode = d.k == 1 ? TC_FLAT : (d.stride == 1 ? TC_HALO : TC_PERTAP);
  // PAIRS needs a dense input (pitch == Cin: the two pixels of a pair are 128 contiguous bytes) and an even width
  if (p.mode == TC_PERTAP && d.stride == 2 && !i8 && p.cb_bytes == 64 && p.ncb == 1 && iw % 2 == 0 && in_pitch == d.cin &&
      (reinterpret_cast<uintptr_t>(in_base) & 127) == 0 && mode_override < 0)
    p.mode = TC_PAIRS;
  if (mode_override >= 0 && d.k == 3) p.mode = mode_override;
  UYD_REQUIRE(!(p.mode == TC_HALO && d.stride != 1), UYD_E_UNSUPPORTED, "conv_tc: HALO mode needs stride 1");
  p.base_offset_mode = base_offset_mode;
  p.layout_type = p.cb_bytes == 128 ? 2u : (p.cb_bytes == 64 ? 4u : 6u);
  // c_format F32 (1) / S32 (2); a,b format 1 = BF16 resp. signed int8; K-major; N >> 3; M >> 4
  p.idesc = ((i8 ? 2u : 1u) << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(p.N >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
  p.w_bytes = (uint32_t)((size_t)d.cin * d.k * d.k * p.N * es);
  p.tiles_x = ceil_div(p.W, kTileW);
  p.tiles_y = ceil_div(p.H, kTileH);
  if (p.mode == TC_HALO) {
    p.halo_pitch = halo_pitch == 16 ? 16 : kTileW + 2;
    p.blk_bytes = (uint32_t)kHaloRows * p.halo_pitch * p.cb_bytes;
    p.tx_bytes = (uint32_t)kHaloRows * (kTileW + 2) * p.cb_bytes;
    p.sbo_a = (uint32_t)p.halo_pitch * p.cb_bytes;
  } else if (p.mode == TC_PAIRS) {
    p.halo_pitch = kPairCols;
    p.blk_bytes = (uint32_t)kPairRows * kPairCols * 128u;
    p.tx_bytes = p.blk_bytes;
    p.sbo_a = 2u * kPairCols * 128u;  // consecutive output rows are two box rows apart
  } else {
    p.blk_bytes = 128u * p.cb_bytes;
    p.tx_bytes = p.blk_bytes;
    p.sbo_a = 8u * p.cb_bytes;
  }
  // blocks must keep 1024-byte alignment so every swizzle mode stays atom-aligned
  p.blk_bytes = (p.blk_bytes + 1023u) & ~1023u;
  // epilogue staging: rows of N * esize bytes (+16 B pad against bank conflicts); usable when a
  // row of real output is a power-of-two number of 16-byte lanes
  const int esize = i8 ? (out_kind >= 2 ? 1 : (out_kind == 1 ? 4 : 2)) : (out_f32 ? 4 : 2);
  const int row_bytes = d.cout * esize;
  const bool can_stage = row_bytes >= 16 && row_bytes <= 512 && (row_bytes & (row_bytes - 1)) == 0 &&
                         (out_pitch * esize) % 16 == 0 && (reinterpret_cast<uintptr_t>(out_base) & 15) == 0;
  p.stage_pitch = can_stage ? p.N * esize + 16 : 0;
  UYD_REQUIRE(!i8 || can_stage, UYD_E_UNSUPPORTED, "conv_tc int8: output rows must be a power-of-two number of 16-byte lanes");
  const size_t wres = (p.w_bytes + 1023u) & ~1023u;
  // as many epilogue groups as the staging tiles leave room for next to the resident weights and two stages
  const size_t two_stages = 2 * (((size_t)(p.mode == TC_HALO ? (uint32_t)kHaloRows * p.halo_pitch * p.cb_bytes : (p.mode == TC_PAIRS ? (uint32_t)kPairRows * kPairCols * 128u : 128u * p.cb_bytes)) + 1023u) & ~(size_t)1023);
  p.ngroups = kEpiGroups;
  while (p.ngroups > 1 && p.stage_pitch && wres + two_stages + kTailFixed + (size_t)128 * p.ngroups * p.stage_pitch > 227 * 1024 - 1024)
    p.ngroups >>= 1;
  size_t tail = kTailFixed + (size_t)128 * p.ngroups * p.stage_pitch;  // barriers + bias + row->pixel map + staging
  if (!i8 && wres + 2 * (size_t)(128u * p.cb_bytes) > 227 * 1024 - 1024 - tail) {
    p.stage_pitch = 0;  // weights leave no room for the staging tile: per-thread row stores
    p.ngroups = kEpiGroups;
    tail = kTailFixed;
  }
  const size_t budget = 227 * 1024 - 1024 - tail;  // (PAIRS may trade epilogue groups for a third stage below)
  if ((p.mode == TC_HALO || p.mode == TC_PAIRS) && wres + 2 * (size_t)p.blk_bytes > budget) {  // blocks too big: one box per tap
    p.mode = TC_PERTAP;
    p.blk_bytes = 128u * p.cb_bytes;
    p.tx_bytes = p.blk_bytes;
    p.sbo_a = 8u * p.cb_bytes;
    p.blk_bytes = (p.blk_bytes + 1023u) & ~1023u;
  }
  UYD_REQUIRE(wres + 2 * (size_t)p.blk_bytes <= budget, UYD_E_UNSUPPORTED, "conv_tc: weights (%u B) leave no room for 2 stages",
              p.w_bytes);
  int stages = (int)((budget - wres) / p.blk_bytes);
  if (p.mode == TC_PAIRS && stages < 3 && p.ngroups > 2 && p.stage_pitch) {
    // a PAIRS stage is a whole tile (39 KB): a third tile in flight hides more TMA latency than epilogue groups 3 and 4
    const size_t tail2 = kTailFixed + (size_t)128 * 2 * p.stage_pitch;
    const int stages2 = (int)((227 * 1024 - 1024 - tail2 - wres) / p.blk_bytes);
    if (stages2 > stages) { p.ngroups = 2; tail = tail2; stages = stages2; }
  }
  const int want = p.mode == TC_HALO ? 4 : (p.mode == TC_PAIRS ? 4 : 12);
  if (stages > want) stages = want;
  if (stages_override > 0 && stages_override < stages) stages = stages_override;
  {  // two issuing warps when the ring can be split between them (see TcParams::dual)
    const int bpt = p.mode == TC_PERTAP ? p.ncb * p.taps : p.ncb;
    const int even = stages - stages % (2 * bpt);  // never trade the third / fourth stage of a deep-latency ring for the second issuer
    p.dual = even >= 2 * bpt && (even == stages || even >= 4) && getenv("UYD_TC_SINGLE_ISSUER") == nullptr;
    if (p.dual) stages = even;
  }
  p.stages = stages;
  p.nacc = 4 * p.N <= 512 ? 4 : 2;
  tc->smem = 1024 + wres + (size_t)stages * p.blk_bytes + tail;
  p.out = out_base;
  p.out_pitch = out_pitch;
  p.out_f32 = out_f32;
  p.res = reinterpret_cast<const __nv_bfloat16 *>(res_base);
  p.res_pitch = res_pitch;
  p.bias = bias_dev;
  p.relu = d.relu;
  tc->w_dev = w_dev;

  const cuuint32_t one4[4] = {1, 1, 1, 1};
  {  // weights: [rows = ncb*taps*N][CB]
    const cuuint64_t dims[2] = {(cuuint64_t)CB, (cuuint64_t)p.ncb * p.taps * p.N};
    const cuuint64_t str[1] = {(cuuint64_t)p.cb_bytes};
    const cuuint32_t box[2] = {(cuuint32_t)CB, (cuuint32_t)p.N};
    int e = encode(&tc->tm_w, w_dev, 2, dims, str, box, one4, p.cb_bytes, i8);
    if (e) return e;
  }
  if (p.mode == TC_FLAT) {
    const cuuint64_t dims[2] = {(cuuint64_t)d.cin, (cuuint64_t)max_batch * ih * iw};
    const cuuint64_t str[1] = {(cuuint64_t)in_pitch * es};
    const cuuint32_t box[2] = {(cuuint32_t)CB, 128};
    int e = encode(&tc->tm_in, in_base, 2, dims, str, box, one4, p.cb_bytes, i8);
    if (e) return e;
  } else if (p.mode == TC_PAIRS) {  // [n][h][w/2][2 c]: a box row = one pixel pair = 128 contiguous bytes
    const cuuint64_t dims[4] = {(cuuint64_t)2 * d.cin, (cuuint64_t)(iw / 2), (cuuint64_t)ih, (cuuint64_t)max_batch};
    const cuuint64_t str[3] = {(cuuint64_t)2 * in_pitch * es, (cuuint64_t)iw * in_pitch * es, (cuuint64_t)ih * iw * in_pitch * es};
    const cuuint32_t box[4] = {(cuuint32_t)2 * CB, (cuuint32_t)kPairCols, (cuuint32_t)kPairRows, 1};
    int e = encode(&tc->tm_in, in_base, 4, dims, str, box, one4, 128, i8);
    if (e) return e;
  } else {
    const cuuint64_t dims[4] = {(cuuint64_t)d.cin, (cuuint64_t)iw, (cuuint64_t)ih, (cuuint64_t)max_batch};
    const cuuint64_t str[3] = {(cuuint64_t)in_pitch * es, (cuuint64_t)iw * in_pitch * es, (cuuint64_t)ih * iw * in_pitch * es};
    if (p.mode == TC_HALO) {
      const cuuint32_t box[4] = {(cuuint32_t)CB, (cuuint32_t)(kTileW + 2), p.halo_pitch == 16 ? 1u : (cuuint32_t)kHaloRows, 1};
      int e = encode(&tc->tm_in, in_base, 4, dims, str, box, one4, p.cb_bytes, i8);
      if (e) return e;
    } else {
      const cuuint32_t s = (cuuint32_t)d.stride;
      const cuuint32_t box[4] = {(cuuint32_t)CB, (cuuint32_t)kTileW * s, (cuuint32_t)kTileH * s, 1};
      const cuuint32_t estr[4] = {1, s, s, 1};
      int e = encode(&tc->tm_in, in_base, 4, dims, str, box, estr, p.cb_bytes, i8);
      if (e) return e;
    }
  }
  if (int e = smem_optin(conv_tc_kernel<false, 1>, 227 * 1024)) return e;
  if (int e = smem_optin(conv_tc_kernel<false, 2>, 227 * 1024)) return e;
  if (int e = smem_optin(conv_tc_kernel<false, 4>, 227 * 1024)) return e;
  if (int e = smem_optin(conv_tc_kernel<true, 1>, 227 * 1024)) return e;
  if (int e = smem_optin(conv_tc_kernel<true, 2>, 227 * 1024)) return e;
  if (int e = smem_optin(conv_tc_kernel<true, 4>, 227 * 1024)) return e;
  return UYD_OK;
}

int tc_launch(const TcConv *tc, int n0, int nb, int sm_count, cudaStream_t s) {
  TcParams p = tc->p;
  p.n0 = n0;
  p.nb = nb;
  p.tpi = (unsigned)((p.big ? p.pairs_x : p.tiles_x) * p.tiles_y);
  if (p.tpi == 0) p.tpi = 1;
  p.m_tpi = fastdiv_magic(p.tpi);
  p.m_tx = fastdiv_magic((unsigned)(p.big ? p.pairs_x : p.tiles_x));
  if (p.big) {
    p.total_tiles = p.mode == TC_FLAT ? ((long long)nb * p.H * p.W + 255) / 256 : (long long)nb * p.pairs_x * p.tiles_y;
    if (p.total_tiles == 0) return UYD_OK;
    UYD_REQUIRE((long long)(p.n0 + nb) * p.H * p.W < (1ll << 31) && p.total_tiles < (1ll << 24), UYD_E_UNSUPPORTED,
                "conv_tc big: %d images of %dx%d exceed the kernel's 32-bit pixel index", p.n0 + nb, p.H, p.W);
    const unsigned grid = (unsigned)(p.total_tiles < sm_count ? p.total_tiles : sm_count);
    if (p.i8) UYD_CUDA(launch_pdl(conv_tc_big_kernel<true>, dim3(grid), dim3(kBigThreads), tc->smem, s, tc->tm_in, tc->tm_w, p));
    else UYD_CUDA(launch_pdl(conv_tc_big_kernel<false>, dim3(grid), dim3(kBigThreads), tc->smem, s, tc->tm_in, tc->tm_w, p));
    return (int)cudaGetLastError();
  }
  p.total_tiles = p.mode == TC_FLAT ? ((long long)nb * p.H * p.W + 127) / 128 : (long long)nb * p.tiles_x * p.tiles_y;
  if (p.total_tiles == 0) return UYD_OK;
  UYD_REQUIRE((long long)(p.n0 + nb) * p.H * p.W < (1ll << 31) && p.total_tiles < (1ll << 24), UYD_E_UNSUPPORTED,
              "conv_tc: %d images of %dx%d exceed the kernel's 32-bit pixel index", p.n0 + nb, p.H, p.W);
  const unsigned grid = (unsigned)(p.total_tiles < sm_count ? p.total_tiles : sm_count);
  const int ks = p.cb_bytes / 32;
#define UYD_TC_LAUNCH(I8V, KS) UYD_CUDA(launch_pdl(conv_tc_kernel<I8V, KS>, dim3(grid), dim3(kThreads), tc->smem, s, tc->tm_in, tc->tm_w, p))
  if (p.i8) {
    if (ks == 1) UYD_TC_LAUNCH(true, 1); else if (ks == 2) UYD_TC_LAUNCH(true, 2); else UYD_TC_LAUNCH(true, 4);
  } else {
    if (ks == 1) UYD_TC_LAUNCH(false, 1); else if (ks == 2) UYD_TC_LAUNCH(false, 2); else UYD_TC_LAUNCH(false, 4);
  }
#undef UYD_TC_LAUNCH
  return (int)cudaGetLastError();
}

void tc_set_pre(TcConv *tc, const float *pre) { tc->p.pre = pre; }
TcConv *tc_new() { return new TcConv(); }
void tc_delete(TcConv *t) { delete t; }
const char *tc_mode_name(const TcConv *t) {
  if (t->p.big) return t->p.mode == TC_FLAT ? "big-flat" : (t->p.mode == TC_HALO ? "big-halo" : "big-pertap");
  return t->p.mode == TC_FLAT ? "flat" : (t->p.mode == TC_HALO ? "halo" : (t->p.mode == TC_PAIRS ? "pairs" : "pertap"));
}

}  // namespace uyd
