/* libuyd.so -- C ABI of the B200-native UNINA-YOLO-DLA inference hot path.
 *
 * Conventions (same as the reference's extern "C" surface,
 * ros2_ws/src/perception/include/gpu_postprocess.h:42-80): every entry point returns an
 * int that is a cudaError_t-compatible code (0 = success; UYD_E_* below for argument /
 * state errors), never throws, takes the cudaStream_t LAST, works on caller-owned device
 * pointers and allocates nothing after create/finalize.  No host synchronisation happens
 * inside any call; counts stay on the device.
 *
 * What each group replaces in the reference:
 *   uyd_create/destroy      <- init_postprocess_resources / cleanup_postprocess_resources
 *                              (gpu_postprocess.h:45,50; global singleton gpu_postprocess.cu:56
 *                              becomes a per-device handle)
 *   uyd_plan_*              <- the conv stack the reference runs through TensorRT
 *                              (perception_node.cpp:611-624) / PyTorch (DetectionModel.forward,
 *                              trainer.py:156; model.py:347-365)
 *   uyd_decode_dfl          <- Ultralytics Detect._inference + DFL (SURVEY.md a-8)
 *   uyd_decode_tlbr         <- decode_yolo_head (gpu_postprocess.h:62-65,
 *                              gpu_postprocess.cu:102-199, postprocess.hpp:94-145)
 *   uyd_nms                 <- Ultralytics non_max_suppression + torchvision.ops.nms
 *                              (train.py:396-405) and run_gpu_nms + copy_valid_detections_to_host
 *                              (gpu_postprocess.h:70-78)
 *   uyd_nms_ex              <- the same with multi_label / classes (DetectionValidator.postprocess,
 *                              YOLO.predict(classes=))
 *   uyd_nms_tlbr            <- decode_yolo_head x3 + run_gpu_nms of a whole batch in one launch
 *                              (perception_node.cpp:581-689)
 */
#ifndef UYD_H
#define UYD_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct uyd_ctx uyd_ctx;   /* per-device handle: workspaces, TMA encoder, SM count */
typedef struct uyd_plan uyd_plan; /* a compiled layer list with its activation buffers    */
typedef void *uyd_stream;         /* cudaStream_t */

enum {
  UYD_OK = 0,
  UYD_E_ARG = 10001,     /* bad argument                      */
  UYD_E_STATE = 10002,   /* call order / plan not finalized   */
  UYD_E_UNSUPPORTED = 10003,
  UYD_E_NOGPU = 10004    /* no sm_100 device                  */
};

enum { UYD_BF16 = 0, UYD_F32 = 1, UYD_S8 = 2 };

/* Which kernel family executes a convolution. AUTO picks tensor cores when the shape
 * allows it.  DIRECT = CUDA-core reference kernel (used for tiny channel counts and as an
 * on-device cross-check). */
enum { UYD_IMPL_AUTO = 0, UYD_IMPL_DIRECT = 1, UYD_IMPL_TC = 2 };

int uyd_version(void);
const char *uyd_last_error(void);
int uyd_create(int device, uyd_ctx **out);
int uyd_destroy(uyd_ctx *ctx);
int uyd_sm_count(const uyd_ctx *ctx);

/* ------------------------------------------------------------------------------------
 * Plan: activation buffers (NHWC, bf16 unless stated) + an ordered list of ops.
 * Buffers are addressed as (id, channel offset): producers write straight into channel
 * slices of wider buffers, so concat / chunk never materialise.
 * ---------------------------------------------------------------------------------- */
int uyd_plan_create(uyd_ctx *ctx, int max_batch, uyd_plan **out);
int uyd_plan_destroy(uyd_plan *plan);

/* Declares an activation buffer [max_batch, h, w, c] of dtype; returns its id (>= 0) in *id. */
int uyd_plan_add_buffer(uyd_plan *plan, int h, int w, int c, int dtype, int *id);

typedef struct uyd_conv {
  int in_buf, in_coff;     /* input slice; in_buf = -1: the network input x (NCHW fp32)   */
  int out_buf, out_coff;   /* output slice                                                 */
  int res_buf, res_coff;   /* residual slice added AFTER the activation, -1 = none         */
  int cin, cout;           /* logical channels                                             */
  int k, stride;           /* 1|3 , 1|2 ; padding k/2                                      */
  int depthwise;           /* 1: groups == cin == cout                                     */
  int relu;                /* 1: ReLU after (folded BN) bias                               */
  int impl;                /* UYD_IMPL_*                                                   */
  int pre_buf_p1;          /* 0: none; else 1 + id of an fp32 buffer [h/2, w/2, cout] that is added,
                              nearest-x2 upsampled, BEFORE the activation: Upsample + Concat + 1x1 Conv is
                              computed as up(W_a * x_low) + W_b * x_skip, the upsampled tensor and the
                              concatenation are never written (tensor-core path only)              */
} uyd_conv;

/* weight: host fp32 [cout][cin/groups][k][k] (PyTorch layout, BN already folded);
 * bias: host fp32 [cout].  Packed to the kernel's layout and uploaded here. */
int uyd_plan_add_conv(uyd_plan *plan, const uyd_conv *desc, const float *weight, const float *bias);

/* Fused stem (csrc/stem_fused.cu): the first two layers of the YAML graph, Conv(3,16,3,2) -> Conv(16,32,3,2)
 * (both Conv+BN+ReLU, BN folded), in one launch reading the network input; the 16-channel tensor between
 * them stays in shared memory.  Must be the first op.  w0 [16][3][3][3], w1 [32][16][3][3] (PyTorch layout).
 * The output buffer has a quarter of the frame extent. */
int uyd_plan_add_stem2(uyd_plan *plan, int out_buf, int out_coff, const float *w0, const float *b0, const float *w1,
                       const float *b1);
/* The same launch with the 1x1 Conv(32,16)+BN+ReLU that consumes the stem folded in (model.2.cv1 of
 * unina-yolo-dla-m.yaml, ultralytics C3k2.cv1): w2 [16][32], b2 [16].  The stem's 32-channel output is rounded to
 * bf16 in registers and never written; the 16-channel output slice needs 8-byte alignment. */
int uyd_plan_add_stem2_pw(uyd_plan *plan, int out_buf, int out_coff, const float *w0, const float *b0, const float *w1,
                          const float *b1, const float *w2, const float *b2);

/* INT8 convolution (QAT fake-quant semantics of qat.py:109-124 as an integer computation,
 * oracle/quant.py): input slice int8 (UYD_S8 buffer), weight int8 [cout][cin][k][k] already
 * quantised, exact int32 accumulation, y = float(acc) * mult[c] + bias[c] (fp32, separate
 * round-to-nearest multiply and add), optional ReLU.  The output buffer's dtype selects the
 * epilogue: UYD_S8 -> q = clamp(rne(y * out_scale), -127, 127) (the consumer's input quantiser),
 * UYD_F32 / UYD_BF16 -> y.  Bit-exact w.r.t. the integer reference.
 * Tensor-core routes (tcgen05 kind::i8, int8 slices 16-byte aligned, 16-byte output rows): weights resident in shared memory
 * for cout <= 128 with a power-of-two number of 16-byte lanes per output row; otherwise, when cin % 128 == 0,
 * cout % 16 == 0, cout <= 256 and there are no partial sums, weights streamed per (channel block, tap)
 * (uyd_plan_op_info: tc:big-halo / big-pertap / big-flat).  Other convs run on CUDA cores (dp4a). */
typedef struct uyd_conv_s8 {
  int in_buf, in_coff, out_buf, out_coff;
  int cin, cout, k, stride, relu;
  float out_scale;
  int impl;
  int depthwise;           /* 1: groups == cin == cout (weight [c][1][k][k])                              */
  int res_buf, res_coff;   /* bf16 residual slice added (fp32) AFTER the activation, res_buf = -1: none */
  int out_round_bf16;      /* UYD_S8 output only: 1 = y is rounded to bf16 before the consumer's quantiser, i.e. the bytes a
                              bf16 activation + uyd_plan_add_quantize would produce, without materialising the activation */
  int pre_buf_p1;          /* 0: none; b + 1: fp32 buffer b [h/2, w/2, cout] of INTEGER partial sums (an int8 1x1 conv with
                              m = 1, b = 0 into a UYD_F32 buffer) added, nearest-x2 upsampled, to the accumulator before the
                              requant: Upsample + Concat + QuantConv2d(1x1) without the upsampled tensor (exact: the sums
                              stay below 2^24).  1x1 convs on the tensor-core path, cout % 16 == 0 */
} uyd_conv_s8;
int uyd_plan_add_conv_s8(uyd_plan *plan, const uyd_conv_s8 *desc, const int8_t *weight_q, const float *mult,
                         const float *bias);

/* Input quantiser of a QuantConv2d (qat.py:109-124): q = clamp(rne(x * scale), -127, 127), scale = 127 / amax,
 * from a bf16 slice into a slice of a UYD_S8 buffer of the same extent (C % 4 == 0). */
int uyd_plan_add_quantize(uyd_plan *plan, int in_buf, int in_coff, int out_buf, int out_coff, int c, float scale);

/* Fused C3k block (Ultralytics C3k with two 3x3 bottlenecks; the interior of every C3k2 of the
 * YAML graph): y = cv3(cat(m1(m0(cv1 x)), cv2 x)), all seven Conv+BN+ReLU layers and both
 * residual adds in one launch, intermediates in shared memory.  weights/biases, BN folded,
 * PyTorch layout: [0] cv1 [c/2][c][1][1], [1] cv2 [c/2][c][1][1], [2..5] m0.cv1, m0.cv2, m1.cv1, m1.cv2
 * [c/2][c/2][3][3], [6] cv3 [c][c][1][1].  c in {8, 16, 32}; W % 40 == 0; H % 32, 20 or 16 == 0. */
typedef struct uyd_c3k {
  int in_buf, in_coff, out_buf, out_coff, c, reserved;
} uyd_c3k;
int uyd_plan_add_c3k(uyd_plan *plan, const uyd_c3k *desc, const float *const weights[7], const float *const biases[7]);

/* The same block of the INT8 (fake-quant) graph, qat.py:109-124: every one of the seven convs is a QuantConv2d.
 * weights[i]: int8 codes of conv i (layouts as above), mult[i] / biases[i]: its per-channel requant pair
 * (y = float(acc) * m_c + b_c), in_scale[i] = 127 / amax of its input quantiser (i in the order cv1, cv2, m0.cv1, m0.cv2,
 * m1.cv1, m1.cv2, cv3).  Input and output slices are bf16 (the activations the graph defines); all integer sums are
 * exact, every rounding is the one the unfused ops (uyd_plan_add_quantize + uyd_plan_add_conv_s8) perform: the output
 * equals theirs bit for bit.  One launch instead of seven convs and four to five quantize passes. */
int uyd_plan_add_c3k_s8(uyd_plan *plan, const uyd_c3k *desc, const int8_t *const weights[7], const float *const mult[7],
                        const float *const biases[7], const float *in_scale);

/* Fused class branch of the Detect head (Detect.cv3[l], non-legacy): DWConv(cin,cin,3) -> Conv(cin,mid,1)
 * -> DWConv(mid,mid,3) -> Conv(mid,mid,1) -> Conv2d(mid,nc,1) in one launch; the nc logits are
 * written as fp32 into a slice of the head buffer.  weights/biases (BN folded): [0] dw1 [cin][1][3][3],
 * [1] pw1 [mid][cin][1][1], [2] dw2 [mid][1][3][3], [3] pw2 [mid][mid][1][1], [4] pw3 [nc][mid][1][1] (+ its bias).
 * cin in {32, 64}, mid == 32, nc <= 8, W % 40 == 0, H % 8 == 0. */
typedef struct uyd_cls_branch {
  int in_buf, in_coff, out_buf, out_coff, cin, mid, nc, reserved;
} uyd_cls_branch;
int uyd_plan_add_cls_branch(uyd_plan *plan, const uyd_cls_branch *desc, const float *const weights[5],
                            const float *const biases[5]);

/* Chained head kernel (csrc/conv_chain.cu): 3x3 stride-1 Conv+BN+ReLU (cin -> n1; dw1 = 1: the
 * depth-wise DWConv(cin,cin,3), cin == n1) followed in the same launch by a 1x1 conv (n1 -> n2) and a
 * fused final stage, all on tcgen05 with the intermediate tile kept in shared memory:
 *   UYD_CHAIN_STORE : bias2 (+ReLU when relu2) -> out slice (bf16 or fp32 buffer)
 *   UYD_CHAIN_PW3   : ReLU -> Conv2d(n2, nc, 1) (w3, b3; Detect.cv3[l][2]) -> raw logits into the out slice
 *                     (when out_buf >= 0) and sigmoid scores into y channels [y_ch0, y_ch0 + nc)
 *   UYD_CHAIN_DFL   : n2 == 64 box logits -> raw fp32 into the out slice (when out_buf >= 0) and the DFL
 *                     softmax-integral decode (cx, cy, w, h) * stride_px into y channels [y_ch0, y_ch0 + 4)
 * y is the decoded output [batch, no, a_total] handed to uyd_plan_run_decoded; this op writes anchors
 * [a_off, a_off + H*W).  cin, n1 in {32, 64}; n2 <= 64; nc <= 8.
 * w1: [n1][cin][3][3] (dw1: [n1][1][3][3]), w2: [n2][n1], w3: [nc][n2]; BN folded, PyTorch layout. */
enum { UYD_CHAIN_STORE = 0, UYD_CHAIN_PW3 = 2, UYD_CHAIN_DFL = 3 };
typedef struct uyd_chain {
  int in_buf, in_coff, cin, n1, n2, dw1, relu2, final_kind;
  int out_buf, out_coff, nc;
  int a_total, a_off, y_ch0, no;
  float stride_px;
} uyd_chain;
int uyd_plan_add_chain(uyd_plan *plan, const uyd_chain *desc, const float *w1, const float *b1, const float *w2,
                       const float *b2, const float *w3, const float *b3);

/* SPPF cascade: reads slice [coff, coff+c) of buf and writes pool5, pool5^2, pool5^3 to
 * slices [coff+c, coff+2c), [coff+2c, ..), [coff+3c, ..) of the same buffer
 * (trainer.py:119-124; -inf padding). */
int uyd_plan_add_sppf_pool(uyd_plan *plan, int buf, int coff, int c);

/* nearest x2 upsample of a slice into a slice of a buffer with twice the extent. */
int uyd_plan_add_upsample2x(uyd_plan *plan, int in_buf, int in_coff, int out_buf, int out_coff, int c);

/* Marks the three raw head buffers ([B,H,W,no] fp32, box logits first then class logits)
 * in level order (stride 4, 8, 16 ...) for uyd_plan_run_decode. */
int uyd_plan_set_heads(uyd_plan *plan, const int *head_bufs, const int *strides, int nl, int reg_max, int nc);

int uyd_plan_finalize(uyd_plan *plan);
size_t uyd_plan_bytes(const uyd_plan *plan);
int uyd_plan_num_launches(const uyd_plan *plan);

/* Device pointer of a buffer (valid after finalize); for layer-level parity checks. */
int uyd_plan_buffer_ptr(uyd_plan *plan, int id, void **ptr);

/* Runs every op for `batch` images.  x: device NCHW fp32 [batch,3,H,W] (the reference
 * forward signature, model.py:347 / DetectionModel.forward).  */
int uyd_plan_run(uyd_plan *plan, const float *x, int batch, uyd_stream stream);

/* Same, for uint8 NCHW frames [batch,3,H,W]: the stem divides by 255 on load, which is the
 * reference predictor's pre-process (im.float() / 255) fused into the first conv. */
int uyd_plan_run_u8(uyd_plan *plan, const uint8_t *x, int batch, uyd_stream stream);

/* Same as uyd_plan_run / _run_u8 (x_dtype = UYD_F32 | UYD_U8) for plans whose head ops decode in their
 * epilogue (uyd_plan_add_chain with PW3 / DFL finals): y [batch, no, a_total] fp32 receives the decoded
 * prediction directly, no raw head tensor is materialised. */
enum { UYD_U8 = 3 };
int uyd_plan_run_decoded(uyd_plan *plan, const void *x, int x_dtype, int batch, float *y, uyd_stream stream);

/* Measurement hooks (CUDA events on `stream`, no effect on results):
 *  - uyd_plan_profile: one pass with every op bracketed; ms[uyd_plan_num_launches]; syncs.
 *  - uyd_plan_set_timed_op / _read: bracket ONE op inside normal uyd_plan_run calls.
 *  - uyd_plan_op_info: description + algorithmic flops / compulsory bytes per image. */
int uyd_plan_profile(uyd_plan *plan, const float *x, int batch, uyd_stream stream, float *ms);
/* decoded-output buffer the profiling pass hands to head ops that decode in their epilogue */
int uyd_plan_set_profile_output(uyd_plan *plan, float *y);
int uyd_plan_set_timed_op(uyd_plan *plan, int op, int max_samples);
int uyd_plan_timed_op_read(uyd_plan *plan, float *total_ms, int *samples);
int uyd_plan_op_info(uyd_plan *plan, int op, char *text, size_t text_len, double *flops_per_image,
                     double *bytes_per_image);

/* DFL decode of the plan's heads -> y [batch, 4+nc, A] fp32 (cx,cy,w,h in pixels, sigmoid
 * class scores), A = sum of H_l*W_l, levels concatenated in head order. */
int uyd_plan_run_decode(uyd_plan *plan, float *y, int batch, uyd_stream stream);

/* INT8 graphs: the DFL projection conv (frozen arange(16) weights) is a QuantConv2d like every other conv
 * (train.py:725): amax_in > 0 makes uyd_plan_run_decode quantise the softmax probabilities with 127 / amax_in
 * and the weights with 127 / 15; 0 switches it off. */
int uyd_plan_set_dfl_quant(uyd_plan *plan, float amax_in);

/* Optional: raw heads as the reference returns them, NCHW fp32 [batch, no, H_l, W_l]. */
int uyd_plan_export_head_nchw(uyd_plan *plan, int level, float *out, int batch, uyd_stream stream);

/* ------------------------------------------------------------------------------------
 * Stand-alone post-processing on caller-owned device memory.
 * ---------------------------------------------------------------------------------- */

/* DFL decode of one level.  head: [batch,H,W,4*reg_max+nc] fp32 (NHWC).
 * Writes y[b, :, a_off + i] for i in [0,H*W), y laid out [batch, 4+nc, a_total]. */
int uyd_decode_dfl(uyd_ctx *ctx, const float *head, int batch, int h, int w, int reg_max, int nc,
                   float stride, float *y, int a_total, int a_off, uyd_stream stream);

/* 32-byte detection record, layout-identical to GpuDetection (gpu_postprocess.h:27-33). */
typedef struct uyd_detection {
  float x1, y1, x2, y2;
  float confidence;
  int class_id;
  int valid;
  int _pad;
} uyd_detection;

/* TLBR decode of one level (signature-compatible superset of decode_yolo_head):
 * cls [nc,H,W], reg [4,H,W] CHW fp32 per image; appends to dets (capacity cap) through the
 * device counter d_count (caller zeroes it); keeps a cell iff conf > thr (strict=1,
 * postprocess.hpp:116) or conf >= thr (strict=0, gpu_postprocess.cu:132). Also writes the
 * flat cell index (+ cell_base, so that levels get disjoint ranges) of every detection to
 * cell_idx when non-NULL: the NMS uses it as a deterministic tie-break. */
int uyd_decode_tlbr(uyd_ctx *ctx, const float *d_cls, const float *d_reg, uyd_detection *dets,
                    int *cell_idx, int *d_count, int cap, int grid_w, int grid_h, int stride,
                    int num_classes, float conf_thr, float conformal_q, int strict,
                    int cell_base, uyd_stream stream);

/* Workspace size needed by uyd_nms for (batch, anchors). */
size_t uyd_nms_workspace_bytes(int batch, int anchors);

/* Ultralytics non_max_suppression on y [batch, 4+nc, anchors] fp32:
 *   keep conf > conf_thr, best class, stable score-descending order (ties: lower anchor
 *   first), top max_nms, class-offset (cls*max_wh) greedy NMS with IoU > iou_thr
 *   (fp32 IoU compared against the double threshold, like torchvision), first max_det.
 * out_det [batch, max_det, 6] fp32 rows (x1,y1,x2,y2,conf,cls); out_idx [batch, max_det]
 * anchor index of every kept row (may be NULL); out_count [batch].  Every output element is
 * written: rows past the count are zeros, their index -1 (no pre-initialisation needed). */
int uyd_nms(uyd_ctx *ctx, const float *y, int batch, int nc, int anchors, float conf_thr,
            double iou_thr, int max_nms, int max_det, float max_wh, void *workspace,
            size_t workspace_bytes, float *out_det, int *out_idx, int *out_count,
            uyd_stream stream);

/* The non_max_suppression options of Ultralytics that uyd_nms does not take. */
typedef struct uyd_nms_options {
  int multi_label;           /* 0: best class per anchor (uyd_nms); 1: every (anchor, class) with score > conf_thr */
  int num_filter_classes;    /* entries of filter_classes (host array); ignored when filter_classes is NULL */
  const int *filter_classes; /* NULL: all classes; non-NULL: keep only these ids (ids outside [0, nc) match nothing,
                                0 entries keep nothing) */
} uyd_nms_options;

/* uyd_nms with options (opt == NULL is uyd_nms itself; no workspace is needed).
 *   multi_label (with nc > 1): every (anchor, class) pair with score > conf_thr is a candidate, ranked by score
 *     descending, then anchor, then class ascending (the row-major order of Ultralytics' torch.where under a stable
 *     sort); the row's conf is that class's score and out_idx its anchor.  max_nms then counts pairs.
 *   filter_classes: applied to the best class of an anchor (an anchor whose best class is not listed is dropped; it
 *     does not fall back to another class), or to each pair under multi_label -- before the max_nms truncation.
 * Class-agnostic NMS is max_wh = 0.  UYD_E_ARG, with nothing launched, for num_filter_classes < 0 or > 0 with a
 * NULL filter_classes, besides the errors of uyd_nms.  No host synchronisation (CUDA-graph capturable). */
int uyd_nms_ex(uyd_ctx *ctx, const float *y, int batch, int nc, int anchors, float conf_thr, double iou_thr,
               int max_nms, int max_det, float max_wh, const uyd_nms_options *opt, float *out_det, int *out_idx,
               int *out_count, uyd_stream stream);

/* Greedy class-aware NMS over uyd_detection records (postprocess.hpp:44-67 semantics:
 * confidence-descending, same class, IoU > thr; ties broken by cell_idx ascending, or by
 * slot when cell_idx is NULL).  Replaces run_gpu_nms + copy_valid_detections_to_host's
 * compaction (gpu_postprocess.h:70-78): `dets` (first min(*d_count, cap) records) is left
 * untouched; survivors are written compacted, in kept order, to `out` (at most 1024, the
 * reference's MAX_DETECTIONS) and their number to *d_out_count (device). */
size_t uyd_nms_detections_workspace_bytes(int cap);
int uyd_nms_detections(uyd_ctx *ctx, const uyd_detection *dets, const int *cell_idx,
                       const int *d_count, int cap, float iou_thr, void *workspace,
                       size_t workspace_bytes, uyd_detection *out, int *d_out_count,
                       uyd_stream stream);

/* In-place form with the semantics run_gpu_nms leaves behind (gpu_postprocess.h:70-71, gpu_postprocess.cu:366-387):
 * the first n (<= 1024, host-side count as in the reference signature) records of `dets` are rewritten in
 * confidence-descending order (ties: cell_idx, or slot when NULL) with valid = 1 for survivors of the exact greedy
 * NMS and 0 for suppressed records; records that arrive with valid == 0 neither suppress nor survive.
 * d_out_count (device, may be NULL) receives the number of survivors. */
int uyd_nms_detections_inplace(uyd_ctx *ctx, uyd_detection *dets, const int *cell_idx, int n, float iou_thr,
                               int *d_out_count, uyd_stream stream);

/* TLBR decode (postprocess.hpp:94-145) + class-aware greedy NMS (postprocess.hpp:44-67) of a whole batch in ONE
 * launch.  heads[l]: [batch, grid_h[l], grid_w[l], num_classes + 4] fp32 (class logits, then l, t, r, b distances).
 * Ties in confidence resolve to the lower cell index (levels numbered consecutively in the given order).
 * max_nms > 0: only the max_nms best candidates per image enter the NMS.  out_det [batch, max_det, 6]
 * (x1,y1,x2,y2,conf,cls), out_count [batch]; every element written.  max_det <= 1024.
 * Per cell, the same statement as uyd_decode_tlbr (conf_thr, conformal_q, strict), so the rows equal those of
 * uyd_decode_tlbr per level followed by uyd_nms_detections.  heads, grid_h, grid_w and strides are host arrays of nl
 * entries.  Nothing is launched and UYD_E_ARG is returned for nl < 1, a NULL pointer, a non-positive batch, class
 * count, grid size or stride, max_nms < 0 or a head not aligned to a float; UYD_E_UNSUPPORTED for nl > 8, max_det
 * outside [1, 1024] or 2^31 cells or more per image.  No host synchronisation. */
int uyd_nms_tlbr(uyd_ctx *ctx, const float *const *heads, const int *grid_h, const int *grid_w, const int *strides,
                 int nl, int batch, int num_classes, float conf_thr, float conformal_q, int strict, float iou_thr,
                 int max_nms, int max_det, float *out_det, int *out_count, uyd_stream stream);

/* Ordered compaction of the valid records among the first n (<= 1024) into `out` + their number (device):
 * the cub::DeviceSelect::If of copy_valid_detections_to_host (gpu_postprocess.cu:412-416). */
int uyd_compact_valid(uyd_ctx *ctx, const uyd_detection *dets, int n, uyd_detection *out, int *d_out_count,
                      uyd_stream stream);

/* max |x| over the first `batch` images of a bf16 slice, as the bit pattern of a non-negative float OR-ed into
 * *d_bits with atomicMax (caller zeroes it): max calibration of the static input scales (qat.py:129-220). */
int uyd_plan_slice_absmax(uyd_plan *plan, int buf, int coff, int c, int batch, unsigned int *d_bits, uyd_stream stream);

/* Histogram of |x| over the first `batch` images of a bf16 slice, ADDED into d_hist[nbins] (caller zeroes it):
 * bin = min(floor(|x| * inv_width), nbins - 1).  The collection step of the histogram / entropy calibrator that
 * qat.py:91-126 configures by default (pytorch-quantization HistogramCalibrator: 2048 bins over [0, first max],
 * the range grows by whole bins when a later batch exceeds it). */
int uyd_plan_slice_histogram(uyd_plan *plan, int buf, int coff, int c, int batch, float inv_width, int nbins,
                             unsigned int *d_hist, uyd_stream stream);

/* Batched evaluation of the detections (the consumer of the gathered [N, 6] rows):
 *   counters[0..2] += small-object TP, FP, FN with the semantics of UninaValidator.update_metrics
 *     (trainer.py:210-265): boxes in pixels, "small" = width and height < size_thr, a match = same class
 *     and Ultralytics box_iou > small_iou_thr; images without a small ground truth are skipped;
 *   scores [batch, max_det] (may be NULL) = 1 - IoU of every prediction greedily matched, in confidence
 *     order, to the best unmatched same-class ground truth with IoU >= match_iou_thr, else -1: the
 *     nonconformity scores of calibrate_conformal_prediction (train.py:335-470).
 * det [batch, max_det, 6] rows (x1,y1,x2,y2,conf,cls) in confidence order with count [batch] valid rows
 * (uyd_nms output); gt [batch, gt_max, 5] rows (cls, x1, y1, x2, y2) in pixels with gt_count [batch]. */
int uyd_eval_update(uyd_ctx *ctx, const float *det, const int *count, int batch, int max_det, const float *gt,
                    const int *gt_count, int gt_max, float size_thr, float small_iou_thr, float match_iou_thr,
                    unsigned long long *counters, float *scores, uyd_stream stream);

/* data_loader.SmallObjectMetric.update (data_loader.py:322-389), the training-time small-object metric, batched:
 * pred [batch, max_det, 6] rows (x_c, y_c, w, h, conf, cls) and gt [batch, gt_max, 5] rows (cls, x_c, y_c, w, h), both
 * normalised to the image, predictions in confidence order, count / gt_count valid rows per image.
 * counters[0..2] += TP, FP, FN (greedy one-to-one matching in confidence order against the small ground truths). */
int uyd_small_object_metric_update(uyd_ctx *ctx, const float *pred, const int *count, int batch, int max_det, const float *gt,
                                   const int *gt_count, int gt_max, double size_thr, double iou_thr, double image_size,
                                   unsigned long long *counters, uyd_stream stream);

/* mAP50 / mAP50-95, stage 1: Ultralytics DetectionValidator.match_predictions for every image of the batch, one
 * launch.  det / count / gt / gt_count as in uyd_eval_update (both in the same pixel space).  For each row i of
 * image b, record r = b * max_det + i gets:
 *   tp_mask[r]  bit t set when the row is a TP at IoU threshold iou_thresholds[t] (box_iou >= t, same class; each
 *               detection keeps its best ground truth, the higher index winning an IoU tie, and each ground truth
 *               its lowest-index detection);
 *   sort_key[r] class << 32 | the confidence's bits ordered so that an ascending sort is a descending confidence
 *               (-0 ranks as +0); rows >= count[b] get INT64_MAX.
 * n_labels[nc] += the ground truths per class.  A ground truth or a valid row whose class is not an integer in
 * [0, nc), or a row whose confidence is NaN, is not indexed: it adds 1 to *dropped and its row gets INT64_MAX.
 * Sorting all records of all calls by key, stably and in (call, image, row) order, gives ap_per_class's order.
 * Limits: 1 <= n_thresholds <= 16, every threshold > 0 (UYD_E_ARG); nc <= 2^20, gt_max <= 1024 and
 * max_det <= 1024 (UYD_E_UNSUPPORTED; gt_max is rejected, never clamped).  Nothing is launched on an error. */
int uyd_eval_match(uyd_ctx *ctx, const float *det, const int *count, int batch, int max_det, const float *gt,
                   const int *gt_count, int gt_max, int nc, const float *iou_thresholds, int n_thresholds,
                   unsigned short *tp_mask, long long *sort_key, long long *n_labels, long long *dropped, uyd_stream stream);

/* mAP50 / mAP50-95, stage 2: Ultralytics metrics.ap_per_class per class, one CTA per class, bit-exact fp64.
 * sorted_key [n_records] ascending (uyd_eval_match keys after a stable sort), order [n_records] the record index of
 * each sorted key into tp_mask, n_labels [nc] from uyd_eval_match.  Writes ap [nc, n_thresholds] (compute_ap, the
 * 101-point interpolation), p_curve / r_curve [nc, 1000] (precision / recall at confidences np.linspace(0, 1, 1000),
 * threshold 0).  A class without records or without labels gets zeros.  Limits: n_records > 0, 1 <= n_thresholds
 * <= 16 (UYD_E_ARG); nc <= 2^20 (UYD_E_UNSUPPORTED). */
int uyd_eval_ap(uyd_ctx *ctx, const long long *sorted_key, const long long *order, const unsigned short *tp_mask,
                long long n_records, const long long *n_labels, int nc, int n_thresholds, double *ap, double *p_curve,
                double *r_curve, uyd_stream stream);

/* ------------------------------------------------------------------------------------
 * Camera-frame pre-processing in front of the plan (drop-in for cuda_preprocess.h:62-84; kernels
 * cuda_preprocess.cu:99-253): BGRA / NV12 bytes -> RGB, (x / 255 - mean) / std, planar CHW fp32.
 * uyd_norm_params is layout-identical to NormParams (cuda_preprocess.h:38-45).  The *_batch variants
 * process `batch` frames `frame_stride` bytes apart into [batch, 3, H, W].
 * ---------------------------------------------------------------------------------- */
typedef struct uyd_norm_params {
  float mean_r, mean_g, mean_b, std_r, std_g, std_b;
} uyd_norm_params;
uyd_norm_params uyd_norm_params_imagenet(void); /* create_norm_params_imagenet */
uyd_norm_params uyd_norm_params_unit(void);     /* mean 0, std 1: plain x / 255 (the Ultralytics predictor's pre-process) */
int uyd_preprocess_bgra_resize(const uint8_t *d_input, float *d_output, int src_width, int src_height, int src_pitch,
                               int dst_width, int dst_height, uyd_norm_params params, uyd_stream stream);
int uyd_preprocess_bgra(const uint8_t *d_input, float *d_output, int width, int height, int pitch, uyd_norm_params params,
                        uyd_stream stream);
int uyd_preprocess_nv12(const uint8_t *d_y_plane, const uint8_t *d_uv_plane, float *d_output, int width, int height,
                        int y_pitch, int uv_pitch, uyd_norm_params params, uyd_stream stream);
int uyd_preprocess_bgra_batch(const uint8_t *d_input, float *d_output, int batch, long long frame_stride, int width,
                              int height, int pitch, uyd_norm_params params, uyd_stream stream);
int uyd_preprocess_bgra_resize_batch(const uint8_t *d_input, float *d_output, int batch, long long frame_stride,
                                     int src_width, int src_height, int src_pitch, int dst_width, int dst_height,
                                     uyd_norm_params params, uyd_stream stream);

/* f-1 as SURVEY 8f ranks it: camera bytes feed model.0 DIRECTLY.  The plan's first op must be a stem with a camera
 * loader: the YAML network's fused stem (uyd_plan_add_stem2 / _pw) or a CUDA-core Conv(3 -> 32, 3x3, stride 2) on the
 * network input with a 16-byte aligned output slice (model.py's stem at base_channels 32); any other plan returns
 * UYD_E_UNSUPPORTED before any launch.  The stem reads the packed BGRA pixels -- bilinearly resampled with the half-pixel rule of
 * preprocess_bgra_resize (cuda_preprocess.cu:140-199) when the frame extent differs from the plan's input -- or the
 * NV12 planes (cuda_preprocess.cu:207-253, frame extent == plan input), normalises ((v / 255) - mean) / std on load
 * and never writes a CHW fp32 tensor (4.9 MB written + read back per 640 x 640 frame otherwise).
 * UYD_CAM_BGRA_LETTERBOX: packed BGRA of any extent, letterboxed as the Ultralytics predictor does
 * (LetterBox(center=True, scaleup=True)): the frame is resized, aspect kept, to (new_w, new_h) of
 * uyd_letterbox_geometry with cv2 4.x's resize(INTER_LINEAR) for uint8, byte for byte, and placed at (top, left) of
 * the plan's input; every other pixel is byte 114.  Those bytes are normalised as UYD_CAM_BGRA's are, so the stem sees
 * what the cv2-letterboxed frame as a uint8 tensor gives.  Same layout rules as UYD_CAM_BGRA; a frame whose
 * letterboxed extent would be empty is UYD_E_ARG.  Boxes go back to frame pixels with uyd_letterbox_boxes.
 * y: decoded output [batch, no, a_total] for plans whose head ops decode in their epilogue, else NULL. */
enum { UYD_CAM_BGRA = 1, UYD_CAM_NV12 = 2, UYD_CAM_BGRA_LETTERBOX = 3 };
typedef struct uyd_camera_frames {
  int format;                 /* UYD_CAM_*                                                         */
  int width, height;          /* camera frame extent in pixels                                     */
  int pitch, uv_pitch;        /* row pitch in bytes of the BGRA pixels / Y plane, and of the UV plane */
  long long frame_stride;     /* bytes between consecutive frames of the batch (data)              */
  long long uv_frame_stride;  /* ... (uv)                                                          */
  const uint8_t *data;        /* device: BGRA pixels, or the Y plane                               */
  const uint8_t *uv;          /* device: interleaved U, V plane (NV12), else NULL                  */
  uyd_norm_params norm;
} uyd_camera_frames;
int uyd_plan_run_camera(uyd_plan *plan, const uyd_camera_frames *frames, int batch, float *y, uyd_stream stream);

/* Letterbox geometry of a src_w x src_h frame in a dst_w x dst_h model input (Ultralytics LetterBox / scale_boxes):
 * gain = min(dst_h / src_h, dst_w / src_w) in double, new_w = round(src_w gain), new_h = round(src_h gain),
 * left = round((dst_w - new_w) / 2 - 0.1), top = round((dst_h - new_h) / 2 - 0.1), rounding half to even as Python's
 * round does.  UYD_E_ARG for a non-positive extent or a NULL output.  Host only, no device work. */
int uyd_letterbox_geometry(int src_w, int src_h, int dst_w, int dst_h, int *new_w, int *new_h, int *left, int *top,
                           double *gain);

/* Boxes of a letterboxed batch back to frame pixels, in place: rows r < count[b] of det [batch, max_det, 6]
 * (x1, y1, x2, y2, conf, cls; uyd_nms / uyd_nms_tlbr output) get x -= left, y -= top, then x, y times the fp32
 * reciprocal of (float)gain, then x clamped to [0, src_w] and y to [0, src_h] (NaN kept) -- the float32 result of
 * Ultralytics' scale_boxes + clip_boxes statements on a CUDA tensor.  Rows past the count and columns 4, 5 are not
 * touched.  One launch, no host synchronisation (CUDA-graph capturable).  Nothing is launched and UYD_E_ARG is
 * returned for a NULL pointer, det not aligned to a float, a non-positive batch, max_det or extent, or an empty
 * letterboxed frame. */
int uyd_letterbox_boxes(uyd_ctx *ctx, float *det, const int *count, int batch, int max_det, int src_w, int src_h, int dst_w,
                        int dst_h, uyd_stream stream);

/* Pinned host staging memory for frame batches (cudaHostAlloc).  write_combined != 0: write-combined pages -- the
 * producer (camera driver, decoder) fills them sequentially, the GPU reads them over PCIe without cache snooping;
 * do not read them back on the CPU. */
int uyd_host_alloc(size_t bytes, int write_combined, void **out);
int uyd_host_free(void *p);

/* Plain device-to-device copy on `stream` (lets a host binding without a CUDA runtime of
 * its own read plan buffers into memory it owns). */
int uyd_memcpy_d2d(void *dst, const void *src, size_t bytes, uyd_stream stream);

#ifdef __cplusplus
}
#endif
#endif /* UYD_H */
