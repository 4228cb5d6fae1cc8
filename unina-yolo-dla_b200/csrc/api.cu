// C-ABI boundary of libuyd: handle, plan (buffers + ops), run, decode, head export.
#include <cstdarg>
#include <cstdlib>
#include <memory>
#include <mutex>
#include <set>
#include <utility>

#include "camera.cuh"
#include "common.cuh"

namespace uyd {

static thread_local char g_err[512] = "";

void set_error(const char *fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// Registry behind smem_optin (common.cuh): the attribute is per (kernel, device).
int smem_optin_impl(const void *kernel, int bytes) {
  static std::mutex mu;
  static std::set<std::pair<const void *, int>> done;
  int dev = 0;
  UYD_CUDA(cudaGetDevice(&dev));
  std::lock_guard<std::mutex> lock(mu);
  if (done.count({kernel, dev})) return UYD_OK;
  UYD_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
  done.insert({kernel, dev});
  return UYD_OK;
}

int current_sm_count() {
  static int sms[64] = {0};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 0;
  if (!sms[dev]) cudaDeviceGetAttribute(&sms[dev], cudaDevAttrMultiProcessorCount, dev);
  return sms[dev];
}

// conv_tc.cu
struct TcConv;
bool tc_supported(const uyd_conv &d, int in_pitch, int in_coff, int out_pitch, int out_coff, bool in_is_network_input);
size_t tc_weight_bytes(const uyd_conv &d);
void tc_pack_weights(const uyd_conv &d, const float *w, void *dst_host);
int tc_prepare(TcConv *tc, const uyd_conv &d, void *in_base, int in_pitch, int ih, int iw, int max_batch, void *out_base,
               int out_pitch, int out_f32, const void *res_base, int res_pitch, void *w_dev, const float *bias_dev,
               int mode_override, int base_offset_mode, int stages_override, int i8 = 0, const float *mult_dev = nullptr,
               float out_scale = 0.f, int out_kind = 0, int halo_pitch = 10);
bool tc_supported_s8(int cin, int cout, int k, int stride, int in_pitch, int in_coff, int out_pitch, int out_coff, int out_esize,
                     bool pre);
size_t tc_weight_bytes_s8(int cin, int cout, int k);
void tc_pack_weights_s8(int cin, int cout, int k, const int8_t *w, void *dst_host);
int tc_launch(const TcConv *tc, int n0, int nb, int sm_count, cudaStream_t s);
TcConv *tc_new();
void tc_delete(TcConv *);
void tc_set_pre(TcConv *tc, const float *pre);
const char *tc_mode_name(const TcConv *);

// c3k_fused.cu
struct C3kArgs {
  const __nv_bfloat16 *in;
  __nv_bfloat16 *out;
  const uint32_t *wfrag;
  const float *bias;
  int n, h, w, in_pitch, out_pitch, th, tiles_x, tiles_y;
};
bool c3k_supported(int c, int h, int w, int in_pitch, int in_coff, int out_pitch, int out_coff);
void c3k_pack(int c, const float *const w[7], const float *const b[7], std::vector<uint32_t> &frags, std::vector<float> &bias);
void c3k_pack_q(int c, const int8_t *const wq[7], const float *const mult[7], const float *const bias[7], const float in_scale[7],
                std::vector<uint32_t> &frags, std::vector<float> &table);
int c3k_launch_q(int c, const C3kArgs &a, cudaStream_t s);
int c3k_launch(int c, const C3kArgs &a, cudaStream_t s);

struct ClsArgs {
  const __nv_bfloat16 *in;
  float *out;
  const __nv_bfloat16 *wdw;
  const uint32_t *wfrag;
  const float *bias;
  int n, h, w, in_pitch, out_pitch, nc, tiles_x, tiles_y;
};
bool cls_branch_supported(int cin, int mid, int nc, int h, int w, int in_pitch, int in_coff, int out_pitch, int out_coff);
void cls_branch_pack(int cin, int nc, const float *const w[5], const float *const b[5], std::vector<__nv_bfloat16> &wdw,
                     std::vector<uint32_t> &frags, std::vector<float> &bias);
int cls_branch_launch(int cin, const ClsArgs &a, cudaStream_t s);

// conv_chain.cu
struct ChainConv;
ChainConv *chain_new();
void chain_delete(ChainConv *);
bool chain_supported(int cin, int n1, int n2, int in_pitch, int in_coff);
size_t chain_w1_bytes(int cin, int n1, bool depthwise);
size_t chain_w2_bytes(int n1, int n2);
void chain_pack_w1(int cin, int n1, bool depthwise, const float *w, void *dst_host);
void chain_pack_w2(int n1, int n2, const float *w, void *dst_host);
int chain_prepare(ChainConv *cc, int cin, int n1, int n2, void *in_base, int in_pitch, int h, int w, int max_batch,
                  void *w1_dev, void *w2_dev, const float *bias1, const float *bias2, int relu2, int final_kind, int nc,
                  const float *w3_dev, const float *bias3_dev, void *out_base, int out_pitch, int out_f32, int a_total,
                  int a_off, int y_ch0, int no, float stride_px, int dw1);
int chain_launch(const ChainConv *cc, int nb, float *y, int sm_count, cudaStream_t s);

// stem_fused.cu
struct StemArgs {
  const void *in;
  __nv_bfloat16 *out;
  const uint32_t *wfrag;
  const float *bias;
  int n, ih, iw, oh, ow, out_pitch, u8, pw;
  CamFrames f;
};
bool stem_fused_supported(int c0, int c1, int ih, int iw, int out_pitch, int out_coff);
void stem_fused_pack(const float *w0, const float *b0, const float *w1, const float *b1, const float *w2, const float *b2,
                     std::vector<uint32_t> &frags, std::vector<float> &bias);
int stem_fused_launch(const StemArgs &a, cudaStream_t s);

static int env_int(const char *name, int dflt) {
  const char *v = getenv(name);
  return v && *v ? atoi(v) : dflt;
}

}  // namespace uyd

using namespace uyd;

struct uyd_ctx {
  int device = 0;
  int sm_count = 0;
};

enum OpKind { OP_CONV = 0, OP_SPPF = 1, OP_UPSAMPLE = 2, OP_CONV_S8 = 3, OP_C3K = 4, OP_CLS = 5, OP_CHAIN = 6, OP_STEM2 = 7, OP_QUANT = 8 };

struct Op {
  OpKind kind;
  uyd_conv conv{};
  bool use_tc = false;
  std::vector<unsigned char> w_host;  // packed weights (until finalize)
  std::vector<float> b_host;
  void *w_dev = nullptr;
  float *b_dev = nullptr;
  TcConv *tc = nullptr;
  // int8 conv
  std::vector<float> m_host;
  float *m_dev = nullptr;
  float out_scale = 0.f;
  int out_kind = 0;
  std::vector<unsigned char> w2_host;  // cls branch: depth-wise weights
  void *w2_dev = nullptr;
  int nc = 0;
  // chained head kernel
  uyd_chain chain{};
  ChainConv *cc = nullptr;
  std::vector<float> b2_host, w3_host, b3_host;
  float *b2_dev = nullptr, *w3_dev = nullptr, *b3_dev = nullptr;
  bool quant = false;  // OP_C3K: INT8 (fake-quant) variant, b_host = [7][32] bias | [7][32] multiplier | 7 input scales
  // sppf / upsample
  int buf = -1, coff = 0, c = 0, out_buf = -1, out_coff = 0;
};

struct uyd_plan {
  uyd_ctx *ctx = nullptr;
  int max_batch = 0;
  bool finalized = false;
  std::vector<Buffer> bufs;
  std::vector<Op> ops;
  std::vector<int> heads, head_strides;
  int reg_max = 16, nc = 0;
  float dfl_amax = 0.f;                // > 0: the DFL projection runs as a QuantConv2d (uyd_plan_set_dfl_quant)
  int in_c = 0, in_h = 0, in_w = 0;  // network input extent (derived from the first conv)
  size_t bytes = 0;
  void *arena = nullptr;
  float *profile_y = nullptr;          // decoded output used by uyd_plan_profile (uyd_plan_set_profile_output)
  uyd_camera_frames cam{};            // frames of the running uyd_plan_run_camera call (x_kind 3)
  int timed_op = -1, timed_used = 0;  // uyd_plan_set_timed_op
  std::vector<cudaEvent_t> timed_ev;
};

namespace uyd {
int ctx_device(const uyd_ctx *ctx) {
  if (ctx) return ctx->device;
  int d = 0;
  cudaGetDevice(&d);
  return d;
}
}  // namespace uyd

extern "C" int uyd_version(void) { return 100; }
extern "C" const char *uyd_last_error(void) { return g_err; }

extern "C" int uyd_create(int device, uyd_ctx **out) {
  UYD_REQUIRE(out, UYD_E_ARG, "uyd_create: out is NULL");
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  UYD_REQUIRE(e == cudaSuccess && count > 0, UYD_E_NOGPU, "uyd_create: no CUDA device (%s)", cudaGetErrorString(e));
  UYD_REQUIRE(device >= 0 && device < count, UYD_E_ARG, "uyd_create: device %d out of range", device);
  cudaDeviceProp prop;
  UYD_CUDA(cudaGetDeviceProperties(&prop, device));
  UYD_REQUIRE(prop.major == 10, UYD_E_NOGPU, "uyd_create: device %d is sm_%d%d; this library is sm_100a only", device,
              prop.major, prop.minor);
  uyd_ctx *c = new uyd_ctx();
  c->device = device;
  c->sm_count = prop.multiProcessorCount;
  *out = c;
  return UYD_OK;
}

extern "C" int uyd_destroy(uyd_ctx *ctx) {
  delete ctx;
  return UYD_OK;
}

extern "C" int uyd_sm_count(const uyd_ctx *ctx) { return ctx ? ctx->sm_count : 0; }

extern "C" int uyd_plan_create(uyd_ctx *ctx, int max_batch, uyd_plan **out) {
  UYD_REQUIRE(ctx && out && max_batch > 0, UYD_E_ARG, "uyd_plan_create: bad arguments");
  uyd_plan *p = new uyd_plan();
  p->ctx = ctx;
  p->max_batch = max_batch;
  *out = p;
  return UYD_OK;
}

extern "C" int uyd_plan_destroy(uyd_plan *plan) {
  if (!plan) return UYD_OK;
  uyd::DeviceGuard guard(plan->ctx->device);
  for (Op &o : plan->ops) {
    if (o.w_dev) cudaFree(o.w_dev);
    if (o.b_dev) cudaFree(o.b_dev);
    if (o.m_dev) cudaFree(o.m_dev);
    if (o.w2_dev) cudaFree(o.w2_dev);
    if (o.tc) tc_delete(o.tc);
    if (o.cc) chain_delete(o.cc);
    if (o.b2_dev) cudaFree(o.b2_dev);
    if (o.w3_dev) cudaFree(o.w3_dev);
    if (o.b3_dev) cudaFree(o.b3_dev);
  }
  if (plan->arena) cudaFree(plan->arena);
  for (cudaEvent_t e : plan->timed_ev) cudaEventDestroy(e);
  delete plan;
  return UYD_OK;
}

extern "C" int uyd_plan_add_buffer(uyd_plan *plan, int h, int w, int c, int dtype, int *id) {
  UYD_REQUIRE(plan && id && h > 0 && w > 0 && c > 0, UYD_E_ARG, "uyd_plan_add_buffer: bad arguments");
  UYD_REQUIRE(!plan->finalized, UYD_E_STATE, "plan already finalized");
  UYD_REQUIRE(dtype == UYD_BF16 || dtype == UYD_F32 || dtype == UYD_S8, UYD_E_ARG, "unknown dtype %d", dtype);
  Buffer b;
  b.h = h; b.w = w; b.c = c; b.dtype = dtype;
  plan->bufs.push_back(b);
  *id = (int)plan->bufs.size() - 1;
  return UYD_OK;
}

static int check_slice(const uyd_plan *p, int buf, int coff, int c, const char *what) {
  UYD_REQUIRE(buf >= 0 && buf < (int)p->bufs.size(), UYD_E_ARG, "%s: buffer id %d out of range", what, buf);
  UYD_REQUIRE(coff >= 0 && c > 0 && coff + c <= p->bufs[buf].c, UYD_E_ARG, "%s: channel slice [%d,%d) exceeds buffer width %d",
              what, coff, coff + c, p->bufs[buf].c);
  return UYD_OK;
}

extern "C" int uyd_plan_add_conv(uyd_plan *plan, const uyd_conv *d, const float *weight, const float *bias) {
  UYD_REQUIRE(plan && d && weight && bias, UYD_E_ARG, "uyd_plan_add_conv: NULL argument");
  UYD_REQUIRE(!plan->finalized, UYD_E_STATE, "plan already finalized");
  UYD_REQUIRE((d->k == 1 || d->k == 3) && (d->stride == 1 || d->stride == 2), UYD_E_UNSUPPORTED, "conv k=%d s=%d unsupported",
              d->k, d->stride);
  UYD_REQUIRE(!d->depthwise || d->cin == d->cout, UYD_E_ARG, "depthwise conv needs cin == cout");
  int e;
  int ih, iw, in_pitch = 0;
  if (d->in_buf < 0) {
    UYD_REQUIRE(plan->ops.empty(), UYD_E_ARG, "only the first op may read the network input");
    if ((e = check_slice(plan, d->out_buf, d->out_coff, d->cout, "conv output"))) return e;
    const Buffer &ob = plan->bufs[d->out_buf];
    ih = ob.h * d->stride; iw = ob.w * d->stride;
    plan->in_c = d->cin; plan->in_h = ih; plan->in_w = iw;
  } else {
    if ((e = check_slice(plan, d->in_buf, d->in_coff, d->cin, "conv input"))) return e;
    UYD_REQUIRE(plan->bufs[d->in_buf].dtype == UYD_BF16, UYD_E_UNSUPPORTED, "conv input must be bf16");
    ih = plan->bufs[d->in_buf].h; iw = plan->bufs[d->in_buf].w; in_pitch = plan->bufs[d->in_buf].c;
  }
  if ((e = check_slice(plan, d->out_buf, d->out_coff, d->cout, "conv output"))) return e;
  const Buffer &ob = plan->bufs[d->out_buf];
  const int pad = d->k / 2;
  UYD_REQUIRE(ob.h == (ih + 2 * pad - d->k) / d->stride + 1 && ob.w == (iw + 2 * pad - d->k) / d->stride + 1, UYD_E_ARG,
              "conv output buffer is %dx%d but the conv produces %dx%d", ob.h, ob.w, (ih + 2 * pad - d->k) / d->stride + 1,
              (iw + 2 * pad - d->k) / d->stride + 1);
  UYD_REQUIRE(ob.dtype == UYD_BF16 || ob.dtype == UYD_F32, UYD_E_UNSUPPORTED, "conv output must be bf16 or fp32");
  if (d->res_buf >= 0) {
    if ((e = check_slice(plan, d->res_buf, d->res_coff, d->cout, "conv residual"))) return e;
    UYD_REQUIRE(plan->bufs[d->res_buf].h == ob.h && plan->bufs[d->res_buf].w == ob.w && plan->bufs[d->res_buf].dtype == UYD_BF16,
                UYD_E_ARG, "residual slice must match the output extent (bf16)");
  }
  if (d->pre_buf_p1) {
    const int pb = d->pre_buf_p1 - 1;
    UYD_REQUIRE(pb >= 0 && pb < (int)plan->bufs.size(), UYD_E_ARG, "conv: partial-sum buffer id out of range");
    const Buffer &b = plan->bufs[pb];
    UYD_REQUIRE(b.dtype == UYD_F32 && b.c == d->cout && b.h * 2 == ob.h && b.w * 2 == ob.w && d->cout % 16 == 0, UYD_E_ARG,
                "conv: the partial-sum buffer must be fp32 [h/2, w/2, cout]");
  }
  Op op;
  op.kind = OP_CONV;
  op.conv = *d;
  const bool f32 = ob.dtype == UYD_F32;
  bool tc_ok = tc_supported(*d, in_pitch, d->in_coff, ob.c, d->out_coff, d->in_buf < 0);
  if (tc_ok && !f32 && d->cout >= 16 && (ob.c % 8 || d->out_coff % 8)) tc_ok = false;
  if (tc_ok && d->res_buf >= 0 && (plan->bufs[d->res_buf].c % 8 || d->res_coff % 8)) tc_ok = false;
  const int min_c = env_int("UYD_TC_MIN_CIN", 16);
  if (d->impl == UYD_IMPL_TC) {
    UYD_REQUIRE(tc_ok, UYD_E_UNSUPPORTED, "conv %d->%d k%d s%d cannot run on the tensor-core path", d->cin, d->cout, d->k, d->stride);
    op.use_tc = true;
  } else if (d->impl == UYD_IMPL_AUTO) {
    op.use_tc = tc_ok && d->cin >= min_c && env_int("UYD_DISABLE_TC", 0) == 0;
  }
  UYD_REQUIRE(!d->pre_buf_p1 || op.use_tc, UYD_E_UNSUPPORTED, "conv: partial sums are only added on the tensor-core path");
  if (op.use_tc) {
    op.w_host.resize(tc_weight_bytes(*d));
    tc_pack_weights(*d, weight, op.w_host.data());
  } else {
    op.w_host.resize(direct_weight_bytes(*d));
    direct_pack_weights(*d, weight, op.w_host.data());
  }
  op.b_host.assign(bias, bias + d->cout);
  plan->ops.push_back(std::move(op));
  return UYD_OK;
}

extern "C" int uyd_plan_add_conv_s8(uyd_plan *plan, const uyd_conv_s8 *d, const int8_t *weight_q, const float *mult,
                                    const float *bias) {
  UYD_REQUIRE(plan && d && weight_q && mult && bias, UYD_E_ARG, "uyd_plan_add_conv_s8: NULL argument");
  UYD_REQUIRE(!plan->finalized, UYD_E_STATE, "plan already finalized");
  UYD_REQUIRE((d->k == 1 || d->k == 3) && (d->stride == 1 || d->stride == 2), UYD_E_UNSUPPORTED, "conv k=%d s=%d unsupported",
              d->k, d->stride);
  int e;
  if ((e = check_slice(plan, d->in_buf, d->in_coff, d->cin, "conv_s8 input"))) return e;
  if ((e = check_slice(plan, d->out_buf, d->out_coff, d->cout, "conv_s8 output"))) return e;
  const Buffer &ib = plan->bufs[d->in_buf], &ob = plan->bufs[d->out_buf];
  UYD_REQUIRE(ib.dtype == UYD_S8, UYD_E_ARG, "conv_s8 input buffer must be UYD_S8");
  const int pad = d->k / 2;
  UYD_REQUIRE(ob.h == (ib.h + 2 * pad - d->k) / d->stride + 1 && ob.w == (ib.w + 2 * pad - d->k) / d->stride + 1, UYD_E_ARG,
              "conv_s8 output extent mismatch");
  UYD_REQUIRE(ob.dtype != UYD_S8 || d->out_scale > 0.f, UYD_E_ARG, "conv_s8: int8 output needs out_scale > 0");
  Op op;
  op.kind = OP_CONV_S8;
  op.conv.in_buf = d->in_buf; op.conv.in_coff = d->in_coff; op.conv.out_buf = d->out_buf; op.conv.out_coff = d->out_coff;
  op.conv.res_buf = d->res_buf; op.conv.res_coff = d->res_coff; op.conv.depthwise = d->depthwise;
  op.conv.cin = d->cin; op.conv.cout = d->cout; op.conv.k = d->k; op.conv.stride = d->stride;
  op.conv.relu = d->relu;
  UYD_REQUIRE(!d->depthwise || (d->cin == d->cout && d->res_buf < 0), UYD_E_ARG, "conv_s8: depth-wise needs cin == cout, no residual");
  if (d->res_buf >= 0) {
    if ((e = check_slice(plan, d->res_buf, d->res_coff, d->cout, "conv_s8 residual"))) return e;
    const Buffer &rb = plan->bufs[d->res_buf];
    UYD_REQUIRE(rb.h == ob.h && rb.w == ob.w && rb.dtype == UYD_BF16, UYD_E_ARG, "conv_s8 residual must match the output extent (bf16)");
  }
  if (d->pre_buf_p1) {
    const int pb = d->pre_buf_p1 - 1;
    UYD_REQUIRE(pb >= 0 && pb < (int)plan->bufs.size(), UYD_E_ARG, "conv_s8: partial-sum buffer id out of range");
    const Buffer &b = plan->bufs[pb];
    UYD_REQUIRE(b.dtype == UYD_F32 && b.c == d->cout && b.h * 2 == ob.h && b.w * 2 == ob.w && d->cout % 16 == 0 && d->k == 1 &&
                    d->stride == 1 && d->res_buf < 0,
                UYD_E_ARG, "conv_s8: partial sums need an fp32 [h/2, w/2, cout] buffer, a 1x1 conv, cout %% 16 == 0, no residual");
    op.conv.pre_buf_p1 = d->pre_buf_p1;
  }
  op.out_scale = d->out_scale;
  op.out_kind = ob.dtype == UYD_S8 ? (d->out_round_bf16 ? 3 : 2) : (ob.dtype == UYD_F32 ? 1 : 0);
  bool tc_ok = !d->depthwise && tc_supported_s8(d->cin, d->cout, d->k, d->stride, ib.c, d->in_coff, ob.c, d->out_coff, (int)ob.elem_bytes(),
                                             d->pre_buf_p1 != 0);
  if (d->impl == UYD_IMPL_TC) {
    UYD_REQUIRE(tc_ok, UYD_E_UNSUPPORTED, "conv_s8 %d->%d k%d s%d cannot run on the tensor-core path", d->cin, d->cout, d->k, d->stride);
    op.use_tc = true;
  } else if (d->impl == UYD_IMPL_AUTO) {
    op.use_tc = tc_ok;
  }
  UYD_REQUIRE(!d->pre_buf_p1 || op.use_tc, UYD_E_UNSUPPORTED, "conv_s8: partial sums are only added on the tensor-core path");
  if (op.use_tc) {
    op.w_host.resize(tc_weight_bytes_s8(d->cin, d->cout, d->k));
    tc_pack_weights_s8(d->cin, d->cout, d->k, weight_q, op.w_host.data());
  } else if (d->depthwise) {
    op.w_host.resize((size_t)d->cin * d->k * d->k);
    direct_pack_weights_s8_dw(d->cin, d->k, weight_q, op.w_host.data());
  } else {
    op.w_host.resize(direct_weight_bytes_s8(d->cin, d->cout, d->k));
    direct_pack_weights_s8(d->cin, d->cout, d->k, weight_q, op.w_host.data());
  }
  op.b_host.assign(bias, bias + d->cout);
  op.m_host.assign(mult, mult + d->cout);
  plan->ops.push_back(std::move(op));
  return UYD_OK;
}

extern "C" int uyd_plan_add_c3k(uyd_plan *plan, const uyd_c3k *d, const float *const weights[7], const float *const biases[7]) {
  UYD_REQUIRE(plan && d && weights && biases, UYD_E_ARG, "uyd_plan_add_c3k: NULL argument");
  UYD_REQUIRE(!plan->finalized, UYD_E_STATE, "plan already finalized");
  int e;
  if ((e = check_slice(plan, d->in_buf, d->in_coff, d->c, "c3k input"))) return e;
  if ((e = check_slice(plan, d->out_buf, d->out_coff, d->c, "c3k output"))) return e;
  const Buffer &ib = plan->bufs[d->in_buf], &ob = plan->bufs[d->out_buf];
  UYD_REQUIRE(ib.dtype == UYD_BF16 && ob.dtype == UYD_BF16 && ib.h == ob.h && ib.w == ob.w, UYD_E_ARG,
              "c3k needs bf16 buffers of equal extent");
  UYD_REQUIRE(c3k_supported(d->c, ib.h, ib.w, ib.c, d->in_coff, ob.c, d->out_coff), UYD_E_UNSUPPORTED,
              "fused c3k: c=%d %dx%d is not supported (c in {8,16,32}, W %% 40 == 0, H %% 32|20|16 == 0, 16-byte slices)",
              d->c, ib.h, ib.w);
  for (int i = 0; i < 7; ++i) UYD_REQUIRE(weights[i] && biases[i], UYD_E_ARG, "uyd_plan_add_c3k: weight %d is NULL", i);
  Op op;
  op.kind = OP_C3K;
  op.buf = d->in_buf; op.coff = d->in_coff; op.out_buf = d->out_buf; op.out_coff = d->out_coff; op.c = d->c;
  std::vector<uint32_t> frags;
  c3k_pack(d->c, weights, biases, frags, op.b_host);
  op.w_host.resize(frags.size() * 4);
  memcpy(op.w_host.data(), frags.data(), op.w_host.size());
  plan->ops.push_back(std::move(op));
  return UYD_OK;
}

extern "C" int uyd_plan_add_c3k_s8(uyd_plan *plan, const uyd_c3k *d, const int8_t *const weights[7], const float *const mult[7],
                                   const float *const biases[7], const float *in_scale) {
  UYD_REQUIRE(plan && d && weights && mult && biases && in_scale, UYD_E_ARG, "uyd_plan_add_c3k_s8: NULL argument");
  UYD_REQUIRE(!plan->finalized, UYD_E_STATE, "plan already finalized");
  int e;
  if ((e = check_slice(plan, d->in_buf, d->in_coff, d->c, "c3k input"))) return e;
  if ((e = check_slice(plan, d->out_buf, d->out_coff, d->c, "c3k output"))) return e;
  const Buffer &ib = plan->bufs[d->in_buf], &ob = plan->bufs[d->out_buf];
  UYD_REQUIRE(ib.dtype == UYD_BF16 && ob.dtype == UYD_BF16 && ib.h == ob.h && ib.w == ob.w, UYD_E_ARG,
              "int8 c3k needs bf16 buffers of equal extent (the block quantises its input itself)");
  UYD_REQUIRE(c3k_supported(d->c, ib.h, ib.w, ib.c, d->in_coff, ob.c, d->out_coff), UYD_E_UNSUPPORTED,
              "fused int8 c3k: c=%d %dx%d is not supported (c in {8,16,32}, W %% 40 == 0, H %% 32|20|16 == 0, 16-byte slices)",
              d->c, ib.h, ib.w);
  for (int i = 0; i < 7; ++i)
    UYD_REQUIRE(weights[i] && mult[i] && biases[i], UYD_E_ARG, "uyd_plan_add_c3k_s8: array %d is NULL", i);
  Op op;
  op.kind = OP_C3K;
  op.quant = true;
  op.buf = d->in_buf; op.coff = d->in_coff; op.out_buf = d->out_buf; op.out_coff = d->out_coff; op.c = d->c;
  std::vector<uint32_t> frags;
  c3k_pack_q(d->c, weights, mult, biases, in_scale, frags, op.b_host);
  op.w_host.resize(frags.size() * 4);
  memcpy(op.w_host.data(), frags.data(), op.w_host.size());
  plan->ops.push_back(std::move(op));
  return UYD_OK;
}

extern "C" int uyd_plan_add_cls_branch(uyd_plan *plan, const uyd_cls_branch *d, const float *const weights[5],
                                       const float *const biases[5]) {
  UYD_REQUIRE(plan && d && weights && biases, UYD_E_ARG, "uyd_plan_add_cls_branch: NULL argument");
  UYD_REQUIRE(!plan->finalized, UYD_E_STATE, "plan already finalized");
  int e;
  if ((e = check_slice(plan, d->in_buf, d->in_coff, d->cin, "cls branch input"))) return e;
  if ((e = check_slice(plan, d->out_buf, d->out_coff, d->nc, "cls branch output"))) return e;
  const Buffer &ib = plan->bufs[d->in_buf], &ob = plan->bufs[d->out_buf];
  UYD_REQUIRE(ib.dtype == UYD_BF16 && ob.dtype == UYD_F32 && ib.h == ob.h && ib.w == ob.w, UYD_E_ARG,
              "cls branch: bf16 input and fp32 output of equal extent");
  UYD_REQUIRE(cls_branch_supported(d->cin, d->mid, d->nc, ib.h, ib.w, ib.c, d->in_coff, ob.c, d->out_coff), UYD_E_UNSUPPORTED,
              "fused cls branch: cin=%d mid=%d nc=%d %dx%d unsupported (cin in {32,64}, mid 32, nc <= 8, W %% 40, H %% 8)",
              d->cin, d->mid, d->nc, ib.h, ib.w);
  for (int i = 0; i < 5; ++i) UYD_REQUIRE(weights[i] && biases[i], UYD_E_ARG, "uyd_plan_add_cls_branch: weight %d is NULL", i);
  Op op;
  op.kind = OP_CLS;
  op.buf = d->in_buf; op.coff = d->in_coff; op.out_buf = d->out_buf; op.out_coff = d->out_coff; op.c = d->cin; op.nc = d->nc;
  std::vector<__nv_bfloat16> wdw;
  std::vector<uint32_t> frags;
  cls_branch_pack(d->cin, d->nc, weights, biases, wdw, frags, op.b_host);
  op.w_host.resize(frags.size() * 4);
  memcpy(op.w_host.data(), frags.data(), op.w_host.size());
  op.w2_host.resize(wdw.size() * 2);
  memcpy(op.w2_host.data(), wdw.data(), op.w2_host.size());
  plan->ops.push_back(std::move(op));
  return UYD_OK;
}

extern "C" int uyd_plan_add_chain(uyd_plan *plan, const uyd_chain *d, const float *w1, const float *b1, const float *w2,
                                  const float *b2, const float *w3, const float *b3) {
  UYD_REQUIRE(plan && d && w1 && b1 && w2 && b2, UYD_E_ARG, "uyd_plan_add_chain: NULL argument");
  UYD_REQUIRE(!plan->finalized, UYD_E_STATE, "plan already finalized");
  int e;
  if ((e = check_slice(plan, d->in_buf, d->in_coff, d->cin, "chain input"))) return e;
  const Buffer &ib = plan->bufs[d->in_buf];
  UYD_REQUIRE(ib.dtype == UYD_BF16, UYD_E_ARG, "chain input must be bf16");
  UYD_REQUIRE(chain_supported(d->cin, d->n1, d->n2, ib.c, d->in_coff), UYD_E_UNSUPPORTED,
              "chain %d -> %d -> %d unsupported (cin, n1 in {32, 64}; n2 <= 64; 16-byte aligned input slice)", d->cin, d->n1, d->n2);
  UYD_REQUIRE(!d->dw1 || d->cin == d->n1, UYD_E_ARG, "chain: a depth-wise first conv needs cin == n1");
  UYD_REQUIRE(d->final_kind == UYD_CHAIN_STORE || d->final_kind == UYD_CHAIN_PW3 || d->final_kind == UYD_CHAIN_DFL, UYD_E_ARG,
              "chain: unknown final stage %d", d->final_kind);
  if (d->out_buf >= 0) {
    const int oc = d->final_kind == UYD_CHAIN_PW3 ? d->nc : d->n2;
    if ((e = check_slice(plan, d->out_buf, d->out_coff, oc, "chain output"))) return e;
    const Buffer &ob = plan->bufs[d->out_buf];
    UYD_REQUIRE(ob.h == ib.h && ob.w == ib.w, UYD_E_ARG, "chain output extent differs from the input");
    if (d->final_kind == UYD_CHAIN_STORE)
      UYD_REQUIRE(d->n2 % 16 == 0 && (ob.c * ob.elem_bytes()) % 16 == 0 && (d->out_coff * ob.elem_bytes()) % 16 == 0 &&
                      (ob.dtype == UYD_BF16 || ob.dtype == UYD_F32), UYD_E_UNSUPPORTED, "chain STORE needs n2 %% 16 == 0 and 16-byte rows");
    else
      UYD_REQUIRE(ob.dtype == UYD_F32 && (d->final_kind == UYD_CHAIN_PW3 || ((ob.c % 4) == 0 && (d->out_coff % 4) == 0)),
                  UYD_E_UNSUPPORTED, "chain PW3 / DFL raw output goes to an fp32 head buffer");
  } else {
    UYD_REQUIRE(d->final_kind != UYD_CHAIN_STORE, UYD_E_ARG, "chain STORE needs an output slice");
  }
  if (d->final_kind == UYD_CHAIN_PW3) UYD_REQUIRE(w3 && b3 && d->nc >= 1 && d->nc <= 8 && d->n2 <= 64, UYD_E_ARG, "chain PW3: w3/b3, nc <= 8");
  if (d->final_kind == UYD_CHAIN_DFL) UYD_REQUIRE(d->n2 == 64, UYD_E_ARG, "chain DFL: n2 must be 4 x 16");
  Op op;
  op.kind = OP_CHAIN;
  op.chain = *d;
  op.w_host.resize(chain_w1_bytes(d->cin, d->n1, d->dw1 != 0));
  chain_pack_w1(d->cin, d->n1, d->dw1 != 0, w1, op.w_host.data());
  op.w2_host.resize(chain_w2_bytes(d->n1, d->n2));
  chain_pack_w2(d->n1, d->n2, w2, op.w2_host.data());
  const int N2 = (d->n2 + 15) / 16 * 16;
  op.b_host.assign(b1, b1 + d->n1);
  op.b2_host.assign(N2, 0.f);
  for (int i = 0; i < d->n2; ++i) op.b2_host[i] = b2[i];
  if (d->final_kind == UYD_CHAIN_PW3) {
    op.w3_host.assign((size_t)d->nc * N2, 0.f);
    for (int c = 0; c < d->nc; ++c)
      for (int k = 0; k < d->n2; ++k) op.w3_host[(size_t)c * N2 + k] = __bfloat162float(__float2bfloat16_rn(w3[(size_t)c * d->n2 + k]));
    op.b3_host.assign(b3, b3 + d->nc);
  }
  plan->ops.push_back(std::move(op));
  return UYD_OK;
}

static int add_stem(uyd_plan *plan, int out_buf, int out_coff, const float *w0, const float *b0, const float *w1, const float *b1,
                    const float *w2, const float *b2) {
  UYD_REQUIRE(plan && w0 && b0 && w1 && b1, UYD_E_ARG, "uyd_plan_add_stem2: NULL argument");
  UYD_REQUIRE(!plan->finalized, UYD_E_STATE, "plan already finalized");
  UYD_REQUIRE(plan->ops.empty(), UYD_E_ARG, "only the first op may read the network input");
  const int cout = w2 ? 16 : 32;
  int e;
  if ((e = check_slice(plan, out_buf, out_coff, cout, "stem2 output"))) return e;
  const Buffer &ob = plan->bufs[out_buf];
  UYD_REQUIRE(ob.dtype == UYD_BF16 && stem_fused_supported(16, 32, ob.h * 4, ob.w * 4, w2 ? 2 * ob.c : ob.c, w2 ? 2 * out_coff : out_coff),
              UYD_E_UNSUPPORTED, "stem2: bf16 output slice, 16-byte aligned (8-byte with the 1x1 folded in)");
  plan->in_c = 3; plan->in_h = ob.h * 4; plan->in_w = ob.w * 4;
  Op op;
  op.kind = OP_STEM2;
  op.out_buf = out_buf; op.out_coff = out_coff; op.c = w2 ? 1 : 0;
  std::vector<uint32_t> frags;
  stem_fused_pack(w0, b0, w1, b1, w2, b2, frags, op.b_host);
  op.w_host.resize(frags.size() * 4);
  memcpy(op.w_host.data(), frags.data(), op.w_host.size());
  plan->ops.push_back(std::move(op));
  return UYD_OK;
}

extern "C" int uyd_plan_add_stem2(uyd_plan *plan, int out_buf, int out_coff, const float *w0, const float *b0, const float *w1,
                                  const float *b1) {
  return add_stem(plan, out_buf, out_coff, w0, b0, w1, b1, nullptr, nullptr);
}

extern "C" int uyd_plan_add_stem2_pw(uyd_plan *plan, int out_buf, int out_coff, const float *w0, const float *b0, const float *w1,
                                     const float *b1, const float *w2, const float *b2) {
  UYD_REQUIRE(w2 && b2, UYD_E_ARG, "uyd_plan_add_stem2_pw: NULL argument");
  return add_stem(plan, out_buf, out_coff, w0, b0, w1, b1, w2, b2);
}

extern "C" int uyd_plan_add_quantize(uyd_plan *plan, int in_buf, int in_coff, int out_buf, int out_coff, int c, float scale) {
  UYD_REQUIRE(plan && !plan->finalized, UYD_E_STATE, "plan missing or finalized");
  int e;
  if ((e = check_slice(plan, in_buf, in_coff, c, "quantize input"))) return e;
  if ((e = check_slice(plan, out_buf, out_coff, c, "quantize output"))) return e;
  const Buffer &a = plan->bufs[in_buf], &b = plan->bufs[out_buf];
  UYD_REQUIRE(a.dtype == UYD_BF16 && b.dtype == UYD_S8 && a.h == b.h && a.w == b.w, UYD_E_ARG, "quantize: bf16 -> int8 buffers of equal extent");
  UYD_REQUIRE(c % 4 == 0 && a.c % 4 == 0 && in_coff % 4 == 0 && b.c % 4 == 0 && out_coff % 4 == 0 && scale > 0.f, UYD_E_UNSUPPORTED,
              "quantize: channel counts / offsets must be multiples of 4 and scale positive");
  Op op;
  op.kind = OP_QUANT;
  op.buf = in_buf; op.coff = in_coff; op.c = c; op.out_buf = out_buf; op.out_coff = out_coff; op.out_scale = scale;
  plan->ops.push_back(std::move(op));
  return UYD_OK;
}

extern "C" int uyd_plan_slice_absmax(uyd_plan *plan, int buf, int coff, int c, int batch, unsigned int *d_bits, uyd_stream stream) {
  UYD_REQUIRE(plan && plan->finalized && d_bits, UYD_E_STATE, "uyd_plan_slice_absmax: plan not finalized / NULL output");
  int e;
  if ((e = check_slice(plan, buf, coff, c, "absmax"))) return e;
  const Buffer &b = plan->bufs[buf];
  UYD_REQUIRE(b.dtype == UYD_BF16 && batch > 0 && batch <= plan->max_batch, UYD_E_ARG, "absmax: bf16 slice, batch within the plan");
  uyd::DeviceGuard guard(plan->ctx->device);
  return absmax_launch((const __nv_bfloat16 *)((char *)b.ptr + (size_t)coff * 2), b.c, (long long)batch * b.h * b.w, c, d_bits,
                       (cudaStream_t)stream);
}

extern "C" int uyd_plan_slice_histogram(uyd_plan *plan, int buf, int coff, int c, int batch, float inv_width, int nbins,
                                        unsigned int *d_hist, uyd_stream stream) {
  UYD_REQUIRE(plan && plan->finalized && d_hist, UYD_E_STATE, "uyd_plan_slice_histogram: plan not finalized / NULL output");
  int e;
  if ((e = check_slice(plan, buf, coff, c, "histogram"))) return e;
  const Buffer &b = plan->bufs[buf];
  UYD_REQUIRE(b.dtype == UYD_BF16 && batch > 0 && batch <= plan->max_batch, UYD_E_ARG, "histogram: bf16 slice, batch within the plan");
  uyd::DeviceGuard guard(plan->ctx->device);
  return abs_histogram_launch((const __nv_bfloat16 *)((char *)b.ptr + (size_t)coff * 2), b.c, (long long)batch * b.h * b.w, c, inv_width,
                              nbins, d_hist, (cudaStream_t)stream);
}

extern "C" int uyd_plan_add_sppf_pool(uyd_plan *plan, int buf, int coff, int c) {
  UYD_REQUIRE(plan && !plan->finalized, UYD_E_STATE, "plan missing or finalized");
  int e;
  if ((e = check_slice(plan, buf, coff, 4 * c, "sppf"))) return e;
  UYD_REQUIRE(plan->bufs[buf].dtype == UYD_BF16, UYD_E_UNSUPPORTED, "sppf works on bf16");
  Op op;
  op.kind = OP_SPPF;
  op.buf = buf; op.coff = coff; op.c = c;
  plan->ops.push_back(std::move(op));
  return UYD_OK;
}

extern "C" int uyd_plan_add_upsample2x(uyd_plan *plan, int in_buf, int in_coff, int out_buf, int out_coff, int c) {
  UYD_REQUIRE(plan && !plan->finalized, UYD_E_STATE, "plan missing or finalized");
  int e;
  if ((e = check_slice(plan, in_buf, in_coff, c, "upsample input"))) return e;
  if ((e = check_slice(plan, out_buf, out_coff, c, "upsample output"))) return e;
  const Buffer &a = plan->bufs[in_buf], &b = plan->bufs[out_buf];
  UYD_REQUIRE(b.h == 2 * a.h && b.w == 2 * a.w && a.dtype == UYD_BF16 && b.dtype == UYD_BF16, UYD_E_ARG,
              "upsample output must be 2x the input extent (bf16)");
  Op op;
  op.kind = OP_UPSAMPLE;
  op.buf = in_buf; op.coff = in_coff; op.c = c; op.out_buf = out_buf; op.out_coff = out_coff;
  plan->ops.push_back(std::move(op));
  return UYD_OK;
}

extern "C" int uyd_plan_set_heads(uyd_plan *plan, const int *head_bufs, const int *strides, int nl, int reg_max, int nc) {
  UYD_REQUIRE(plan && head_bufs && strides && nl > 0 && nl <= 8, UYD_E_ARG, "uyd_plan_set_heads: bad arguments");
  for (int i = 0; i < nl; ++i) {
    UYD_REQUIRE(head_bufs[i] >= 0 && head_bufs[i] < (int)plan->bufs.size(), UYD_E_ARG, "head buffer id out of range");
    const Buffer &b = plan->bufs[head_bufs[i]];
    UYD_REQUIRE(b.dtype == UYD_F32 && b.c == 4 * reg_max + nc, UYD_E_ARG, "head buffer %d must be fp32 with %d channels", i,
                4 * reg_max + nc);
  }
  plan->heads.assign(head_bufs, head_bufs + nl);
  plan->head_strides.assign(strides, strides + nl);
  plan->reg_max = reg_max;
  plan->nc = nc;
  return UYD_OK;
}

static void *slice_ptr(const uyd_plan *p, int buf, int coff) {
  const Buffer &b = p->bufs[buf];
  return (char *)b.ptr + (size_t)coff * b.elem_bytes();
}

extern "C" int uyd_plan_finalize(uyd_plan *plan) {
  UYD_REQUIRE(plan && !plan->finalized, UYD_E_STATE, "plan missing or already finalized");
  UYD_REQUIRE(!plan->arena, UYD_E_STATE, "uyd_plan_finalize failed before on this plan: destroy it (uyd_plan_destroy frees the partial allocations)");
  uyd::DeviceGuard guard(plan->ctx->device);
  UYD_CUDA(guard.err);
  size_t total = 0;
  std::vector<size_t> offs;
  for (Buffer &b : plan->bufs) {
    offs.push_back(total);
    total += (b.bytes_per_image() * plan->max_batch + 1023) & ~(size_t)1023;
  }
  UYD_CUDA(cudaMalloc(&plan->arena, total ? total : 1024));
  UYD_CUDA(cudaMemset(plan->arena, 0, total ? total : 1024));
  for (size_t i = 0; i < plan->bufs.size(); ++i) plan->bufs[i].ptr = (char *)plan->arena + offs[i];
  plan->bytes = total;
  const int halo_fallback = env_int("UYD_TC_NO_HALO", 0);
  // Measured on B200 (profiles/r01_probe.md): the UMMA swizzle XOR is a function of the absolute
  // shared-memory address, so tap-shifted HALO descriptors need base_offset = 0 (mode 1, the
  // "(addr >> 7) & 7" reading of the PTX text, produces wrong results and is kept as a probe).
  const int bo_mode = env_int("UYD_TC_BASE_OFFSET", 0);
  const int stages = env_int("UYD_TC_STAGES", 0);
  const int halo_pitch = env_int("UYD_TC_HALO_PITCH", 10);
  for (Op &o : plan->ops) {
    if (o.kind != OP_CONV && o.kind != OP_CONV_S8 && o.kind != OP_C3K && o.kind != OP_CLS && o.kind != OP_CHAIN && o.kind != OP_STEM2) continue;
    UYD_CUDA(cudaMalloc(&o.w_dev, o.w_host.size()));
    UYD_CUDA(cudaMemcpy(o.w_dev, o.w_host.data(), o.w_host.size(), cudaMemcpyHostToDevice));
    UYD_CUDA(cudaMalloc((void **)&o.b_dev, o.b_host.size() * 4));
    UYD_CUDA(cudaMemcpy(o.b_dev, o.b_host.data(), o.b_host.size() * 4, cudaMemcpyHostToDevice));
    plan->bytes += o.w_host.size() + o.b_host.size() * 4;
    o.w_host.clear();
    o.w_host.shrink_to_fit();
    if (o.kind == OP_CLS) {
      UYD_CUDA(cudaMalloc(&o.w2_dev, o.w2_host.size()));
      UYD_CUDA(cudaMemcpy(o.w2_dev, o.w2_host.data(), o.w2_host.size(), cudaMemcpyHostToDevice));
      continue;
    }
    if (o.kind == OP_CHAIN) {
      const uyd_chain &d = o.chain;
      UYD_CUDA(cudaMalloc(&o.w2_dev, o.w2_host.size()));
      UYD_CUDA(cudaMemcpy(o.w2_dev, o.w2_host.data(), o.w2_host.size(), cudaMemcpyHostToDevice));
      UYD_CUDA(cudaMalloc((void **)&o.b2_dev, o.b2_host.size() * 4));
      UYD_CUDA(cudaMemcpy(o.b2_dev, o.b2_host.data(), o.b2_host.size() * 4, cudaMemcpyHostToDevice));
      if (!o.w3_host.empty()) {
        UYD_CUDA(cudaMalloc((void **)&o.w3_dev, o.w3_host.size() * 4));
        UYD_CUDA(cudaMemcpy(o.w3_dev, o.w3_host.data(), o.w3_host.size() * 4, cudaMemcpyHostToDevice));
        UYD_CUDA(cudaMalloc((void **)&o.b3_dev, o.b3_host.size() * 4));
        UYD_CUDA(cudaMemcpy(o.b3_dev, o.b3_host.data(), o.b3_host.size() * 4, cudaMemcpyHostToDevice));
      }
      const Buffer &ib = plan->bufs[d.in_buf];
      void *out = nullptr;
      int out_pitch = 0, out_f32 = 0;
      if (d.out_buf >= 0) {
        out = slice_ptr(plan, d.out_buf, d.out_coff);
        out_pitch = plan->bufs[d.out_buf].c;
        out_f32 = plan->bufs[d.out_buf].dtype == UYD_F32;
      }
      o.cc = chain_new();
      int e = chain_prepare(o.cc, d.cin, d.n1, d.n2, slice_ptr(plan, d.in_buf, d.in_coff), ib.c, ib.h, ib.w, plan->max_batch, o.w_dev,
                            o.w2_dev, o.b_dev, o.b2_dev, d.relu2, d.final_kind, d.nc, o.w3_dev, o.b3_dev, out, out_pitch, out_f32,
                            d.a_total, d.a_off, d.y_ch0, d.no, d.stride_px, d.dw1);
      if (e) return e;
      continue;
    }
    if (o.kind == OP_C3K || o.kind == OP_STEM2) continue;
    if (o.kind == OP_CONV_S8) {
      UYD_CUDA(cudaMalloc((void **)&o.m_dev, o.m_host.size() * 4));
      UYD_CUDA(cudaMemcpy(o.m_dev, o.m_host.data(), o.m_host.size() * 4, cudaMemcpyHostToDevice));
      if (o.use_tc) {
        const uyd_conv &d = o.conv;
        const Buffer &ib = plan->bufs[d.in_buf], &ob = plan->bufs[d.out_buf];
        o.tc = tc_new();
        const void *res = d.res_buf >= 0 ? slice_ptr(plan, d.res_buf, d.res_coff) : nullptr;
        int e = tc_prepare(o.tc, d, slice_ptr(plan, d.in_buf, d.in_coff), ib.c, ib.h, ib.w, plan->max_batch,
                           slice_ptr(plan, d.out_buf, d.out_coff), ob.c, 0, res, d.res_buf >= 0 ? plan->bufs[d.res_buf].c : 0, o.w_dev,
                           o.b_dev, halo_fallback ? 2 : -1, bo_mode, stages, 1, o.m_dev, o.out_scale, o.out_kind, halo_pitch);
        if (e) return e;
        if (d.pre_buf_p1) tc_set_pre(o.tc, (const float *)plan->bufs[d.pre_buf_p1 - 1].ptr);
      }
      continue;
    }
    if (o.use_tc) {
      const uyd_conv &d = o.conv;
      const Buffer &ib = plan->bufs[d.in_buf], &ob = plan->bufs[d.out_buf];
      o.tc = tc_new();
      const void *res = d.res_buf >= 0 ? slice_ptr(plan, d.res_buf, d.res_coff) : nullptr;
      int e = tc_prepare(o.tc, d, slice_ptr(plan, d.in_buf, d.in_coff), ib.c, ib.h, ib.w, plan->max_batch,
                         slice_ptr(plan, d.out_buf, d.out_coff), ob.c, ob.dtype == UYD_F32, res,
                         d.res_buf >= 0 ? plan->bufs[d.res_buf].c : 0, o.w_dev, o.b_dev, halo_fallback ? 2 : -1, bo_mode, stages, 0,
                         nullptr, 0.f, 0, halo_pitch);
      if (e) return e;
      if (d.pre_buf_p1) tc_set_pre(o.tc, (const float *)plan->bufs[d.pre_buf_p1 - 1].ptr);
    }
  }
  plan->finalized = true;
  return UYD_OK;
}

extern "C" size_t uyd_plan_bytes(const uyd_plan *plan) { return plan ? plan->bytes : 0; }
extern "C" int uyd_plan_num_launches(const uyd_plan *plan) { return plan ? (int)plan->ops.size() : 0; }

extern "C" int uyd_plan_buffer_ptr(uyd_plan *plan, int id, void **ptr) {
  UYD_REQUIRE(plan && ptr && plan->finalized, UYD_E_STATE, "plan not finalized");
  UYD_REQUIRE(id >= 0 && id < (int)plan->bufs.size(), UYD_E_ARG, "buffer id %d out of range", id);
  *ptr = plan->bufs[id].ptr;
  return UYD_OK;
}

// the frames of a uyd_plan_run_camera call as the stem kernels read them
static CamFrames cam_frames(const uyd_camera_frames &c) {
  CamFrames f{};
  f.cam = c.format; f.src_w = c.width; f.src_h = c.height; f.src_pitch = c.pitch; f.uv_pitch = c.uv_pitch;
  f.frame_stride = c.frame_stride; f.uv_frame_stride = c.uv_frame_stride; f.uv = c.uv;
  f.mean[0] = c.norm.mean_r; f.mean[1] = c.norm.mean_g; f.mean[2] = c.norm.mean_b;
  f.stdv[0] = c.norm.std_r; f.stdv[1] = c.norm.std_g; f.stdv[2] = c.norm.std_b;
  return f;
}

// arguments of a CUDA-core OP_CONV (in_buf < 0: the network input x of kind x_kind)
static ConvArgs direct_conv_args(uyd_plan *plan, const uyd_conv &d, const void *x, int x_kind, int batch, const Op &o) {
  const Buffer &ob = plan->bufs[d.out_buf];
  ConvArgs a{};
  a.n = batch;
  if (d.in_buf < 0) {
    a.in = x; a.ih = plan->in_h; a.iw = plan->in_w; a.in_pitch = 0; a.in_nchw_f32 = x_kind;
  } else {
    const Buffer &ib = plan->bufs[d.in_buf];
    a.in = slice_ptr(plan, d.in_buf, d.in_coff); a.ih = ib.h; a.iw = ib.w; a.in_pitch = ib.c;
  }
  a.out = slice_ptr(plan, d.out_buf, d.out_coff);
  a.oh = ob.h; a.ow = ob.w; a.out_pitch = ob.c; a.out_f32 = ob.dtype == UYD_F32;
  if (d.res_buf >= 0) { a.res = slice_ptr(plan, d.res_buf, d.res_coff); a.res_pitch = plan->bufs[d.res_buf].c; }
  a.w = o.w_dev; a.bias = o.b_dev; a.cin = d.cin; a.cout = d.cout; a.k = d.k; a.stride = d.stride; a.relu = d.relu;
  return a;
}

// x_kind: 1 = NCHW fp32 frames, 2 = NCHW uint8 frames (divided by 255 on load), 3 = plan->cam (uyd_plan_run_camera)
static int launch_op(uyd_plan *plan, const Op &o, const void *x, int x_kind, int batch, cudaStream_t s, float *y = nullptr) {
  {
    int e = UYD_OK;
    if (o.kind == OP_CONV) {
      const uyd_conv &d = o.conv;
      if (o.use_tc) {
        e = tc_launch(o.tc, 0, batch, plan->ctx->sm_count, s);
      } else {
        if (d.in_buf < 0) UYD_REQUIRE(x, UYD_E_ARG, "uyd_plan_run: x is NULL");
        const ConvArgs a = direct_conv_args(plan, d, x, x_kind, batch, o);
        e = d.in_buf < 0 && x_kind == 3 ? stem_camera_launch(a, cam_frames(plan->cam), s) : direct_conv_launch(a, d.depthwise != 0, s);
      }
    } else if (o.kind == OP_C3K) {
      const Buffer &ib = plan->bufs[o.buf], &ob = plan->bufs[o.out_buf];
      C3kArgs a{};
      a.in = (const __nv_bfloat16 *)slice_ptr(plan, o.buf, o.coff);
      a.out = (__nv_bfloat16 *)slice_ptr(plan, o.out_buf, o.out_coff);
      a.wfrag = (const uint32_t *)o.w_dev; a.bias = o.b_dev;
      a.n = batch; a.h = ib.h; a.w = ib.w; a.in_pitch = ib.c; a.out_pitch = ob.c;
      e = o.quant ? c3k_launch_q(o.c, a, s) : c3k_launch(o.c, a, s);
    } else if (o.kind == OP_STEM2) {
      UYD_REQUIRE(x, UYD_E_ARG, "uyd_plan_run: x is NULL");
      const Buffer &ob = plan->bufs[o.out_buf];
      StemArgs a{};
      a.in = x; a.out = (__nv_bfloat16 *)slice_ptr(plan, o.out_buf, o.out_coff);
      a.wfrag = (const uint32_t *)o.w_dev; a.bias = o.b_dev;
      a.n = batch; a.ih = plan->in_h; a.iw = plan->in_w; a.oh = ob.h; a.ow = ob.w; a.out_pitch = ob.c; a.u8 = x_kind == 2; a.pw = o.c;
      if (x_kind == 3) a.f = cam_frames(plan->cam);
      e = stem_fused_launch(a, s);
    } else if (o.kind == OP_CHAIN) {
      UYD_REQUIRE(y || o.chain.out_buf >= 0, UYD_E_ARG, "this plan decodes in its head kernels: run it with uyd_plan_run_decoded");
      e = chain_launch(o.cc, batch, y, plan->ctx->sm_count, s);
    } else if (o.kind == OP_CLS) {
      const Buffer &ib = plan->bufs[o.buf], &ob = plan->bufs[o.out_buf];
      ClsArgs a{};
      a.in = (const __nv_bfloat16 *)slice_ptr(plan, o.buf, o.coff);
      a.out = (float *)slice_ptr(plan, o.out_buf, o.out_coff);
      a.wdw = (const __nv_bfloat16 *)o.w2_dev; a.wfrag = (const uint32_t *)o.w_dev; a.bias = o.b_dev;
      a.n = batch; a.h = ib.h; a.w = ib.w; a.in_pitch = ib.c; a.out_pitch = ob.c; a.nc = o.nc;
      e = cls_branch_launch(o.c, a, s);
    } else if (o.kind == OP_CONV_S8) {
      const uyd_conv &d = o.conv;
      if (o.use_tc) {
        e = tc_launch(o.tc, 0, batch, plan->ctx->sm_count, s);
      } else {
        const Buffer &ib = plan->bufs[d.in_buf], &ob = plan->bufs[d.out_buf];
        ConvArgs a{};
        a.n = batch; a.in = slice_ptr(plan, d.in_buf, d.in_coff); a.ih = ib.h; a.iw = ib.w; a.in_pitch = ib.c;
        a.out = slice_ptr(plan, d.out_buf, d.out_coff); a.oh = ob.h; a.ow = ob.w; a.out_pitch = ob.c;
        a.w = o.w_dev; a.bias = o.b_dev; a.cin = d.cin; a.cout = d.cout; a.k = d.k; a.stride = d.stride; a.relu = d.relu;
        if (d.res_buf >= 0) { a.res = slice_ptr(plan, d.res_buf, d.res_coff); a.res_pitch = plan->bufs[d.res_buf].c; }
        e = d.depthwise ? direct_conv_s8_dw_launch(a, o.m_dev, o.out_scale, o.out_kind, s)
                        : direct_conv_s8_launch(a, o.m_dev, o.out_scale, o.out_kind, s);
      }
    } else if (o.kind == OP_QUANT) {
      const Buffer &ib = plan->bufs[o.buf], &ob = plan->bufs[o.out_buf];
      e = quantize_s8_launch((const __nv_bfloat16 *)slice_ptr(plan, o.buf, o.coff), ib.c, (int8_t *)slice_ptr(plan, o.out_buf, o.out_coff),
                             ob.c, (long long)batch * ib.h * ib.w, o.c, o.out_scale, s);
    } else if (o.kind == OP_SPPF) {
      const Buffer &b = plan->bufs[o.buf];
      e = sppf_pool_launch((__nv_bfloat16 *)slice_ptr(plan, o.buf, o.coff), batch, b.h, b.w, b.c, o.c, s);
    } else {
      const Buffer &a = plan->bufs[o.buf], &b = plan->bufs[o.out_buf];
      e = upsample2x_launch((const __nv_bfloat16 *)slice_ptr(plan, o.buf, o.coff), a.c,
                            (__nv_bfloat16 *)slice_ptr(plan, o.out_buf, o.out_coff), b.c, batch, a.h, a.w, o.c, s);
    }
    return e;
  }
}

static int run_ops(uyd_plan *plan, const void *x, int x_kind, int batch, uyd_stream stream, float *y = nullptr) {
  UYD_REQUIRE(plan && plan->finalized, UYD_E_STATE, "plan not finalized");
  UYD_REQUIRE(batch > 0 && batch <= plan->max_batch, UYD_E_ARG, "batch %d outside (0, %d]", batch, plan->max_batch);
  uyd::DeviceGuard guard(plan->ctx->device);  // the stream must belong to the plan's device
  UYD_CUDA(guard.err);
  cudaStream_t s = (cudaStream_t)stream;
  for (size_t i = 0; i < plan->ops.size(); ++i) {
    const bool timed = (int)i == plan->timed_op && plan->timed_used < (int)plan->timed_ev.size() / 2;
    if (timed) UYD_CUDA(cudaEventRecord(plan->timed_ev[2 * plan->timed_used], s));
    int e = launch_op(plan, plan->ops[i], x, x_kind, batch, s, y);
    if (e) return e;
    if (timed) UYD_CUDA(cudaEventRecord(plan->timed_ev[2 * plan->timed_used++ + 1], s));
  }
  return UYD_OK;
}

extern "C" int uyd_plan_run(uyd_plan *plan, const float *x, int batch, uyd_stream stream) {
  return run_ops(plan, x, 1, batch, stream);
}

extern "C" int uyd_plan_run_u8(uyd_plan *plan, const uint8_t *x, int batch, uyd_stream stream) {
  return run_ops(plan, x, 2, batch, stream);
}

extern "C" int uyd_plan_run_decoded(uyd_plan *plan, const void *x, int x_dtype, int batch, float *y, uyd_stream stream) {
  UYD_REQUIRE(x_dtype == UYD_F32 || x_dtype == UYD_U8, UYD_E_ARG, "uyd_plan_run_decoded: x_dtype must be UYD_F32 or UYD_U8");
  UYD_REQUIRE(y, UYD_E_ARG, "uyd_plan_run_decoded: y is NULL");
  return run_ops(plan, x, x_dtype == UYD_F32 ? 1 : 2, batch, stream, y);
}

// Pinned host staging memory for frames (cudaHostAlloc): write_combined != 0 asks for write-combined pages, which the
// CPU fills sequentially and the GPU reads over PCIe without snooping the CPU caches.
extern "C" int uyd_host_alloc(size_t bytes, int write_combined, void **out) {
  UYD_REQUIRE(out && bytes > 0, UYD_E_ARG, "uyd_host_alloc: bad arguments");
  UYD_CUDA(cudaHostAlloc(out, bytes, write_combined ? cudaHostAllocWriteCombined : cudaHostAllocDefault));
  return UYD_OK;
}

extern "C" int uyd_host_free(void *p) {
  if (p) UYD_CUDA(cudaFreeHost(p));
  return UYD_OK;
}

extern "C" int uyd_plan_run_camera(uyd_plan *plan, const uyd_camera_frames *f, int batch, float *y, uyd_stream stream) {
  UYD_REQUIRE(plan && plan->finalized && f && f->data, UYD_E_ARG, "uyd_plan_run_camera: plan not finalized / NULL frames");
  UYD_REQUIRE(!plan->ops.empty(), UYD_E_UNSUPPORTED, "uyd_plan_run_camera: empty plan");
  const Op &stem = plan->ops[0];
  // the YAML network's fused stem, or model.py's Conv 3 -> 32 on the mma stem kernel: the stems with a camera loader
  const bool conv_stem = stem.kind == OP_CONV && !stem.use_tc && stem.conv.in_buf < 0 && !stem.conv.depthwise &&
                         stem_camera_supported(direct_conv_args(plan, stem.conv, f->data, 3, 1, stem));
  UYD_REQUIRE(stem.kind == OP_STEM2 || conv_stem, UYD_E_UNSUPPORTED,
              "uyd_plan_run_camera: the plan must start with the fused stem (uyd_plan_add_stem2 / _pw) or a Conv(3, 32, 3, 2) on the "
              "network input");
  UYD_REQUIRE(f->format == UYD_CAM_BGRA || f->format == UYD_CAM_NV12 || f->format == UYD_CAM_BGRA_LETTERBOX, UYD_E_ARG,
              "uyd_plan_run_camera: unknown frame format %d", f->format);
  UYD_REQUIRE(f->width > 0 && f->height > 0 && f->norm.std_r != 0.f && f->norm.std_g != 0.f && f->norm.std_b != 0.f, UYD_E_ARG, "uyd_plan_run_camera: bad extent or zero std");
  if (f->format == UYD_CAM_BGRA_LETTERBOX) {
    const LetterboxGeom g = letterbox_geometry(f->width, f->height, plan->in_w, plan->in_h);
    UYD_REQUIRE(g.new_w > 0 && g.new_h > 0, UYD_E_ARG, "uyd_plan_run_camera: a %d x %d frame letterboxes to nothing in %d x %d", f->width,
                f->height, plan->in_w, plan->in_h);
  }
  if (f->format != UYD_CAM_NV12) {
    UYD_REQUIRE(f->pitch >= 4 * f->width && f->pitch % 4 == 0 && f->frame_stride % 4 == 0 && (reinterpret_cast<uintptr_t>(f->data) & 3) == 0,
                UYD_E_ARG, "uyd_plan_run_camera: BGRA pixels must be 4-byte aligned (pitch %% 4 == 0)");
  } else {
    UYD_REQUIRE(f->uv && f->pitch >= f->width && f->uv_pitch >= f->width && f->width == plan->in_w && f->height == plan->in_h, UYD_E_ARG,
                "uyd_plan_run_camera: NV12 needs the UV plane and a frame of the plan's input extent (%d x %d)", plan->in_w, plan->in_h);
  }
  plan->cam = *f;
  return run_ops(plan, f->data, 3, batch, stream, y);
}

// Times every op separately with CUDA events on `stream` (one pass, ops serialised as in a
// normal run).  ms: [uyd_plan_num_launches].  Synchronises the stream.
extern "C" int uyd_plan_profile(uyd_plan *plan, const float *x, int batch, uyd_stream stream, float *ms) {
  UYD_REQUIRE(plan && plan->finalized && ms, UYD_E_STATE, "uyd_plan_profile: plan not finalized / ms NULL");
  UYD_REQUIRE(batch > 0 && batch <= plan->max_batch, UYD_E_ARG, "batch %d outside (0, %d]", batch, plan->max_batch);
  cudaStream_t s = (cudaStream_t)stream;
  const size_t n = plan->ops.size();
  uyd::DeviceGuard guard(plan->ctx->device);
  UYD_CUDA(guard.err);
  struct Events {  // destroyed on every return path
    std::vector<cudaEvent_t> ev;
    ~Events() { for (cudaEvent_t e : ev) if (e) cudaEventDestroy(e); }
  } E;
  E.ev.assign(n + 1, nullptr);
  auto &ev = E.ev;
  for (auto &e : ev) UYD_CUDA(cudaEventCreate(&e));
  UYD_CUDA(cudaEventRecord(ev[0], s));
  for (size_t i = 0; i < n; ++i) {
    int e = launch_op(plan, plan->ops[i], x, 1, batch, s, plan->profile_y);
    if (e) return e;
    UYD_CUDA(cudaEventRecord(ev[i + 1], s));
  }
  UYD_CUDA(cudaStreamSynchronize(s));
  for (size_t i = 0; i < n; ++i) UYD_CUDA(cudaEventElapsedTime(&ms[i], ev[i], ev[i + 1]));
  return UYD_OK;
}

extern "C" int uyd_plan_set_profile_output(uyd_plan *plan, float *y) {
  UYD_REQUIRE(plan, UYD_E_ARG, "uyd_plan_set_profile_output: plan is NULL");
  plan->profile_y = y;
  return UYD_OK;
}

// Brackets op `op` with CUDA events in every following uyd_plan_run (up to `max_samples`
// runs); op = -1 switches it off.  uyd_plan_timed_op_read synchronises those events.
extern "C" int uyd_plan_set_timed_op(uyd_plan *plan, int op, int max_samples) {
  UYD_REQUIRE(plan && plan->finalized, UYD_E_STATE, "plan not finalized");
  UYD_REQUIRE(op >= -1 && op < (int)plan->ops.size() && max_samples >= 0 && max_samples <= 4096, UYD_E_ARG,
              "uyd_plan_set_timed_op: bad arguments");
  for (cudaEvent_t e : plan->timed_ev) cudaEventDestroy(e);
  plan->timed_ev.clear();
  plan->timed_used = 0;
  plan->timed_op = op;
  if (op >= 0) {
    plan->timed_ev.resize(2 * (size_t)max_samples);
    for (auto &e : plan->timed_ev) UYD_CUDA(cudaEventCreate(&e));
  }
  return UYD_OK;
}

extern "C" int uyd_plan_timed_op_read(uyd_plan *plan, float *total_ms, int *samples) {
  UYD_REQUIRE(plan && total_ms && samples, UYD_E_ARG, "uyd_plan_timed_op_read: NULL argument");
  float tot = 0.f;
  for (int i = 0; i < plan->timed_used; ++i) {
    float ms = 0.f;
    UYD_CUDA(cudaEventSynchronize(plan->timed_ev[2 * i + 1]));
    UYD_CUDA(cudaEventElapsedTime(&ms, plan->timed_ev[2 * i], plan->timed_ev[2 * i + 1]));
    tot += ms;
  }
  *total_ms = tot;
  *samples = plan->timed_used;
  return UYD_OK;
}

// Human-readable description of op `op` plus its algorithmic work per image:
// flops (2*MAC) and compulsory bytes (input slice + output slice, weights excluded).
extern "C" int uyd_plan_op_info(uyd_plan *plan, int op, char *text, size_t text_len, double *flops_per_image,
                                double *bytes_per_image) {
  UYD_REQUIRE(plan && op >= 0 && op < (int)plan->ops.size() && text && text_len > 0, UYD_E_ARG, "uyd_plan_op_info: bad arguments");
  const Op &o = plan->ops[op];
  double fl = 0, by = 0;
  if (o.kind == OP_CONV || o.kind == OP_CONV_S8) {
    const uyd_conv &d = o.conv;
    const Buffer &ob = plan->bufs[d.out_buf];
    const int ih = d.in_buf < 0 ? plan->in_h : plan->bufs[d.in_buf].h, iw = d.in_buf < 0 ? plan->in_w : plan->bufs[d.in_buf].w;
    const double macs = (double)ob.h * ob.w * d.cout * d.k * d.k * (d.depthwise ? 1 : d.cin);
    fl = 2 * macs;
    by = (double)ih * iw * d.cin * (d.in_buf < 0 ? 4 : (o.kind == OP_CONV_S8 ? 1 : 2)) + (double)ob.h * ob.w * d.cout * ob.elem_bytes() +
         (d.res_buf >= 0 ? (double)ob.h * ob.w * d.cout * 2 : 0);
    snprintf(text, text_len, "conv%s %d->%d k%d s%d%s %dx%d %s%s%s", o.kind == OP_CONV_S8 ? "_s8" : "", d.cin, d.cout, d.k, d.stride,
             d.depthwise ? " dw" : "", ob.h, ob.w, o.use_tc ? "tc:" : "direct", o.use_tc ? tc_mode_name(o.tc) : "",
             d.res_buf >= 0 ? " +res" : (d.pre_buf_p1 ? " +up(partial)" : ""));
  } else if (o.kind == OP_QUANT) {
    const Buffer &b = plan->bufs[o.buf];
    by = (double)b.h * b.w * o.c * 3;
    snprintf(text, text_len, "quantize c%d %dx%d bf16->s8", o.c, b.h, b.w);
  } else if (o.kind == OP_STEM2) {
    const Buffer &b = plan->bufs[o.out_buf];
    fl = 2.0 * (4.0 * b.h * b.w * 16 * 27 + (double)b.h * b.w * 32 * 144 + (o.c ? (double)b.h * b.w * 16 * 32 : 0.0));
    by = 16.0 * b.h * b.w * 3 * 4 + (double)b.h * b.w * (o.c ? 16 : 32) * 2;
    snprintf(text, text_len, "stem2 3->16 k3 s2 + 16->32 k3 s2%s fused -> %dx%d", o.c ? " + 32->16 k1" : "", b.h, b.w);
  } else if (o.kind == OP_CHAIN) {
    const uyd_chain &d = o.chain;
    const Buffer &b = plan->bufs[d.in_buf];
    const double px = (double)b.h * b.w;
    fl = 2.0 * px * ((d.dw1 ? 9.0 * d.cin : 9.0 * d.cin * d.n1) + (double)d.n1 * d.n2 + (d.final_kind == UYD_CHAIN_PW3 ? (double)d.n2 * d.nc : 0.0));
    const double dec = d.final_kind == UYD_CHAIN_DFL ? 16 : (d.final_kind == UYD_CHAIN_PW3 ? 4.0 * d.nc : 0);
    const double rawb = d.out_buf >= 0 ? (d.final_kind == UYD_CHAIN_PW3 ? 4.0 * d.nc : d.n2 * (double)plan->bufs[d.out_buf].elem_bytes()) : 0;
    by = px * (d.cin * 2.0 + rawb + (d.out_buf >= 0 && d.final_kind != UYD_CHAIN_STORE ? 0 : dec));
    snprintf(text, text_len, "chain %s%d->%d k3 + %d->%d k1 + %s %dx%d tc", d.dw1 ? "dw" : "", d.cin, d.n1, d.n1, d.n2,
             d.final_kind == UYD_CHAIN_DFL ? "dfl" : (d.final_kind == UYD_CHAIN_PW3 ? "pw3" : "store"), b.h, b.w);
  } else if (o.kind == OP_CLS) {
    const Buffer &b = plan->bufs[o.buf];
    const double c = o.c;
    fl = 2.0 * b.h * b.w * (9 * c + c * 32 + 9 * 32 + 32 * 32 + 32 * o.nc);
    by = (double)b.h * b.w * (c * 2 + o.nc * 4);
    snprintf(text, text_len, "cls_branch_fused c%d %dx%d (5 convs)", o.c, b.h, b.w);
  } else if (o.kind == OP_C3K) {
    const Buffer &b = plan->bufs[o.buf];
    const double c = o.c, h = c / 2;
    fl = 2.0 * b.h * b.w * (2 * c * h + 4 * 9 * h * h + c * c);
    by = (double)b.h * b.w * c * 2 * 2;
    snprintf(text, text_len, "%s c%d %dx%d (7 convs)", o.quant ? "c3k_fused_s8" : "c3k_fused", o.c, b.h, b.w);
  } else if (o.kind == OP_SPPF) {
    const Buffer &b = plan->bufs[o.buf];
    by = (double)b.h * b.w * o.c * 2 * 4;
    snprintf(text, text_len, "sppf_pool c%d %dx%d", o.c, b.h, b.w);
  } else {
    const Buffer &b = plan->bufs[o.out_buf];
    by = (double)b.h * b.w * o.c * 2 * 1.25;
    snprintf(text, text_len, "upsample2x c%d -> %dx%d", o.c, b.h, b.w);
  }
  if (flops_per_image) *flops_per_image = fl;
  if (bytes_per_image) *bytes_per_image = by;
  return UYD_OK;
}

extern "C" int uyd_plan_run_decode(uyd_plan *plan, float *y, int batch, uyd_stream stream) {
  UYD_REQUIRE(plan && plan->finalized && !plan->heads.empty(), UYD_E_STATE, "plan has no heads / not finalized");
  UYD_REQUIRE(y && batch > 0 && batch <= plan->max_batch, UYD_E_ARG, "uyd_plan_run_decode: bad arguments");
  uyd::DeviceGuard guard(plan->ctx->device);
  int a_total = 0;
  for (int h : plan->heads) a_total += plan->bufs[h].h * plan->bufs[h].w;
  int a_off = 0;
  for (size_t i = 0; i < plan->heads.size(); ++i) {
    const Buffer &b = plan->bufs[plan->heads[i]];
    int e = decode_dfl_launch((const float *)b.ptr, batch, b.h, b.w, plan->reg_max, plan->nc, (float)plan->head_strides[i], y,
                              a_total, a_off, (cudaStream_t)stream, plan->dfl_amax);
    if (e) return e;
    a_off += b.h * b.w;
  }
  return UYD_OK;
}

extern "C" int uyd_plan_set_dfl_quant(uyd_plan *plan, float amax_in) {
  UYD_REQUIRE(plan && amax_in >= 0.f, UYD_E_ARG, "uyd_plan_set_dfl_quant: bad arguments");
  plan->dfl_amax = amax_in;
  return UYD_OK;
}

extern "C" int uyd_plan_export_head_nchw(uyd_plan *plan, int level, float *out, int batch, uyd_stream stream) {
  UYD_REQUIRE(plan && plan->finalized && level >= 0 && level < (int)plan->heads.size() && out, UYD_E_ARG,
              "uyd_plan_export_head_nchw: bad arguments");
  const Buffer &b = plan->bufs[plan->heads[level]];
  uyd::DeviceGuard guard(plan->ctx->device);
  return nhwc_to_nchw_f32_launch((const float *)b.ptr, out, batch, b.h, b.w, b.c, (cudaStream_t)stream);
}

extern "C" int uyd_memcpy_d2d(void *dst, const void *src, size_t bytes, uyd_stream stream) {
  UYD_REQUIRE(dst && src, UYD_E_ARG, "uyd_memcpy_d2d: NULL pointer");
  cudaPointerAttributes at;  // run on the device that owns the destination (the stream must belong to it)
  int dev = -1;
  if (cudaPointerGetAttributes(&at, dst) == cudaSuccess && at.type == cudaMemoryTypeDevice) dev = at.device;
  uyd::DeviceGuard guard(dev >= 0 ? dev : uyd::ctx_device(nullptr));
  UYD_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)stream));
  return UYD_OK;
}
