// C ABI of libcdrhead.so: error state, packed-weight handles, workspace planning and the
// orchestration of the head / decoder forward passes (include/cdrhead.h).
#include <initializer_list>
#include <new>
#include <string.h>

#include "kernels.h"
#include "tc_api.h"

namespace cdr {

static unsigned int* g_debug_host = nullptr;
int tc_set_debug(unsigned int* d);      // gemm_tc.cu / heatmap.cu: point their copy of g_cdr_debug at the words
int heat_set_debug(unsigned int* d);

static thread_local char g_err[512] = "";
static thread_local unsigned long long g_launches = 0;

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// ---- optional per-launch timing (bench.py's live roofline numbers): one event after every
// launch on the timing stream; durations are differences of consecutive events.
constexpr int kMaxTimed = 512;
struct StageTiming {
  bool on = false;
  cudaStream_t stream = nullptr;
  int n = 0;
  cudaEvent_t ev[kMaxTimed + 1] = {};
  char name[kMaxTimed][48];
  const char* label = nullptr;
};
static thread_local StageTiming g_timing;

void set_stage(const char* label) { g_timing.label = label; }
// called at the entry of a forward: if nothing has been timed yet, move the start marker here so
// the first stage does not include the caller's host-side latency
void timing_restart() {
  StageTiming& t = g_timing;
  if (t.on && t.n == 0) cudaEventRecord(t.ev[0], t.stream);
}
void count_launch(const char* kernel) {
  g_launches += 1;
  StageTiming& t = g_timing;
  if (!t.on || t.n >= kMaxTimed) return;
  const int i = t.n + 1;
  if (!t.ev[i] && cudaEventCreate(&t.ev[i]) != cudaSuccess) return;
  if (cudaEventRecord(t.ev[i], t.stream) != cudaSuccess) return;
  snprintf(t.name[t.n], sizeof(t.name[t.n]), "%s", t.label ? t.label : kernel);
  t.n = i;
}

struct Bump {  // 256-byte aligned bump allocator over a caller-provided region
  uint8_t* base;
  size_t off = 0;
  explicit Bump(void* b) : base((uint8_t*)b) {}
  template <typename T>
  T* take(size_t count) {
    T* p = base ? (T*)(base + off) : nullptr;
    off += round_up<size_t>(count * sizeof(T), 256);
    return p;
  }
};

}  // namespace cdr

using namespace cdr;

// ------------------------------------------------------------------------------------------
struct CdrWeights {
  int precision = 0, joints = 0, has_fusion = 0, fin_npad = 0;
  FusionDims fd;
  void* pool = nullptr;
  // fp32 path: B operands as [K][n_pad]
  float *w_cf1 = nullptr, *b_cf1 = nullptr, *w_cf2a = nullptr, *b_cf2a = nullptr;
  float *w_cf2b = nullptr, *b_cf2b = nullptr, *w_out = nullptr, *b_out = nullptr;
  float *w_dc[3] = {nullptr, nullptr, nullptr}, *b_dc[3] = {nullptr, nullptr, nullptr};
  float *w_fin = nullptr, *b_fin = nullptr;
  TcWeights tc;  // bf16 tensor-core path (gemm_tc.cu)
};

static const int kDcCin[3] = {kFeatC, kDecC, kDecC};

static void plan_fp32_weights(CdrWeights& w, Bump& b) {
  const FusionDims& fd = w.fd;
  if (w.has_fusion) {
    w.w_cf1 = b.take<float>((size_t)kFeatC * fd.n1_pad());
    w.b_cf1 = b.take<float>(fd.n1_pad());
    w.w_cf2a = b.take<float>((size_t)2 * fd.h2 * fd.n2_pad());
    w.b_cf2a = b.take<float>(fd.n2_pad());
    w.w_cf2b = b.take<float>((size_t)fd.h2 * fd.n2_pad());
    w.b_cf2b = b.take<float>(fd.n2_pad());
    w.w_out = b.take<float>((size_t)2 * fd.h1p * kFeatC);
    w.b_out = b.take<float>((size_t)2 * kFeatC);
  }
  for (int i = 0; i < 3; ++i) {
    w.w_dc[i] = b.take<float>((size_t)16 * kDcCin[i] * kDecC);
    w.b_dc[i] = b.take<float>(kDecC);
  }
  w.w_fin = b.take<float>((size_t)kDecC * w.fin_npad);
  w.b_fin = b.take<float>(w.fin_npad);
}

extern "C" int cdr_abi_version(void) { return CDRHEAD_ABI_VERSION; }
extern "C" const char* cdr_last_error(void) { return g_err; }
extern "C" unsigned long long cdr_launch_count(void) { return g_launches; }
extern "C" void cdr_launch_count_reset(void) { g_launches = 0; }

extern "C" int cdr_stage_timing_begin(void* stream) {
  StageTiming& t = g_timing;
  if (!t.ev[0]) CDR_CUDA(cudaEventCreate(&t.ev[0]));
  t.stream = (cudaStream_t)stream;
  t.n = 0;
  t.label = nullptr;
  CDR_CUDA(cudaEventRecord(t.ev[0], t.stream));
  t.on = true;
  return CDR_OK;
}

extern "C" int cdr_stage_timing_end(int capacity, char* names, float* ms, int* count) {
  StageTiming& t = g_timing;
  CDR_CHECK_ARG(t.on, "cdr_stage_timing_end: timing was not started");
  CDR_CHECK_ARG(names && ms && count && capacity > 0, "cdr_stage_timing_end: bad args");
  t.on = false;
  t.label = nullptr;
  if (t.n > 0) CDR_CUDA(cudaEventSynchronize(t.ev[t.n]));
  const int n = t.n < capacity ? t.n : capacity;
  for (int i = 0; i < n; ++i) {
    CDR_CUDA(cudaEventElapsedTime(&ms[i], t.ev[i], t.ev[i + 1]));
    memcpy(names + (size_t)i * 48, t.name[i], 48);
  }
  *count = n;
  return CDR_OK;
}

extern "C" int cdr_weights_create(const CdrWeightPtrs* src, int precision, void* stream,
                                  CdrWeights** out) {
  CDR_CHECK_ARG(src && out, "cdr_weights_create: null argument");
  CDR_CHECK_ARG(precision == CDR_PREC_FP32 || precision == CDR_PREC_BF16 || precision == CDR_PREC_TF32X3 ||
                    precision == CDR_PREC_F16X2,
                "cdr_weights_create: unknown precision %d", precision);
  CDR_CHECK_ARG(src->num_joints > 0 && src->num_joints <= kMaxJoints,
                "cdr_weights_create: num_joints must be 1..%d", kMaxJoints);
  for (int i = 0; i < 3; ++i)
    CDR_CHECK_ARG(src->deconv[i].weight && src->deconv[i].bn_weight && src->deconv[i].bn_bias &&
                      src->deconv[i].bn_mean && src->deconv[i].bn_var,
                  "cdr_weights_create: decoder.deconv%d tensors missing", i + 1);
  CDR_CHECK_ARG(src->final_layer.weight && src->final_layer.bias,
                "cdr_weights_create: decoder.final_layer tensors missing");
  if (src->has_fusion) {
    const CdrConvBn* cf[5] = {&src->cf_conv1, &src->cf_conv2a, &src->cf_conv2b, &src->cf_out[0],
                              &src->cf_out[1]};
    for (const CdrConvBn* c : cf)
      CDR_CHECK_ARG(c->weight && c->bias && c->bn_weight && c->bn_bias && c->bn_mean && c->bn_var,
                    "cdr_weights_create: a CF.* tensor is missing");
  }
  cudaStream_t st = (cudaStream_t)stream;
  CdrWeights* w = new (std::nothrow) CdrWeights();
  CDR_CHECK_ARG(w, "cdr_weights_create: out of host memory");
  w->precision = precision;
  w->joints = src->num_joints;
  w->has_fusion = src->has_fusion;
  w->fin_npad = src->num_joints <= 32 ? 32 : round_up(src->num_joints, 128);
  if (src->has_fusion && (src->fusion_hid_ch1 || src->fusion_hid_ch2)) {
    if (!fusion_dims_ok(src->fusion_hid_ch1, src->fusion_hid_ch2)) {
      set_error("cdr_weights_create: fusion widths %d / %d: need hid_ch2 = 4/3 hid_ch1 (the reference's ftl) and "
                "hid_ch1 %% 12 == 0", src->fusion_hid_ch1, src->fusion_hid_ch2);
      delete w;
      return CDR_ERR_UNSUPPORTED;
    }
    w->fd = make_fusion_dims(src->fusion_hid_ch1, src->fusion_hid_ch2);
  }

  int rc = CDR_OK;
  auto fail = [&](int code) {
    if (w->pool) cudaFree(w->pool);
    tc_weights_destroy(w->tc);          // frees the TcPack and its device pool if packing got that far (no-op otherwise)
    delete w;
    return code;
  };
  if (precision == CDR_PREC_FP32) {
    Bump sizing(nullptr);
    plan_fp32_weights(*w, sizing);
    cudaError_t e = cudaMalloc(&w->pool, sizing.off);
    if (e != cudaSuccess) {
      set_error("cdr_weights_create: cudaMalloc(%zu) failed: %s", sizing.off, cudaGetErrorString(e));
      w->pool = nullptr;
      return fail(CDR_ERR_CUDA);
    }
    Bump b(w->pool);
    plan_fp32_weights(*w, b);
    if (w->has_fusion) {
      if ((rc = launch_pack_conv1x1_f32(src->cf_conv1, w->fd.h1, kFeatC, kFeatC, w->fd.n1_pad(), w->w_cf1, w->b_cf1, st))) return fail(rc);
      if ((rc = launch_pack_conv1x1_f32(src->cf_conv2a, w->fd.h2, 2 * w->fd.h2, 2 * w->fd.h2, w->fd.n2_pad(), w->w_cf2a, w->b_cf2a, st))) return fail(rc);
      if ((rc = launch_pack_conv1x1_f32(src->cf_conv2b, w->fd.h2, w->fd.h2, w->fd.h2, w->fd.n2_pad(), w->w_cf2b, w->b_cf2b, st))) return fail(rc);
      for (int v = 0; v < 2; ++v)
        if ((rc = launch_pack_conv1x1_f32(src->cf_out[v], kFeatC, w->fd.h1, w->fd.h1p, kFeatC,
                                          w->w_out + (size_t)v * w->fd.h1p * kFeatC,
                                          w->b_out + (size_t)v * kFeatC, st)))
          return fail(rc);
    }
    for (int i = 0; i < 3; ++i)
      if ((rc = launch_pack_deconv_f32(src->deconv[i], kDcCin[i], kDecC, kDecC, w->w_dc[i], w->b_dc[i], st)))
        return fail(rc);
    if ((rc = launch_pack_conv1x1_f32(src->final_layer, w->joints, kDecC, kDecC, w->fin_npad, w->w_fin, w->b_fin, st)))
      return fail(rc);
  } else {
    const int mode = precision == CDR_PREC_BF16 ? 0 : precision == CDR_PREC_TF32X3 ? 1 : 2;
    if ((rc = tc_weights_create(*src, mode, w->tc, st))) return fail(rc);
  }
  cudaError_t e = cudaStreamSynchronize(st);
  if (e != cudaSuccess) {
    set_error("cdr_weights_create: packing failed: %s", cudaGetErrorString(e));
    return fail(CDR_ERR_CUDA);
  }
  *out = w;
  return CDR_OK;
}

extern "C" int cdr_weights_destroy(CdrWeights* w) {
  if (!w) return CDR_OK;
  if (w->pool) cudaFree(w->pool);
  tc_weights_destroy(w->tc);
  delete w;
  return CDR_OK;
}

// ------------------------------------------------------------------------------------------
// workspace plans
struct HeadWs {
  float *pinv, *x0, *y1, *z, *f1, *f2, *g, *x1, *d1, *d2, *d3, *hm;
  size_t bytes;
};
static HeadWs plan_head_f32(void* base, int B, int J, const FusionDims& fd) {
  Bump b(base);
  const size_t N = 2 * (size_t)B;
  HeadWs w;
  w.pinv = b.take<float>(N * 12);
  w.x0 = b.take<float>(N * kFeatHW * kFeatC);
  w.y1 = b.take<float>(N * kFeatHW * fd.h1p);
  w.z = b.take<float>((size_t)B * kFeatHW * 2 * fd.h2);
  w.f1 = b.take<float>((size_t)B * kFeatHW * fd.h2);
  w.f2 = b.take<float>((size_t)B * kFeatHW * fd.h2);
  w.g = b.take<float>(N * kFeatHW * fd.h1p);
  w.x1 = b.take<float>(N * kFeatHW * kFeatC);
  w.d1 = b.take<float>(N * 256 * kDecC);
  w.d2 = b.take<float>(N * 1024 * kDecC);
  w.d3 = b.take<float>(N * 4096 * kDecC);
  w.hm = b.take<float>(N * J * 4096);
  w.bytes = b.off;
  return w;
}
struct DecWs {
  float *x1, *d1, *d2, *d3;
  size_t bytes;
};
static DecWs plan_dec_f32(void* base, int N) {
  Bump b(base);
  DecWs w;
  w.x1 = b.take<float>((size_t)N * kFeatHW * kFeatC);
  w.d1 = b.take<float>((size_t)N * 256 * kDecC);
  w.d2 = b.take<float>((size_t)N * 1024 * kDecC);
  w.d3 = b.take<float>((size_t)N * 4096 * kDecC);
  w.bytes = b.off;
  return w;
}

extern "C" int cdr_head_workspace_bytes(const CdrWeights* w, int batch, size_t* bytes) {
  CDR_CHECK_ARG(w && bytes && batch > 0, "cdr_head_workspace_bytes: bad args");
  CDR_CHECK_ARG(w->has_fusion, "cdr_head_workspace_bytes: decoder-only weights");
  if (w->precision != CDR_PREC_FP32) return tc_head_workspace_bytes(w->tc, batch, bytes);
  *bytes = plan_head_f32(nullptr, batch, w->joints, w->fd).bytes;
  return CDR_OK;
}
extern "C" int cdr_decoder_workspace_bytes(const CdrWeights* w, int n_images, size_t* bytes) {
  CDR_CHECK_ARG(w && bytes && n_images > 0, "cdr_decoder_workspace_bytes: bad args");
  if (w->precision != CDR_PREC_FP32) return tc_decoder_workspace_bytes(w->tc, n_images, bytes);
  *bytes = plan_dec_f32(nullptr, n_images).bytes;
  return CDR_OK;
}

// ------------------------------------------------------------------------------------------
// fp32 decoder: three transposed convs + the 1x1 head (models/decoder.py:39-46)
static int decoder_f32(const CdrWeights* w, const float* x1, int N, float* d1, float* d2, float* d3,
                       float* heat, cudaStream_t st) {
  const float* in = x1;
  float* outs[3] = {d1, d2, d3};
  int side = 8;
  static const char* const kDcName[3] = {"deconv1", "deconv2", "deconv3"};
  for (int i = 0; i < 3; ++i) {
    set_stage(kDcName[i]);
    TapGemmParams p{};
    p.A = in;
    p.a_pitch = kDcCin[i];
    p.n_img = N;
    p.H = p.W = side;
    p.cin = kDcCin[i];
    p.deconv = 1;
    p.Wp = w->w_dc[i];
    p.w_group_stride = (long long)4 * kDcCin[i] * kDecC;
    p.bias = w->b_dc[i];
    p.bias_group_stride = 0;
    p.n_pad = kDecC;
    p.n = kDecC;
    p.C = outs[i];
    p.c_pitch = kDecC;
    p.c_fill = kDecC;
    p.relu = 1;
    p.out_mode = kOutDeconv;
    if (int rc = launch_tap_gemm_ffma(p, 4, st)) return rc;
    in = outs[i];
    side *= 2;
  }
  set_stage("final_1x1");
  TapGemmParams p{};
  p.A = d3;
  p.a_pitch = kDecC;
  p.n_img = N;
  p.H = p.W = kHeat;
  p.cin = kDecC;
  p.Wp = w->w_fin;
  p.bias = w->b_fin;
  p.n_pad = w->fin_npad;
  p.n = w->joints;
  p.C = heat;
  p.c_pitch = 4;
  p.c_fill = 4;
  p.relu = 0;
  p.out_mode = kOutPlanar;
  const int rc = launch_tap_gemm_ffma(p, 1, st);
  set_stage(nullptr);
  return rc;
}

static int copy_tap(float* dst, const float* src, size_t count, cudaStream_t st) {
  if (!dst) return CDR_OK;
  CDR_CUDA(cudaMemcpyAsync(dst, src, count * sizeof(float), cudaMemcpyDeviceToDevice, st));
  return CDR_OK;
}

extern "C" int cdr_head_forward(const CdrWeights* w, const float* feat_l, const float* feat_r,
                                const float* P_l, const float* P_r, const float* pinv_l,
                                const float* pinv_r, double pinv_rtol, int batch, int img_size,
                                float* kp2d_l, float* kp2d_r, float* xyz, const CdrHeadTaps* taps,
                                void* workspace, size_t workspace_bytes, void* stream) {
  CDR_CHECK_ARG(w && feat_l && feat_r && P_l && P_r && kp2d_l && kp2d_r && xyz && workspace,
                "cdr_head_forward: null pointer");
  CDR_CHECK_ARG(w->has_fusion, "cdr_head_forward: weights were created without the fusion block");
  CDR_CHECK_ARG(batch > 0 && img_size > 0, "cdr_head_forward: bad batch/img_size");
  CDR_CHECK_ARG((pinv_l == nullptr) == (pinv_r == nullptr),
                "cdr_head_forward: give both pseudo-inverses or neither");
  CDR_CHECK_ARG(((uintptr_t)workspace & 255) == 0, "cdr_head_forward: workspace must be 256-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  timing_restart();
  const float scale = (float)img_size / (float)kHeat;   // models/cdrnet.py:250
  if (w->precision != CDR_PREC_FP32)
    return tc_head_forward(w->tc, nullptr, 0, feat_l, feat_r, P_l, P_r, pinv_l, pinv_r, pinv_rtol, batch, scale,
                           kp2d_l, kp2d_r, xyz, taps, workspace, workspace_bytes, st);

  const int B = batch, N = 2 * batch, J = w->joints;
  HeadWs ws = plan_head_f32(workspace, B, J, w->fd);
  if (ws.bytes > workspace_bytes) {
    set_error("cdr_head_forward: workspace %zu < required %zu bytes", workspace_bytes, ws.bytes);
    return CDR_ERR_WORKSPACE;
  }
  int rc;
  const FusionDims& fd = w->fd;
  // (1) P^+  — models/cdrnet.py:236-237
  set_stage("pinv");
  const float* pinv[2] = {pinv_l, pinv_r};
  if (!pinv_l) {
    if ((rc = launch_pinv2(P_l, P_r, B, pinv_rtol, ws.pinv, nullptr, st))) return rc;
    pinv[0] = ws.pinv;
    pinv[1] = ws.pinv + (size_t)B * 12;
  }
  // (2) encoder latents NCHW -> pixel-major rows, views stacked (conv_layer1 is shared)
  set_stage("nchw_to_rows");
  if ((rc = launch_nchw_to_rows_f32(feat_l, feat_r, B, kFeatC, kFeatHW, ws.x0, kFeatC, st))) return rc;
  // (3) conv_layer1 2048 -> 300 (+BN+ReLU) — :62
  set_stage("cf_conv1");
  {
    TapGemmParams p{};
    p.A = ws.x0; p.a_pitch = kFeatC; p.n_img = N; p.H = p.W = 8; p.cin = kFeatC;
    p.Wp = w->w_cf1; p.bias = w->b_cf1; p.n_pad = fd.n1_pad(); p.n = fd.h1;
    p.C = ws.y1; p.c_pitch = fd.h1p; p.c_fill = fd.h1p; p.relu = 1; p.out_mode = kOutRows;
    if ((rc = launch_tap_gemm_ffma(p, 1, st))) return rc;
  }
  // (4) inverse FTL into the concatenated (B,64,800) buffer — :65,70
  set_stage("ftl_inv");
  {
    const float* ins[2] = {ws.y1, ws.y1 + (size_t)B * kFeatHW * fd.h1p};
    float* outs[2] = {ws.z, ws.z + fd.h2};
    if ((rc = launch_ftl2<float>(ins, fd.h1p, pinv, 4, 3, fd.blk, B, kFeatHW, outs, 2 * fd.h2, fd.h2, 2, st)))
      return rc;
  }
  // (5) conv_layer2: 800 -> 400 -> 400 — :74
  set_stage("cf_conv2");
  {
    TapGemmParams p{};
    p.A = ws.z; p.a_pitch = 2 * fd.h2; p.n_img = B; p.H = p.W = 8; p.cin = 2 * fd.h2;
    p.Wp = w->w_cf2a; p.bias = w->b_cf2a; p.n_pad = fd.n2_pad(); p.n = fd.h2;
    p.C = ws.f1; p.c_pitch = fd.h2; p.c_fill = fd.h2; p.relu = 1; p.out_mode = kOutRows;
    if ((rc = launch_tap_gemm_ffma(p, 1, st))) return rc;
    p.A = ws.f1; p.a_pitch = fd.h2; p.cin = fd.h2; p.Wp = w->w_cf2b; p.bias = w->b_cf2b; p.C = ws.f2;
    if ((rc = launch_tap_gemm_ffma(p, 1, st))) return rc;
  }
  // (6) forward FTL per view — :79
  set_stage("ftl_fwd");
  const float* Pv[2] = {P_l, P_r};
  {
    const float* ins[2] = {ws.f2, ws.f2};
    float* outs[2] = {ws.g, ws.g + (size_t)B * kFeatHW * fd.h1p};
    if ((rc = launch_ftl2<float>(ins, fd.h2, Pv, 3, 4, fd.blk, B, kFeatHW, outs, fd.h1p, fd.h1p, 2, st)))
      return rc;
  }
  // (7) out_layer[v] 300 -> 2048, per-view weights = 2 groups — :81
  set_stage("cf_out");
  {
    TapGemmParams p{};
    p.A = ws.g; p.a_group_stride = (long long)B * kFeatHW * fd.h1p; p.a_pitch = fd.h1p;
    p.n_img = B; p.H = p.W = 8; p.cin = fd.h1p;
    p.Wp = w->w_out; p.w_group_stride = (long long)fd.h1p * kFeatC;
    p.bias = w->b_out; p.bias_group_stride = kFeatC; p.n_pad = kFeatC; p.n = kFeatC;
    p.C = ws.x1; p.c_group_stride = (long long)B * kFeatHW * kFeatC; p.c_pitch = kFeatC;
    p.c_fill = kFeatC; p.relu = 1; p.out_mode = kOutRows;
    if ((rc = launch_tap_gemm_ffma(p, 2, st))) return rc;
  }
  // (8) decoder on both views at once (shared weights) — :243-244
  if ((rc = decoder_f32(w, ws.x1, N, ws.d1, ws.d2, ws.d3, ws.hm, st))) return rc;
  // (9) soft-argmax + DLT — :247-266
  set_stage("softargmax_dlt");
  if ((rc = cdr_softargmax_dlt(ws.hm, ws.hm + (size_t)B * J * 4096, 0, P_l, P_r, B, J, kHeat, kHeat,
                               scale, kp2d_l, kp2d_r, xyz, nullptr, nullptr, nullptr, nullptr,
                               nullptr, st)))
    return rc;
  set_stage(nullptr);
  if (taps) {
    if ((rc = copy_tap(taps->pinv, pinv[0], (size_t)B * 12, st))) return rc;
    if ((rc = copy_tap(taps->pinv ? taps->pinv + (size_t)B * 12 : nullptr, pinv[1], (size_t)B * 12, st))) return rc;
    if ((rc = copy_tap(taps->cf_cat, ws.z, (size_t)B * kFeatHW * 2 * fd.h2, st))) return rc;
    if ((rc = copy_tap(taps->cf_f, ws.f2, (size_t)B * kFeatHW * fd.h2, st))) return rc;
    if ((rc = copy_tap(taps->f_out, ws.x1, (size_t)N * kFeatHW * kFeatC, st))) return rc;
    if ((rc = copy_tap(taps->heatmaps, ws.hm, (size_t)N * J * 4096, st))) return rc;
  }
  return CDR_OK;
}

extern "C" int cdr_decoder_forward(const CdrWeights* w, const float* feat, int n_images,
                                   float* heatmaps, void* workspace, size_t workspace_bytes,
                                   void* stream) {
  CDR_CHECK_ARG(w && feat && heatmaps && workspace && n_images > 0, "cdr_decoder_forward: bad args");
  CDR_CHECK_ARG(((uintptr_t)workspace & 255) == 0, "cdr_decoder_forward: workspace must be 256-byte aligned");
  cudaStream_t st = (cudaStream_t)stream;
  if (w->precision != CDR_PREC_FP32)
    return tc_decoder_forward(w->tc, nullptr, 0, feat, n_images, heatmaps, workspace, workspace_bytes, st);
  DecWs ws = plan_dec_f32(workspace, n_images);
  if (ws.bytes > workspace_bytes) {
    set_error("cdr_decoder_forward: workspace %zu < required %zu bytes", workspace_bytes, ws.bytes);
    return CDR_ERR_WORKSPACE;
  }
  if (int rc = launch_nchw_to_rows_f32(feat, nullptr, n_images, kFeatC, kFeatHW, ws.x1, kFeatC, st)) return rc;
  return decoder_f32(w, ws.x1, n_images, ws.d1, ws.d2, ws.d3, heatmaps, st);
}

// ------------------------------------------------------------------------------------------
// tcgen05 encoder + head on its row-major output
extern "C" int cdr_head_forward_rows(const CdrWeights* w, const void* feat_rows, const float* P_l, const float* P_r,
                                     const float* pinv_l, const float* pinv_r, double pinv_rtol, int batch,
                                     int img_size, float* kp2d_l, float* kp2d_r, float* xyz,
                                     const CdrHeadTaps* taps, void* workspace, size_t workspace_bytes,
                                     void* stream) {
  CDR_CHECK_ARG(w && feat_rows && P_l && P_r && kp2d_l && kp2d_r && xyz && workspace,
                "cdr_head_forward_rows: null pointer");
  CDR_CHECK_ARG(w->has_fusion, "cdr_head_forward_rows: weights were created without the fusion block");
  CDR_CHECK_ARG(w->precision != CDR_PREC_FP32, "cdr_head_forward_rows: needs a tensor-core precision");
  CDR_CHECK_ARG(batch > 0 && img_size > 0, "cdr_head_forward_rows: bad batch/img_size");
  CDR_CHECK_ARG((pinv_l == nullptr) == (pinv_r == nullptr), "cdr_head_forward_rows: give both pseudo-inverses or neither");
  CDR_CHECK_ARG(((uintptr_t)workspace & 255) == 0 && ((uintptr_t)feat_rows & 15) == 0,
                "cdr_head_forward_rows: workspace must be 256-byte, features 16-byte aligned");
  timing_restart();
  return tc_head_forward(w->tc, feat_rows, 0, nullptr, nullptr, P_l, P_r, pinv_l, pinv_r, pinv_rtol, batch,
                         (float)img_size / (float)kHeat, kp2d_l, kp2d_r, xyz, taps, workspace, workspace_bytes,
                         (cudaStream_t)stream);
}
extern "C" int cdr_head_forward_planes(const CdrWeights* w, const void* feat_planes, const float* P_l, const float* P_r,
                                       const float* pinv_l, const float* pinv_r, double pinv_rtol, int batch,
                                       int img_size, float* kp2d_l, float* kp2d_r, float* xyz,
                                       const CdrHeadTaps* taps, void* workspace, size_t workspace_bytes,
                                       void* stream) {
  CDR_CHECK_ARG(w && feat_planes && P_l && P_r && kp2d_l && kp2d_r && xyz && workspace,
                "cdr_head_forward_planes: null pointer");
  CDR_CHECK_ARG(w->has_fusion, "cdr_head_forward_planes: weights were created without the fusion block");
  CDR_CHECK_ARG(w->precision == CDR_PREC_F16X2, "cdr_head_forward_planes: needs the f16x2 (\"fp32\") precision");
  CDR_CHECK_ARG(batch > 0 && img_size > 0, "cdr_head_forward_planes: bad batch/img_size");
  CDR_CHECK_ARG((pinv_l == nullptr) == (pinv_r == nullptr), "cdr_head_forward_planes: give both pseudo-inverses or neither");
  CDR_CHECK_ARG(((uintptr_t)workspace & 255) == 0 && ((uintptr_t)feat_planes & 255) == 0,
                "cdr_head_forward_planes: workspace must be 256-byte, the planes buffer 256-byte aligned");
  timing_restart();
  return tc_head_forward(w->tc, feat_planes, 1, nullptr, nullptr, P_l, P_r, pinv_l, pinv_r, pinv_rtol, batch,
                         (float)img_size / (float)kHeat, kp2d_l, kp2d_r, xyz, taps, workspace, workspace_bytes,
                         (cudaStream_t)stream);
}

struct CdrEncoder {
  void* impl = nullptr;
};

extern "C" int cdr_encoder_create(const CdrEncoderSpec* spec, void* stream, CdrEncoder** out) {
  return cdr_encoder_create_prec(spec, CDR_PREC_BF16, stream, out);
}
extern "C" int cdr_encoder_create_prec(const CdrEncoderSpec* spec, int precision, void* stream, CdrEncoder** out) {
  CDR_CHECK_ARG(spec && out, "cdr_encoder_create: null argument");
  CDR_CHECK_ARG(precision == CDR_PREC_BF16 || precision == CDR_PREC_F16X2,
                "cdr_encoder_create: precision must be CDR_PREC_BF16 or CDR_PREC_F16X2");
  CdrEncoder* e = new (std::nothrow) CdrEncoder();
  CDR_CHECK_ARG(e, "cdr_encoder_create: out of host memory");
  int rc = tc_encoder_create(*spec, precision == CDR_PREC_F16X2 ? 2 : 0, &e->impl, (cudaStream_t)stream);
  if (rc == CDR_OK && cudaStreamSynchronize((cudaStream_t)stream) != cudaSuccess) {
    set_error("cdr_encoder_create: packing failed: %s", cudaGetErrorString(cudaGetLastError()));
    rc = CDR_ERR_CUDA;
  }
  if (rc != CDR_OK) {
    tc_encoder_destroy(e->impl);
    delete e;
    return rc;
  }
  *out = e;
  return CDR_OK;
}
extern "C" int cdr_encoder_destroy(CdrEncoder* e) {
  if (!e) return CDR_OK;
  tc_encoder_destroy(e->impl);
  delete e;
  return CDR_OK;
}
extern "C" int cdr_encoder_workspace_bytes(const CdrEncoder* e, int n_images, int in_h, int in_w, size_t* bytes) {
  CDR_CHECK_ARG(e && bytes && n_images > 0 && in_h > 0 && in_w > 0, "cdr_encoder_workspace_bytes: bad args");
  return tc_encoder_workspace_bytes(e->impl, n_images, in_h, in_w, bytes);
}
extern "C" int cdr_encoder_out_bytes(const CdrEncoder* e, int n_images, int in_h, int in_w, size_t* bytes) {
  CDR_CHECK_ARG(e && bytes && n_images > 0 && in_h > 0 && in_w > 0, "cdr_encoder_out_bytes: bad args");
  return tc_encoder_out_bytes(e->impl, n_images, in_h, in_w, bytes);
}
extern "C" int cdr_encoder_out_shape(const CdrEncoder* e, int in_h, int in_w, int* out_h, int* out_w, int* out_c) {
  CDR_CHECK_ARG(e && out_h && out_w && out_c, "cdr_encoder_out_shape: bad args");
  return tc_encoder_out_shape(e->impl, in_h, in_w, out_h, out_w, out_c);
}
extern "C" int cdr_encoder_forward(const CdrEncoder* e, const void* x_nhwc_bf16, int n_images, int in_h, int in_w,
                                   void* out_rows_bf16, void* workspace, size_t workspace_bytes, void* stream) {
  CDR_CHECK_ARG(e && x_nhwc_bf16 && out_rows_bf16 && workspace && n_images > 0, "cdr_encoder_forward: bad args");
  CDR_CHECK_ARG(((uintptr_t)workspace & 255) == 0 && ((uintptr_t)x_nhwc_bf16 & 15) == 0 &&
                    ((uintptr_t)out_rows_bf16 & 15) == 0,
                "cdr_encoder_forward: workspace must be 256-byte, tensors 16-byte aligned");
  timing_restart();
  return tc_encoder_forward(e->impl, x_nhwc_bf16, n_images, in_h, in_w, out_rows_bf16, workspace, workspace_bytes,
                            (cudaStream_t)stream);
}
extern "C" int cdr_encoder_workspace_bytes_images(const CdrEncoder* e, int n_images, int img_h, int img_w,
                                                  size_t* bytes) {
  CDR_CHECK_ARG(e && bytes && n_images > 0 && img_h > 0 && img_w > 0, "cdr_encoder_workspace_bytes_images: bad args");
  return tc_encoder_workspace_bytes_images(e->impl, n_images, img_h, img_w, bytes);
}
extern "C" int cdr_encoder_forward_images(const CdrEncoder* e, const float* images, int n_images, int img_h, int img_w,
                                          void* out_rows_bf16, void* workspace, size_t workspace_bytes, void* stream) {
  CDR_CHECK_ARG(e && images && out_rows_bf16 && workspace && n_images > 0, "cdr_encoder_forward_images: bad args");
  CDR_CHECK_ARG(((uintptr_t)workspace & 255) == 0 && ((uintptr_t)images & 15) == 0 && ((uintptr_t)out_rows_bf16 & 15) == 0,
                "cdr_encoder_forward_images: workspace must be 256-byte, tensors 16-byte aligned");
  timing_restart();
  return tc_encoder_forward_images(e->impl, images, 0, nullptr, nullptr, n_images, img_h, img_w, out_rows_bf16, workspace,
                                   workspace_bytes, (cudaStream_t)stream);
}
extern "C" int cdr_encoder_forward_frames_u8(const CdrEncoder* e, const uint8_t* frames, const float* mean_host,
                                             const float* std_host, int n_images, int img_h, int img_w,
                                             void* out_rows_bf16, void* workspace, size_t workspace_bytes,
                                             void* stream) {
  CDR_CHECK_ARG(e && frames && mean_host && std_host && out_rows_bf16 && workspace && n_images > 0,
                "cdr_encoder_forward_frames_u8: bad args");
  CDR_CHECK_ARG(((uintptr_t)workspace & 255) == 0 && ((uintptr_t)out_rows_bf16 & 15) == 0,
                "cdr_encoder_forward_frames_u8: workspace must be 256-byte, output 16-byte aligned");
  timing_restart();
  return tc_encoder_forward_images(e->impl, frames, 1, mean_host, std_host, n_images, img_h, img_w, out_rows_bf16,
                                   workspace, workspace_bytes, (cudaStream_t)stream);
}

// Diagnostics: 16 host-mapped words; word 0 == 0xdeadbeef after an mbarrier wait inside a kernel timed out
// (then 1..6 = block, thread, shared-memory address of the barrier, parity, gridDim.x, blockDim.x).
extern "C" const unsigned int* cdr_debug_words(void) {
  if (!g_debug_host) {
    unsigned int* h = nullptr;
    if (cudaHostAlloc(&h, 16 * sizeof(unsigned int), cudaHostAllocMapped) != cudaSuccess) return nullptr;
    for (int i = 0; i < 16; ++i) h[i] = 0;
    unsigned int* d = nullptr;
    if (cudaHostGetDevicePointer(&d, h, 0) != cudaSuccess) return nullptr;
    if (tc_set_debug(d) != CDR_OK || heat_set_debug(d) != CDR_OK) return nullptr;
    g_debug_host = h;
  }
  return g_debug_host;
}

extern "C" int cdr_decoder_forward_rows(const CdrWeights* w, const void* feat_rows, int n_images, float* heatmaps,
                                        void* workspace, size_t workspace_bytes, void* stream) {
  CDR_CHECK_ARG(w && feat_rows && heatmaps && workspace && n_images > 0, "cdr_decoder_forward_rows: bad args");
  CDR_CHECK_ARG(w->precision != CDR_PREC_FP32, "cdr_decoder_forward_rows: needs a tensor-core precision");
  CDR_CHECK_ARG(((uintptr_t)workspace & 255) == 0 && ((uintptr_t)feat_rows & 15) == 0,
                "cdr_decoder_forward_rows: workspace must be 256-byte, features 16-byte aligned");
  timing_restart();
  return tc_decoder_forward(w->tc, feat_rows, 0, nullptr, n_images, heatmaps, workspace, workspace_bytes,
                            (cudaStream_t)stream);
}
extern "C" int cdr_decoder_forward_planes(const CdrWeights* w, const void* feat_planes, int n_images, float* heatmaps,
                                          void* workspace, size_t workspace_bytes, void* stream) {
  CDR_CHECK_ARG(w && feat_planes && heatmaps && workspace && n_images > 0, "cdr_decoder_forward_planes: bad args");
  CDR_CHECK_ARG(w->precision == CDR_PREC_F16X2, "cdr_decoder_forward_planes: needs the f16x2 (\"fp32\") precision");
  CDR_CHECK_ARG(((uintptr_t)workspace & 255) == 0 && ((uintptr_t)feat_planes & 255) == 0,
                "cdr_decoder_forward_planes: workspace must be 256-byte, the planes buffer 256-byte aligned");
  timing_restart();
  return tc_decoder_forward(w->tc, feat_planes, 1, nullptr, n_images, heatmaps, workspace, workspace_bytes,
                            (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------
// SURVEY 8f rank 3, second slice (train_ops.cu): train-mode BatchNorm2d and the reference's losses
extern "C" int cdr_bn_train_forward(const float* x, int n, int c, int hw, const float* gamma, const float* beta,
                                    double eps, double momentum, float* running_mean, float* running_var, int relu,
                                    float* y, float* save_mean, float* save_invstd, void* stream) {
  CDR_CHECK_ARG(x && y && save_mean && save_invstd && n > 0 && c > 0 && hw > 0, "cdr_bn_train_forward: bad args");
  CDR_CHECK_ARG((long long)n * hw > 1, "cdr_bn_train_forward: more than one value per channel expected (as torch)");
  return launch_bn_train_forward(x, n, c, hw, gamma, beta, eps, momentum, running_mean, running_var, relu, y, save_mean,
                                 save_invstd, (cudaStream_t)stream);
}
extern "C" int cdr_bn_train_backward(const float* x, const float* dy, int n, int c, int hw, const float* gamma,
                                     const float* beta, const float* save_mean, const float* save_invstd, int relu,
                                     float* dx, float* dgamma, float* dbeta, void* stream) {
  CDR_CHECK_ARG(x && dy && save_mean && save_invstd && dx && dgamma && dbeta && n > 0 && c > 0 && hw > 0,
                "cdr_bn_train_backward: bad args");
  return launch_bn_train_backward(x, dy, n, c, hw, gamma, beta, save_mean, save_invstd, relu, dx, dgamma, dbeta,
                                  (cudaStream_t)stream);
}
extern "C" size_t cdr_joint_loss_scratch_bytes(void) { return joint_loss_scratch_bytes(); }
extern "C" int cdr_joint_loss_forward(int kind, const float* pred, const float* target, const float* weight,
                                      long long rows, int d, double threshold, float* loss, void* scratch, void* stream) {
  CDR_CHECK_ARG(kind >= 0 && kind <= 2 && pred && target && loss && scratch && rows > 0 && d > 0,
                "cdr_joint_loss_forward: bad args");
  CDR_CHECK_ARG(((uintptr_t)scratch & 7) == 0, "cdr_joint_loss_forward: scratch must be 8-byte aligned");
  return launch_joint_loss_forward(kind, pred, target, weight, rows, d, threshold, loss, (double*)scratch,
                                   (cudaStream_t)stream);
}
extern "C" int cdr_joint_loss_backward(int kind, const float* pred, const float* target, const float* weight,
                                       long long rows, int d, double threshold, const float* grad_loss, float* grad_pred,
                                       void* stream) {
  CDR_CHECK_ARG(kind >= 0 && kind <= 2 && pred && target && grad_loss && grad_pred && rows > 0 && d > 0,
                "cdr_joint_loss_backward: bad args");
  return launch_joint_loss_backward(kind, pred, target, weight, rows, d, threshold, grad_loss, grad_pred,
                                    (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------
// Training convolutions (gemm_tc.cu: make_train_conv, tc_train_conv_*).  Each op keeps its own domain check and codes.
// The decoder's transposed convolutions:
static int deconv_train_shape(const char* fn, int n, int cin, int cout, int h, int w) {
  CDR_CHECK_ARG(n > 0 && cin > 0 && cout > 0 && h > 0 && w > 0, "%s: bad shape n=%d cin=%d cout=%d h=%d w=%d", fn, n, cin,
                cout, h, w);
  if (cin % 64 != 0 || cout % 64 != 0 || h != w || (w != 8 && w != 16 && w != 32)) {
    set_error("%s: unsupported shape cin=%d cout=%d h=%d w=%d (channels multiples of 64, h == w in {8, 16, 32})", fn,
              cin, cout, h, w);
    return CDR_ERR_UNSUPPORTED;
  }
  return CDR_OK;
}
// 1x1 convolutions:
static int conv1x1_train_shape(const char* fn, int n, int cin, int cout, int h, int w) {
  CDR_CHECK_ARG(n >= 1 && cin >= 1 && cin <= 4096 && cout >= 1 && cout <= 4096 && h >= 1 && w >= 1 &&
                    ((long long)h * w) % 64 == 0 && (long long)n * h * w <= (1LL << 22),
                "%s: unsupported shape n=%d cin=%d cout=%d h=%d w=%d (1 <= Cin, Cout <= 4096, h*w a multiple of 64, "
                "n*h*w <= 2^22)", fn, n, cin, cout, h, w);
  return CDR_OK;
}
// 3x3 convolutions.  h, w: the input map.  The output map's H*W must be 64 or a multiple of 128: the tap-GEMM's
// 128-pixel tile is one 4-D box of whole rows (or of two whole 64-pixel images).
static int conv3x3_train_shape(const char* fn, int n, int cin, int cout, int h, int w, int stride) {
  const bool s_ok = stride == 1 || stride == 2;
  const bool c_ok = cin >= 64 && cin <= 2048 && cin % 64 == 0 && cout >= 64 && cout <= 2048 && cout % 64 == 0;
  const bool g_ok = s_ok && h >= 1 && w >= 1 && h % stride == 0 && w % stride == 0;
  const long long ho = g_ok ? h / stride : 0, wo = g_ok ? w / stride : 0, hw = ho * wo;
  const bool o_ok = g_ok && (wo == 8 || wo == 16 || wo == 32 || wo == 64) && (hw == 64 || hw % 128 == 0);
  CDR_CHECK_ARG(n >= 1 && c_ok && o_ok && (long long)n * hw <= (1LL << 22),
                "%s: unsupported shape n=%d cin=%d cout=%d h=%d w=%d stride=%d (stride 1 or 2, Cin and Cout multiples of 64 "
                "in [64, 2048], h and w divisible by the stride; output W a power of two in [8, 64], output H*W = 64 or a "
                "multiple of 128, n*H*W <= 2^22)", fn, n, cin, cout, h, w, stride);
  return CDR_OK;
}

// The stem's 7x7 stride-2 pad-3 convolution (stem.cu).  h, w: the input images.
static int stem_train_shape(const char* fn, int n, int cin, int cout, int h, int w) {
  CDR_CHECK_ARG(n >= 1 && cin == 3 && cout == 64 && h >= 16 && w >= 64 && h % 16 == 0 && w % 64 == 0 &&
                    (long long)n * (h / 2) * (w / 2) <= (1LL << 22),
                "%s: unsupported shape n=%d cin=%d cout=%d h=%d w=%d (Cin = 3, Cout = 64, h %% 16 == 0, w %% 64 == 0, "
                "n*(h/2)*(w/2) <= 2^22)", fn, n, cin, cout, h, w);
  return CDR_OK;
}

static int train_null_args(const char* fn, std::initializer_list<const void*> need) {
  for (const void* p : need) CDR_CHECK_ARG(p, "%s: null pointer", fn);
  return CDR_OK;
}
// The tensors are 16-byte aligned (null allowed: an output not wanted), the bias 4-byte, saved and the workspace
// 256-byte, and saved holds the forward's x planes (saved_bytes = SIZE_MAX: the backward, which has no size to check).
static int train_buffer_args(const char* fn, std::initializer_list<const void*> tensors, const void* bias, bool bias_note,
                             const void* saved, size_t saved_bytes, size_t saved_need, const void* workspace) {
  bool aligned = ((uintptr_t)bias & 3) == 0 && ((uintptr_t)saved & 255) == 0 && ((uintptr_t)workspace & 255) == 0;
  for (const void* p : tensors) aligned = aligned && ((uintptr_t)p & 15) == 0;
  CDR_CHECK_ARG(aligned, "%s: tensors must be 16-byte%s, saved / workspace 256-byte aligned", fn,
                bias_note ? " (bias 4-byte)" : "");
  if (saved_bytes != SIZE_MAX && saved_bytes < saved_need) {
    set_error("%s: saved %zu < required %zu bytes", fn, saved_bytes, saved_need);
    return CDR_ERR_WORKSPACE;
  }
  return CDR_OK;
}

// What every cdr_<op>_train_* entry point checks, in this order: the pointers in `need` are not null, the shape is in
// the op's domain, then train_buffer_args.  On success *d describes the op.
static int train_conv_args(const char* fn, int kind, int n, int cin, int cout, int h, int w, int stride,
                           std::initializer_list<const void*> need, std::initializer_list<const void*> tensors,
                           const void* bias, const void* saved, size_t saved_bytes, const void* workspace, TrainConv* d) {
  if (int rc = train_null_args(fn, need)) return rc;
  const int rc = kind == kTrainDeconv    ? deconv_train_shape(fn, n, cin, cout, h, w)
                 : kind == kTrainConv1x1 ? conv1x1_train_shape(fn, n, cin, cout, h, w)
                                         : conv3x3_train_shape(fn, n, cin, cout, h, w, stride);
  if (rc) return rc;
  *d = make_train_conv(kind, n, cin, cout, h, w, stride);
  return train_buffer_args(fn, tensors, bias, kind == kTrainConv1x1, saved, saved_bytes, train_conv_saved_bytes(*d),
                           workspace);
}
static int stem_train_args(const char* fn, int n, int cin, int cout, int h, int w, std::initializer_list<const void*> need,
                           std::initializer_list<const void*> tensors, const void* saved, size_t saved_bytes,
                           const void* workspace) {
  if (int rc = train_null_args(fn, need)) return rc;
  if (int rc = stem_train_shape(fn, n, cin, cout, h, w)) return rc;
  return train_buffer_args(fn, tensors, nullptr, false, saved, saved_bytes, stem_train_saved_bytes(n, h, w), workspace);
}
static int train_conv_sizes(const char* fn, int kind, int n, int cin, int cout, int h, int w, int stride,
                            size_t* saved_bytes, size_t* workspace_bytes) {
  TrainConv d;
  if (int rc = train_conv_args(fn, kind, n, cin, cout, h, w, stride, {saved_bytes, workspace_bytes}, {}, nullptr, nullptr,
                               SIZE_MAX, nullptr, &d))
    return rc;
  *saved_bytes = train_conv_saved_bytes(d);
  *workspace_bytes = train_conv_workspace_bytes(d);
  return CDR_OK;
}
static int train_conv_forward(const char* fn, int kind, const float* x, const float* weight, const float* bias, int n,
                              int cin, int cout, int h, int w, int stride, float* y, void* saved, size_t saved_bytes,
                              void* workspace, size_t workspace_bytes, void* stream) {
  TrainConv d;
  if (int rc = train_conv_args(fn, kind, n, cin, cout, h, w, stride, {x, weight, y, saved, workspace}, {x, weight, y},
                               bias, saved, saved_bytes, workspace, &d))
    return rc;
  return tc_train_conv_forward(d, x, weight, bias, y, saved, workspace, workspace_bytes, (cudaStream_t)stream);
}
static int train_conv_backward(const char* fn, int kind, const void* saved, const float* weight, const float* dy, int n,
                               int cin, int cout, int h, int w, int stride, float* dx, float* dweight, float* dbias,
                               void* workspace, size_t workspace_bytes, void* stream) {
  TrainConv d;
  if (int rc = train_conv_args(fn, kind, n, cin, cout, h, w, stride, {saved, weight, dy, workspace},
                               {weight, dy, dx, dweight}, dbias, saved, SIZE_MAX, workspace, &d))
    return rc;
  return tc_train_conv_backward(d, saved, weight, dy, dx, dweight, dbias, workspace, workspace_bytes,
                                (cudaStream_t)stream);
}

extern "C" int cdr_deconv_train_workspace_bytes(int n, int cin, int cout, int h, int w, size_t* saved_bytes,
                                                size_t* workspace_bytes) {
  return train_conv_sizes("cdr_deconv_train_workspace_bytes", kTrainDeconv, n, cin, cout, h, w, 1, saved_bytes,
                          workspace_bytes);
}
extern "C" int cdr_deconv_train_forward(const float* x, const float* weight, int n, int cin, int cout, int h, int w,
                                        float* y, void* saved, size_t saved_bytes, void* workspace,
                                        size_t workspace_bytes, void* stream) {
  return train_conv_forward("cdr_deconv_train_forward", kTrainDeconv, x, weight, nullptr, n, cin, cout, h, w, 1, y, saved,
                            saved_bytes, workspace, workspace_bytes, stream);
}
extern "C" int cdr_deconv_train_backward(const void* saved, const float* weight, const float* dy, int n, int cin,
                                         int cout, int h, int w, float* dx, float* dweight, void* workspace,
                                         size_t workspace_bytes, void* stream) {
  return train_conv_backward("cdr_deconv_train_backward", kTrainDeconv, saved, weight, dy, n, cin, cout, h, w, 1, dx,
                             dweight, nullptr, workspace, workspace_bytes, stream);
}

extern "C" int cdr_conv1x1_train_workspace_bytes(int n, int cin, int cout, int h, int w, size_t* saved_bytes,
                                                 size_t* workspace_bytes) {
  return train_conv_sizes("cdr_conv1x1_train_workspace_bytes", kTrainConv1x1, n, cin, cout, h, w, 1, saved_bytes,
                          workspace_bytes);
}
extern "C" int cdr_conv1x1_train_forward(const float* x, const float* weight, const float* bias, int n, int cin,
                                         int cout, int h, int w, float* y, void* saved, size_t saved_bytes,
                                         void* workspace, size_t workspace_bytes, void* stream) {
  return train_conv_forward("cdr_conv1x1_train_forward", kTrainConv1x1, x, weight, bias, n, cin, cout, h, w, 1, y, saved,
                            saved_bytes, workspace, workspace_bytes, stream);
}
extern "C" int cdr_conv1x1_train_backward(const void* saved, const float* weight, const float* dy, int n, int cin,
                                          int cout, int h, int w, float* dx, float* dweight, float* dbias,
                                          void* workspace, size_t workspace_bytes, void* stream) {
  return train_conv_backward("cdr_conv1x1_train_backward", kTrainConv1x1, saved, weight, dy, n, cin, cout, h, w, 1, dx,
                             dweight, dbias, workspace, workspace_bytes, stream);
}

extern "C" int cdr_conv3x3_train_workspace_bytes(int n, int cin, int cout, int h, int w, int stride, size_t* saved_bytes,
                                                 size_t* workspace_bytes) {
  return train_conv_sizes("cdr_conv3x3_train_workspace_bytes", kTrainConv3x3, n, cin, cout, h, w, stride, saved_bytes,
                          workspace_bytes);
}
extern "C" int cdr_conv3x3_train_forward(const float* x, const float* weight, int n, int cin, int cout, int h, int w,
                                         int stride, float* y, void* saved, size_t saved_bytes, void* workspace,
                                         size_t workspace_bytes, void* stream) {
  return train_conv_forward("cdr_conv3x3_train_forward", kTrainConv3x3, x, weight, nullptr, n, cin, cout, h, w, stride, y,
                            saved, saved_bytes, workspace, workspace_bytes, stream);
}
extern "C" int cdr_conv3x3_train_backward(const void* saved, const float* weight, const float* dy, int n, int cin,
                                          int cout, int h, int w, int stride, float* dx, float* dweight, void* workspace,
                                          size_t workspace_bytes, void* stream) {
  return train_conv_backward("cdr_conv3x3_train_backward", kTrainConv3x3, saved, weight, dy, n, cin, cout, h, w, stride,
                             dx, dweight, nullptr, workspace, workspace_bytes, stream);
}

extern "C" int cdr_stem_train_workspace_bytes(int n, int cin, int cout, int h, int w, size_t* saved_bytes,
                                              size_t* workspace_bytes) {
  const char* fn = "cdr_stem_train_workspace_bytes";
  if (int rc = stem_train_args(fn, n, cin, cout, h, w, {saved_bytes, workspace_bytes}, {}, nullptr, SIZE_MAX, nullptr))
    return rc;
  *saved_bytes = stem_train_saved_bytes(n, h, w);
  *workspace_bytes = stem_train_workspace_bytes(n, h, w);
  return CDR_OK;
}
extern "C" int cdr_stem_train_forward(const float* x, const float* weight, int n, int cin, int cout, int h, int w, float* y,
                                      void* saved, size_t saved_bytes, void* workspace, size_t workspace_bytes,
                                      void* stream) {
  const char* fn = "cdr_stem_train_forward";
  if (int rc = stem_train_args(fn, n, cin, cout, h, w, {x, weight, y, saved, workspace}, {x, weight, y}, saved, saved_bytes,
                               workspace))
    return rc;
  return launch_stem_train_forward(x, weight, n, h, w, y, saved, workspace, workspace_bytes, (cudaStream_t)stream);
}
extern "C" int cdr_stem_train_backward(const void* saved, const float* weight, const float* dy, int n, int cin, int cout,
                                       int h, int w, float* dx, float* dweight, void* workspace, size_t workspace_bytes,
                                       void* stream) {
  const char* fn = "cdr_stem_train_backward";
  CDR_CHECK_ARG(!dx, "%s: the stem has no input gradient (its input is the image batch): dx must be NULL", fn);
  if (int rc = stem_train_args(fn, n, cin, cout, h, w, {saved, weight, dy, workspace}, {weight, dy, dweight}, saved,
                               SIZE_MAX, workspace))
    return rc;
  return launch_stem_train_backward(saved, dy, n, h, w, dweight, workspace, workspace_bytes, (cudaStream_t)stream);
}

// ------------------------------------------------------------------------------------------
// The stem's 3x3 stride-2 pad-1 max-pool in training (stem.cu)
static int maxpool3x3_train_args(const char* fn, const void* argmax, const float* a, const float* b, int n, int c, int h,
                                 int w) {
  if (int rc = train_null_args(fn, {argmax, a, b})) return rc;
  CDR_CHECK_ARG(n >= 1 && c >= 1 && h >= 1 && w >= 1 && (long long)n * c * h * w < (1LL << 31),
                "%s: unsupported shape n=%d c=%d h=%d w=%d (every size >= 1, n*c*h*w < 2^31)", fn, n, c, h, w);
  CDR_CHECK_ARG(((uintptr_t)a & 3) == 0 && ((uintptr_t)b & 3) == 0, "%s: fp32 tensors must be 4-byte aligned", fn);
  return CDR_OK;
}
extern "C" int cdr_maxpool3x3_train_forward(const float* x, int n, int c, int h, int w, float* y, uint8_t* argmax,
                                            void* stream) {
  if (int rc = maxpool3x3_train_args("cdr_maxpool3x3_train_forward", argmax, x, y, n, c, h, w)) return rc;
  return launch_maxpool3x3_train_forward(x, n, c, h, w, y, argmax, (cudaStream_t)stream);
}
extern "C" int cdr_maxpool3x3_train_backward(const uint8_t* argmax, const float* dy, int n, int c, int h, int w, float* dx,
                                             void* stream) {
  if (int rc = maxpool3x3_train_args("cdr_maxpool3x3_train_backward", argmax, dy, dx, n, c, h, w)) return rc;
  return launch_maxpool3x3_train_backward(argmax, dy, n, c, h, w, dx, (cudaStream_t)stream);
}
