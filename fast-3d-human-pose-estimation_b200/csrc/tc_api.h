// Interface between api.cu and the bf16 tensor-core path (gemm_tc.cu).
#pragma once
#include "kernels.h"

namespace cdr {

struct TcWeights {
  void* pool = nullptr;   // one cudaMalloc holding every packed layer
  void* impl = nullptr;   // TcPack (gemm_tc.cu): per-layer pointers + weight tensor maps
  int joints = 0, has_fusion = 0, fin_npad = 0;
  int kind = 0;           // pack mode: 0 = bf16, 1 = tf32x3, 2 = f16x2 (gemm_tc.cu: TcMode)
  FusionDims fd;          // fusion widths (common.cuh)
};

int tc_weights_create(const CdrWeightPtrs& src, int mode, TcWeights& w, cudaStream_t st);
void tc_weights_destroy(TcWeights& w);
int tc_head_workspace_bytes(const TcWeights& w, int batch, size_t* bytes);
int tc_decoder_workspace_bytes(const TcWeights& w, int n_images, size_t* bytes);
// feat_rows != NULL: latents given as pixel-major rows (2*batch*64, 2048), left view first — bf16 (feat_planes = 0)
// or an "fp16 planes" buffer [hi | lo | {amax, scale}] (feat_planes = 1, include/cdrhead.h)
int tc_head_forward(const TcWeights& w, const void* feat_rows, int feat_planes, const float* feat_l, const float* feat_r,
                    const float* P_l, const float* P_r, const float* pinv_l, const float* pinv_r, double pinv_rtol,
                    int batch, float scale, float* kp2d_l, float* kp2d_r, float* xyz,
                    const CdrHeadTaps* taps, void* workspace, size_t workspace_bytes,
                    cudaStream_t st);
int tc_decoder_forward(const TcWeights& w, const void* feat_rows, int feat_planes, const float* feat, int n_images,
                       float* heatmaps, void* workspace, size_t workspace_bytes, cudaStream_t st);

// ResNet bottleneck encoder (tcgen05; kind 0 = bf16 rows, 2 = f16x2: scaled fp16 hi/lo planes) — gemm_tc.cu
int tc_encoder_create(const CdrEncoderSpec& spec, int kind, void** out, cudaStream_t st);
int tc_encoder_kind(const void* enc);
int tc_encoder_out_bytes(const void* enc, int n, int h, int w, size_t* bytes);
void tc_encoder_destroy(void* enc);
int tc_encoder_workspace_bytes(const void* enc, int n, int h, int w, size_t* bytes);
int tc_encoder_workspace_bytes_images(const void* enc, int n, int H, int W, size_t* bytes);
int tc_encoder_forward_images(const void* enc, const void* images, int is_u8, const float* mean, const float* std,
                              int n, int H, int W, void* out_rows, void* workspace, size_t workspace_bytes,
                              cudaStream_t st);
int tc_encoder_out_shape(const void* enc, int h, int w, int* oh, int* ow, int* oc);
int tc_encoder_forward(const void* enc, const void* x, int n, int h, int w, void* out_rows, void* workspace,
                       size_t workspace_bytes, cudaStream_t st);

// Training convolutions at fp32 accuracy (f16x2) — gemm_tc.cu.  make_train_conv is the only code that maps an op onto
// the tap-GEMM; the planner, the size functions, the forward and the backward read the descriptor alone.
enum TrainConvKind { kTrainDeconv, kTrainConv1x1, kTrainConv3x3 };
struct TcLayer;
struct TrainPlanes { int c, h, w, pitch; };   // x or dy as fp16 planes: c channels of an n x h x w map, rows `pitch` apart
// the forward (A = the x planes) or data-gradient (A = the dy planes) GEMM; B = the weight packed per call by `pack`
struct TrainGemm {
  void (*pack)(const CdrConvBn& s, int nout, int cin, const TcLayer& L, cudaStream_t st);
  int k, bn, n_pad, groups;  // packed layer: groups * n_pad rows of k (groups = 4: one per output phase of kTapDeconv)
  int tap, stride, H, W, n;  // TapMode (gemm_tc.cu), A box stride, pixel grid (TcLaunch::H, W), output channels
};
struct TrainConv {
  int kind, n;
  TrainPlanes x, dy;
  TrainGemm fwd, dgrad;
  bool wgrad_a_is_x;         // wgrad A = x, B = dy (transposed conv) or A = dy, B = x (convs): the summation order
  int b_k, b_stride;         // wgrad B through the stride-b_stride box, b_k x b_k taps (b_k = 1: a plain 2-D map)
  int slices;                // wgrad K slices
};
// h, w: the input map; stride: the 3x3 conv's (1 or 2).  The shape must be in the op's domain.
TrainConv make_train_conv(int kind, int n, int cin, int cout, int h, int w, int stride);
size_t train_conv_saved_bytes(const TrainConv& d);
size_t train_conv_workspace_bytes(const TrainConv& d);
int tc_train_conv_forward(const TrainConv& d, const float* x, const float* weight, const float* bias, float* y,
                          void* saved, void* workspace, size_t workspace_bytes, cudaStream_t st);
int tc_train_conv_backward(const TrainConv& d, const void* saved, const float* weight, const float* dy, float* dx,
                           float* dw, float* db, void* workspace, size_t workspace_bytes, cudaStream_t st);

}  // namespace cdr
