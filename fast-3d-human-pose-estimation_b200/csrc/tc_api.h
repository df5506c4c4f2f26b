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

// Training a ConvTranspose2d(k4, s2, p1, bias=False) at fp32 accuracy (f16x2) — gemm_tc.cu
size_t deconv_train_saved_bytes(int n, int cin, int cout, int h, int w);
size_t deconv_train_workspace_bytes(int n, int cin, int cout, int h, int w);
int tc_deconv_train_forward(const float* x, const float* weight, int n, int cin, int cout, int h, int w, float* y,
                            void* saved, void* workspace, size_t workspace_bytes, cudaStream_t st);
int tc_deconv_train_backward(const void* saved, const float* weight, const float* dy, int n, int cin, int cout, int h,
                             int w, float* dx, float* dw, void* workspace, size_t workspace_bytes, cudaStream_t st);

// Training a 1x1 Conv2d(Cin, Cout, bias optional) at fp32 accuracy (f16x2) — gemm_tc.cu
size_t conv1x1_train_saved_bytes(int n, int cin, int cout, int h, int w);
size_t conv1x1_train_workspace_bytes(int n, int cin, int cout, int h, int w);
int tc_conv1x1_train_forward(const float* x, const float* weight, const float* bias, int n, int cin, int cout, int h,
                             int w, float* y, void* saved, void* workspace, size_t workspace_bytes, cudaStream_t st);
int tc_conv1x1_train_backward(const void* saved, const float* weight, const float* dy, int n, int cin, int cout, int h,
                              int w, float* dx, float* dw, float* db, void* workspace, size_t workspace_bytes,
                              cudaStream_t st);

// Training a 3x3 pad-1 Conv2d(Cin, Cout, stride 1 or 2, bias=False) at fp32 accuracy (f16x2) — gemm_tc.cu
size_t conv3x3_train_saved_bytes(int n, int cin, int cout, int h, int w, int stride);
size_t conv3x3_train_workspace_bytes(int n, int cin, int cout, int h, int w, int stride);
int tc_conv3x3_train_forward(const float* x, const float* weight, int n, int cin, int cout, int h, int w, int stride,
                             float* y, void* saved, void* workspace, size_t workspace_bytes, cudaStream_t st);
int tc_conv3x3_train_backward(const void* saved, const float* weight, const float* dy, int n, int cin, int cout, int h,
                              int w, int stride, float* dx, float* dw, void* workspace, size_t workspace_bytes,
                              cudaStream_t st);

}  // namespace cdr
