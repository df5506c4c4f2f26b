// Internal launcher declarations shared by the translation units of libcdrhead.so.
#pragma once
#include "common.cuh"

namespace cdr {

enum OutMode { kOutRows = 0, kOutDeconv = 1, kOutPlanar = 2 };

// One "tap-GEMM" problem (see gemm_ffma.cu / gemm_tc.cu for the arithmetic).
struct TapGemmParams {
  const void* A;            // pixel-major activations (n_img, H, W, a_pitch); fp32 or bf16
  long long a_group_stride; // elements between groups (non-deconv grouped launches)
  int a_pitch;              // channel pitch in elements
  int n_img, H, W;          // M = n_img*H*W
  int cin;                  // K per tap
  int deconv;               // 1: 4 taps, group index = output phase (py*2+px)
  const void* Wp;           // packed weights, layout depends on the path (pack.cu)
  long long w_group_stride; // elements between groups / phases
  const float* bias;        // (groups, n_pad) folded bias, fp32
  int bias_group_stride;
  int n_pad;                // padded output channels of the packed weights
  int n;                    // valid output channels
  void* C;
  long long c_group_stride;
  int c_pitch;              // output row pitch (elements) for kOutRows / kOutDeconv
  int c_fill;               // columns [n, c_fill) are written as zeros
  int relu;
  int out_mode;
};

int launch_tap_gemm_ffma(const TapGemmParams& p, int groups, cudaStream_t st);

// layout.cu
// in2 (may be NULL): a second (n_img, C, HW) tensor converted by the same launch; its rows follow in `out`
int launch_nchw_to_rows_f32(const float* in, const float* in2, int n_img, int C, int HW, float* out, int out_pitch,
                            cudaStream_t st);
int launch_nchw_to_rows_bf16(const float* in, const float* in2, int n_img, int C, int HW, __nv_bfloat16* out,
                             int out_pitch, cudaStream_t st);
// fp32 hi/lo planes for the 3xTF32 tensor-core path (common.cuh: split_tf32)
int launch_nchw_to_rows_split(const float* in, const float* in2, int n_img, int C, int HW, float* out_hi, float* out_lo,
                              int out_pitch, cudaStream_t st);
// FTL of `views` (1 or 2) tensors in one launch
int launch_ftl_split2(const float* const in_hi[2], const float* const in_lo[2], int in_pitch, const float* const mats[2],
                      int rows, int cols, int blk, int n, int hw, float* const out_hi[2], float* const out_lo[2],
                      int out_pitch, int out_fill, int views, cudaStream_t st);
int launch_ftl_f16p2(const void* const in_hi[2], const void* const in_lo[2], int in_pitch, const float* const mats[2],
                     int rows, int cols, int blk, int n, int hw, void* const out_hi[2], void* const out_lo[2],
                     int out_pitch, int out_fill, const float* scale_in, const float* amax_in, const float* l1max,
                     float* scale_out, float* amax_out, cudaStream_t st);
int launch_mats_l1max(const float* a0, const float* a1, int ra, int ca, const float* b0, const float* b1, int rb, int cb,
                      int n, float* out, cudaStream_t st);
template <typename T>
int launch_ftl2(const T* const in[2], int in_pitch, const float* const mats[2], int rows, int cols, int blk, int n,
                int hw, T* const out[2], int out_pitch, int out_fill, int views, cudaStream_t st);
// pinv of two (n,3,4) stacks in one launch: out[0..n) from P_a, out[n..2n) from P_b
int launch_pinv2(const float* P_a, const float* P_b, int n, double rtol, float* out, float* l1max, cudaStream_t st);
// scaled fp16 hi/lo planes for the f16x2 tensor-core path (gemm_tc.cu: kFmtF16P)
int launch_amax_f32(const float* in, const float* in2, long long n, float* amax, cudaStream_t st);   // in2 may be NULL
int launch_nchw_to_rows_f16p(const float* in, const float* in2, int n_img, int C, int HW, void* out_hi, void* out_lo,
                             int out_pitch, const float* amax, float* scale_out, cudaStream_t st);
bool nchw_rowscale_ok(const float* in, const float* in2, int n_img, int C, int HW, int out_pitch);
int launch_nchw_to_rows_f16p_rowscale(const float* in, const float* in2, int n_img, int C, int HW, void* out_hi,
                                      void* out_lo, int out_pitch, float* row_scale, float* amax_out, cudaStream_t st);
template <typename T>
int launch_ftl(const T* in, int in_pitch, const float* mats, int rows, int cols, int blk, int n,
               int hw, T* out, int out_pitch, int out_fill, cudaStream_t st);

// pack.cu: BN folding + re-layout of the reference's parameter tensors
//   conv 1x1 (Cout,Cin) -> fp32 [k_pad][n_pad] (rows k >= Cin and cols n >= Cout zero)
int launch_pack_conv1x1_f32(const CdrConvBn& src, int cout, int cin, int k_pad, int n_pad,
                            float* w_out, float* bias_out, cudaStream_t st);
//   deconv (Cin,Cout,4,4) -> fp32 [phase][tap][Cin][n_pad]
int launch_pack_deconv_f32(const CdrConvBn& src, int cin, int cout, int n_pad, float* w_out,
                           float* bias_out, cudaStream_t st);

// stem.cu: ResNet stem (conv 7x7 s2 + BN + ReLU, max-pool 3x3 s2), fp32 NCHW -> bf16 NHWC
int launch_pack_stem(const CdrConvBn& s, void* w, float* bias, cudaStream_t st);
size_t stem_weight_bytes();
// x: fp32 NCHW (is_u8 = 0) or uint8 NHWC frames normalised on the fly with HOST arrays mean[3], std[3]
int launch_stem(const void* x, int is_u8, const float* mean, const float* std, int n, int H, int W, const void* w,
                const float* bias, void* conv_out, void* pooled, cudaStream_t st);
// the same at fp32 accuracy (fp16 hi/lo operands on mma.sync): weights as fp16 hi/lo planes + per-channel scales,
// conv_out fp32 NHWC scratch, pooled as scaled fp16 hi/lo planes; slot = {amax, scale} of the pooled tensor (amax pre-zeroed)
int launch_pack_stem_f16x2(const CdrConvBn& s, void* w, float* bias, cudaStream_t st);
size_t stem_weight_bytes_f16x2();
int launch_stem_f32(const void* x, int is_u8, const float* mean, const float* std, int n, int H, int W, const void* w,
                    const float* bias, float* conv_out, void* pooled_hi, void* pooled_lo, float* slot, cudaStream_t st);
// training (include/cdrhead.h: cdr_stem_train_*, cdr_maxpool3x3_train_*); the shape must be in the op's domain
size_t stem_train_saved_bytes(int n, int H, int W);
size_t stem_train_workspace_bytes(int n, int H, int W);
int stem_train_slices(int n, int H, int W);
int launch_stem_train_forward(const float* x, const float* weight, int n, int H, int W, float* y, void* saved,
                              void* workspace, size_t workspace_bytes, cudaStream_t st);
int launch_stem_train_backward(const void* saved, const float* dy, int n, int H, int W, float* dweight, void* workspace,
                               size_t workspace_bytes, cudaStream_t st);
int launch_maxpool3x3_train_forward(const float* x, int n, int c, int H, int W, float* y, uint8_t* argmax, cudaStream_t st);
int launch_maxpool3x3_train_backward(const uint8_t* argmax, const float* dy, int n, int c, int H, int W, float* dx,
                                     cudaStream_t st);

// gemm_tc.cu: dw[r][c][tap] = (sum over slices, in order, of part[slice][tap][r][c]) / (*sx * *sdy), part rows ldc apart
int launch_wgrad_reduce(const float* part, int slices, int taps, int rows, int cols, int ldc, const float* sx,
                        const float* sdy, float* dw, cudaStream_t st);

// train_ops.cu: BatchNorm2d in training mode (+ optional fused ReLU) and the reference's three losses, forward / backward
int launch_bn_train_forward(const float* x, int n, int c, int hw, const float* gamma, const float* beta, double eps,
                            double momentum, float* running_mean, float* running_var, int relu, float* y, float* save_mean,
                            float* save_invstd, cudaStream_t st);
int launch_bn_train_backward(const float* x, const float* dy, int n, int c, int hw, const float* gamma, const float* beta,
                             const float* save_mean, const float* save_invstd, int relu, float* dx, float* dgamma,
                             float* dbeta, cudaStream_t st);
int launch_joint_loss_forward(int kind, const float* pred, const float* target, const float* weight, long long rows, int D,
                              double threshold, float* loss, double* scratch, cudaStream_t st);
int launch_joint_loss_backward(int kind, const float* pred, const float* target, const float* weight, long long rows, int D,
                               double threshold, const float* grad_loss, float* grad_pred, cudaStream_t st);
size_t joint_loss_scratch_bytes();

}  // namespace cdr
