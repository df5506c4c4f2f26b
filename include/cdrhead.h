/*
 * cdrhead.h — C ABI of libcdrhead.so: the CDRNet post-backbone hot path on B200 (sm_100a).
 *
 * The reference (eddie0509tw/Fast-3D-Human-Pose-Estimation) is pure Python and has no
 * FFI layer; the interfaces this library stands behind are Python call signatures
 * (SURVEY.md §8b).  Each entry point below names the reference lines it replaces.
 * The Python shim in fast-3d-human-pose-estimation_b200/ binds these with ctypes and
 * re-creates the reference's `CDRNet.forward`, `PoseResNet.forward`, `calc_mpjpe`,
 * `get_max_preds` and `triangulation` signatures on top (INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless its name ends in `_host`;
 *   - `stream` is a cudaStream_t passed as void*; every call is asynchronous on it and
 *     performs no allocation, no synchronisation and no host<->device copy, so the calls
 *     can be captured into a CUDA graph;  cdr_weights_create/destroy are the exception
 *     (they allocate / free and synchronise the stream they are given);
 *   - every function returns 0 on success or a CdrStatus code; cdr_last_error() returns a
 *     thread-local message for the last non-zero return.  No partial output is defined
 *     after an error;
 *   - there is NO CPU fallback: without a CUDA device every compute entry point fails
 *     with CDR_ERR_CUDA.
 *
 * HBM layouts
 *   - encoder features / heat-maps: NCHW, exactly as torch produces / the reference
 *     returns them;
 *   - projection matrices: (B,3,4) row-major fp32, pseudo-inverses (B,4,3);
 *   - 2D joints (B,J,2) fp32 in image pixels (x,y); 3D joints (B,J,3) fp32;
 *   - intermediates inside the workspace are pixel-major ("NHWC") — see DESIGN.md.
 */
#ifndef CDRHEAD_H_
#define CDRHEAD_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif
#if defined(__GNUC__)
#pragma GCC visibility push(default) /* the library is built with -fvisibility=hidden */
#endif

#define CDRHEAD_ABI_VERSION 1

typedef enum CdrStatus {
  CDR_OK = 0,
  CDR_ERR_INVALID = 1,   /* bad argument (null pointer, size, alignment, unsupported shape) */
  CDR_ERR_CUDA = 2,      /* a CUDA runtime call or kernel launch failed */
  CDR_ERR_WORKSPACE = 3, /* workspace too small */
  CDR_ERR_UNSUPPORTED = 4
} CdrStatus;

/* Arithmetic the convolutions run in.  Soft-argmax, pinv, DLT and MPJPE always use
 * fp32 inputs with fp64 internals. */
typedef enum CdrPrecision {
  CDR_PREC_FP32 = 0,  /* fp32 FFMA implicit-GEMM kernels (CUDA cores) */
  CDR_PREC_BF16 = 1,  /* bf16 operands on tcgen05 tensor cores, fp32 accumulation in TMEM */
  CDR_PREC_TF32X3 = 2,/* fp32 accuracy on tcgen05: every operand split into two tf32 terms,
                         three kind::tf32 MMAs per product, fp32 accumulation in TMEM */
  CDR_PREC_F16X2 = 3  /* fp32 accuracy on tcgen05 at the full 16-bit rate: decoder operands as two
                         scaled fp16 terms (data-dependent power-of-two tensor scales), three
                         kind::f16 MMAs per product; the fusion block stays 3xTF32 */
} CdrPrecision;

/* One conv (or transposed conv) + eval-mode BatchNorm2d, reference tensor layouts. */
typedef struct CdrConvBn {
  const float* weight;   /* Conv2d: (Cout,Cin,1,1);  ConvTranspose2d: (Cin,Cout,4,4) */
  const float* bias;     /* (Cout) or NULL (the transposed convs have bias=False)   */
  const float* bn_weight;
  const float* bn_bias;
  const float* bn_mean;
  const float* bn_var;   /* all (Cout); NULL bn_weight => no BN (final_layer)         */
} CdrConvBn;

/* The head's parameters in the reference's state_dict order (SURVEY.md Appendix B).
 * models/cdrnet.py:17-43 (CF.*) and models/decoder.py:8-21 (decoder.*).
 * A decoder-only handle (PoseResNet, models/poseresnet.py:17-21) sets has_fusion = 0. */
typedef struct CdrWeightPtrs {
  int num_joints;        /* cfg.MODEL.NUM_JOINTS (19 for MADS) */
  int has_fusion;
  CdrConvBn cf_conv1;    /* CF.conv_layer1.{0,1}: 2048 -> 300             */
  CdrConvBn cf_conv2a;   /* CF.conv_layer2.{0,1}:  800 -> 400             */
  CdrConvBn cf_conv2b;   /* CF.conv_layer2.{3,4}:  400 -> 400             */
  CdrConvBn cf_out[2];   /* CF.out_layer.{0,1}.{0,1}: 300 -> 2048 per view */
  CdrConvBn deconv[3];   /* decoder.deconv{1,2,3}.{0,1}                    */
  CdrConvBn final_layer; /* decoder.final_layer: 256 -> J, bias, no BN     */
  /* CDRNet(cfg, fusion_hid_ch1=.., fusion_hid_ch2=..), models/cdrnet.py:89-101.  0 / 0 = the defaults 300 / 400.  The
   * reference's forward only type-checks when hid_ch2 = 4/3 hid_ch1 (ftl maps 3 channel blocks to 4 and back,
   * :45-56,65,79); this library also needs hid_ch1 % 12 == 0 (block size a multiple of 4).  n_views and fusion_in_dim
   * are not parameters here: the reference itself only runs with n_views = 2 (two out_layer heads, :32-43,255) and
   * 2048 channels (the decoder's input, models/decoder.py:8-9). */
  int fusion_hid_ch1, fusion_hid_ch2;
} CdrWeightPtrs;

typedef struct CdrWeights CdrWeights; /* opaque: BN-folded, re-laid-out device buffers */

/* Optional stage taps of cdr_head_forward (any member may be NULL). Used by the parity
 * tests; layouts as documented per member. */
typedef struct CdrHeadTaps {
  float* pinv;      /* (2,B,4,3)            P_v^+ as used (models/cdrnet.py:236-237)   */
  float* cf_cat;    /* (B,64,800)  NHWC     concat of the two inverse-FTL outputs (:70) */
  float* cf_f;      /* (B,64,400)  NHWC     conv_layer2 output (:74)                    */
  float* f_out;     /* (2,B,64,2048) NHWC   out_layer outputs (:81), view-major         */
  float* heatmaps;  /* (2,B,J,64,64) NCHW   decoder outputs (:244), view-major          */
} CdrHeadTaps;

int cdr_abi_version(void);
/* Diagnostics: arms (first call) and returns 16 host-mapped words.  Word 0 becomes 0xdeadbeef if an
 * mbarrier wait inside a kernel timed out (a protocol bug): 1..6 = block, thread, shared-memory address
 * of the barrier, parity, gridDim.x, blockDim.x. */
const unsigned int* cdr_debug_words(void);
const char* cdr_last_error(void);
/* Number of kernels this library has launched from the calling thread since the last
 * reset (bench.py's `gpu_launches`). */
unsigned long long cdr_launch_count(void);
void cdr_launch_count_reset(void);

/* Per-launch device timing for bench.py's live roofline numbers.  _begin records a CUDA event
 * on `stream` and arms the calling thread; every kernel this library then launches from that
 * thread is followed by another event on the same stream.  _end synchronises the last event,
 * disarms, and returns for launch i its stage label (48-byte slots in `names`) and the time
 * between the events around it.  All launches in between must be on `stream`. */
int cdr_stage_timing_begin(void* stream);
int cdr_stage_timing_end(int capacity, char* names, float* ms, int* count);

/* Fold BN into the convs, convert/re-lay-out for `precision`, on `stream`.
 * Replaces nn.Module parameter storage + eval-mode BN of models/cdrnet.py:17-43 and
 * models/decoder.py:8-37.  The source tensors may be freed once this returns. */
int cdr_weights_create(const CdrWeightPtrs* src, int precision, void* stream, CdrWeights** out);
int cdr_weights_destroy(CdrWeights* w);

/* Workspace (bytes) cdr_head_forward / cdr_decoder_forward need for a batch of `batch`
 * stereo pairs (head) or `batch` images (decoder) at the handle's precision. */
int cdr_head_workspace_bytes(const CdrWeights* w, int batch, size_t* bytes);
int cdr_decoder_workspace_bytes(const CdrWeights* w, int n_images, size_t* bytes);

/* CDRNet.forward after the encoder — models/cdrnet.py:236-268.
 *   feat_l/feat_r (B,2048,8,8) fp32 NCHW; P_l/P_r (B,3,4); pinv_l/pinv_r (B,4,3) or both
 *   NULL (then computed on device with `pinv_rtol`, torch.linalg.pinv semantics);
 *   kp2d_l/kp2d_r (B,J,2), xyz (B,J,3) outputs. img_size = xs[0].size(2) (256). */
int cdr_head_forward(const CdrWeights* w, const float* feat_l, const float* feat_r,
                     const float* P_l, const float* P_r, const float* pinv_l,
                     const float* pinv_r, double pinv_rtol, int batch, int img_size,
                     float* kp2d_l, float* kp2d_r, float* xyz, const CdrHeadTaps* taps,
                     void* workspace, size_t workspace_bytes, void* stream);

/* cdr_head_forward on latents that are already pixel-major bf16 rows: feat_rows (2*B*64, 2048),
 * the left view's B*64 rows first — the layout cdr_encoder_forward writes.  Tensor-core
 * precisions only. */
int cdr_head_forward_rows(const CdrWeights* w, const void* feat_rows, const float* P_l, const float* P_r,
                          const float* pinv_l, const float* pinv_r, double pinv_rtol, int batch,
                          int img_size, float* kp2d_l, float* kp2d_r, float* xyz, const CdrHeadTaps* taps,
                          void* workspace, size_t workspace_bytes, void* stream);

/* cdr_head_forward / cdr_decoder_forward on the fp16 planes buffer of a CDR_PREC_F16X2 encoder (see
 * cdr_encoder_create_prec); CDR_PREC_F16X2 weights only. */
int cdr_head_forward_planes(const CdrWeights* w, const void* feat_planes, const float* P_l, const float* P_r,
                            const float* pinv_l, const float* pinv_r, double pinv_rtol, int batch,
                            int img_size, float* kp2d_l, float* kp2d_r, float* xyz, const CdrHeadTaps* taps,
                            void* workspace, size_t workspace_bytes, void* stream);
int cdr_decoder_forward_planes(const CdrWeights* w, const void* feat_planes, int n_images, float* heatmaps,
                               void* workspace, size_t workspace_bytes, void* stream);

/* cdr_decoder_forward on bf16 pixel-major latents (n_images*64, 2048) — PoseResNet.forward with the encoder
 * of this library (models/poseresnet.py:17-21).  Tensor-core precisions only. */
int cdr_decoder_forward_rows(const CdrWeights* w, const void* feat_rows, int n_images, float* heatmaps,
                             void* workspace, size_t workspace_bytes, void* stream);

/* ---- SURVEY §8f rank 1: the ResNet bottleneck stages of the encoder (models/encoder.py:38-131,
 * layer1..layer4) on the same tcgen05 tap-GEMM kernel, bf16 activations, eval-mode BN folded.
 * The 7x7 stem + max-pool (models/encoder.py:93-97,122-125) stay with the caller (torch/cuDNN);
 * their output, NHWC bf16, is this function's input. */
typedef struct CdrEncoderBlock {  /* one Bottleneck, models/encoder.py:38-76 */
  CdrConvBn conv1, conv2, conv3;  /* conv weight (Cout,Cin,kh,kw) fp32, bias NULL, + BN tensors        */
  CdrConvBn downsample;           /* weight NULL when the block has no downsample branch              */
  int planes;                     /* conv1: Cin->planes 1x1; conv2: 3x3 stride; conv3: ->4*planes 1x1 */
  int stride;
} CdrEncoderBlock;
typedef struct CdrEncoderSpec {
  int num_blocks;                 /* over layer1..layer4, in order (ResNet-101: 3+4+23+3)             */
  const CdrEncoderBlock* blocks;  /* HOST array of device-pointer structs                             */
  int in_channels;                /* 64                                                                */
  CdrConvBn stem;                 /* conv1 (64,3,7,7) + bn1 — models/encoder.py:93-95; weight NULL: the
                                     caller runs the stem itself and uses cdr_encoder_forward only      */
} CdrEncoderSpec;
typedef struct CdrEncoder CdrEncoder;
int cdr_encoder_create(const CdrEncoderSpec* spec, void* stream, CdrEncoder** out);   /* CDR_PREC_BF16 */
/* The same encoder at the reference's precision (models/encoder.py runs in fp32): precision = CDR_PREC_F16X2 keeps
 * every activation as scaled fp16 hi/lo planes (2^-24 relative) and runs every conv as 3 kind::f16 MMAs per product
 * (gemm_tc.cu: kKindF16X2), the residual add in the epilogue; the 7x7 stem runs as three fp16 mma.sync per product.  Such a handle
 *   - starts from images only (cdr_encoder_forward_images / _frames_u8; cdr_encoder_forward returns CDR_ERR_INVALID),
 *   - writes its latents as an "fp16 planes" buffer instead of bf16 rows:
 *       [hi plane: rows*C fp16 | lo plane: rows*C fp16 | float amax, float scale]
 *     each plane padded to a multiple of 1024 bytes, x = (hi + lo * 2^-11) / scale; size from cdr_encoder_out_bytes,
 *     1024-byte aligned.  cdr_head_forward_planes / cdr_decoder_forward_planes consume it as conv_layer1's /
 *     deconv1's operand without a conversion pass. */
int cdr_encoder_create_prec(const CdrEncoderSpec* spec, int precision, void* stream, CdrEncoder** out);
/* bytes of the latent buffer the forward functions write for (n_images, in_h, in_w) = the stem's OUTPUT grid
 * (img/4): bf16 rows, or the fp16 planes buffer above */
int cdr_encoder_out_bytes(const CdrEncoder* e, int n_images, int in_h, int in_w, size_t* bytes);
int cdr_encoder_destroy(CdrEncoder* e);
int cdr_encoder_workspace_bytes(const CdrEncoder* e, int n_images, int in_h, int in_w, size_t* bytes);
int cdr_encoder_out_shape(const CdrEncoder* e, int in_h, int in_w, int* out_h, int* out_w, int* out_c);
/* x (n_images, in_h, in_w, 64) bf16 NHWC -> out_rows (n_images*out_h*out_w, out_c) bf16 pixel-major rows. */
int cdr_encoder_forward(const CdrEncoder* e, const void* x_nhwc_bf16, int n_images, int in_h, int in_w,
                        void* out_rows_bf16, void* workspace, size_t workspace_bytes, void* stream);

/* The whole encoder, models/encoder.py:121-131: images (n,3,H,W) fp32 NCHW (H % 16 == 0, W % 64 == 0) ->
 * stem (conv 7x7 s2 + BN + ReLU on warp-level tensor-core MMAs, max-pool 3x3 s2) -> layer1..4.
 * Needs a spec with `stem` set; workspace from cdr_encoder_workspace_bytes_images. */
int cdr_encoder_workspace_bytes_images(const CdrEncoder* e, int n_images, int img_h, int img_w, size_t* bytes);
int cdr_encoder_forward_images(const CdrEncoder* e, const float* images, int n_images, int img_h, int img_w,
                               void* out_rows_bf16, void* workspace, size_t workspace_bytes, void* stream);

/* SURVEY §8f rank 2 — device-side input pipeline: the same from raw uint8 frames (n, H, W, 3) HWC with
 * torchvision's ToTensor + Normalize(mean, std) of inference.py:40-44 fused into the stem's patch load
 * (x / 255, - mean, / std in fp32, the reference's operation order).  mean/std: HOST float[3]. */
int cdr_encoder_forward_frames_u8(const CdrEncoder* e, const uint8_t* frames, const float* mean_host,
                                  const float* std_host, int n_images, int img_h, int img_w, void* out_rows_bf16,
                                  void* workspace, size_t workspace_bytes, void* stream);

/* PoseDecoder.forward — models/decoder.py:39-46 (also the decoder half of
 * PoseResNet.forward, models/poseresnet.py:17-21).  feat (N,2048,8,8) -> heatmaps
 * (N,J,64,64) fp32 NCHW. */
int cdr_decoder_forward(const CdrWeights* w, const float* feat, int n_images, float* heatmaps,
                        void* workspace, size_t workspace_bytes, void* stream);

/* torch.linalg.pinv on (n,3,4) -> (n,4,3) — models/cdrnet.py:236-237.  One-sided Jacobi
 * SVD in fp64; singular values <= rtol * sigma_max are dropped (torch default rtol for
 * fp32 input is 4*eps = 4.76837158203125e-07). */
int cdr_pinv(const float* P, int n, double rtol, float* pinv, void* stream);

/* CanonicalFusion.ftl — models/cdrnet.py:45-56, on pixel-major activations.
 *   in  (n, hw, in_pitch) with rows*... channel blocks of `blk` (=100) channels;
 *   mats (n, rows, cols) row-major; out[(i,p), r*blk + c] = sum_k mats[i,r,k] * in[(i,p), k*blk + c]
 *   written at out + out_offset with pitch out_pitch; columns rows*blk..out_fill-1 are zeroed. */
int cdr_ftl(const float* in, int in_pitch, const float* mats, int rows, int cols, int blk,
            int n, int hw, float* out, int out_pitch, int out_fill, void* stream);

/* process_heatmap (+ the x img/heatmap scale) — models/cdrnet.py:120-149,250.
 * heat (n_maps,H,W) fp32 -> kp (n_maps,2) = (x,y)*scale. */
int cdr_softargmax(const float* heat, long long n_maps, int H, int W, float scale, float* kp,
                   void* stream);

/* CDRNet.dlt looped over joints — models/cdrnet.py:151-179,262-266.
 * P_l/P_r (B,3,4), kp_l/kp_r (B,J,2) -> xyz (B,J,3).  fp64 Jacobi SVD per joint. */
int cdr_dlt(const float* P_l, const float* P_r, const float* kp_l, const float* kp_r, int batch,
            int joints, float* xyz, void* stream);

/* Fused soft-argmax + DLT (+ optional per-pose MPJPE partial sums) — the streaming kernel
 * for models/cdrnet.py:243-266 (+ models/metrics.py:82-95).
 *   heat_l/heat_r (B,J,H,W) fp32 (or bf16 if heat_is_bf16); outputs as cdr_head_forward.
 *   If gt3d != NULL: gt3d (B,J,3), gt2d_l/gt2d_r (B,J,2) fp64, vis (B,J) fp64 or NULL;
 *   pose_err (B,3) fp64 receives per-pose sums of ||d2d_l||, ||d2d_r||, ||d3d||. */
int cdr_softargmax_dlt(const void* heat_l, const void* heat_r, int heat_is_bf16, const float* P_l,
                       const float* P_r, long long batch, int joints, int H, int W, float scale,
                       float* kp2d_l, float* kp2d_r, float* xyz, const double* gt3d,
                       const double* gt2d_l, const double* gt2d_r, const double* vis,
                       double* pose_err, void* stream);

/* get_max_preds + `*4.0` + astype(uint8) — tools/utils.py:30-58, baseline.py:51-53.
 * heat (n_maps,H,W) fp32 -> preds (n_maps,2) fp32 (x,y; zero where max<=0), maxvals
 * (n_maps) fp32 (either may be NULL), and pts_u8 (n_maps,2) = uint8(preds*scale) or NULL. */
int cdr_argmax(const float* heat, long long n_maps, int H, int W, float scale, float* preds,
               float* maxvals, uint8_t* pts_u8, void* stream);

/* Projection matrices on the device — tools/common.py:28-32 (get_projection_matrix: P = K @ [R | t]), the crop /
 * resize affine of dataset/mads_3d.py:223-226 and tools/load.py:60-67 (T = eye(4), T[:2,:3] = trans; P = T @ P) and
 * inference.py:53-56 (first three rows, float32).  K (3,3) fp64 shared (k_batched = 0) or per camera (n,3,3);
 * R (n,3,3), t (n,3) fp64; trans (n,2,3) fp64 or NULL (T = identity) -> P (n,3,4) fp32, products and sums in fp64 in
 * numpy's order. */
int cdr_projection_matrices(const double* K, int k_batched, const double* R, const double* t, const double* trans,
                            int n, float* P, void* stream);

/* triangulation — tools/common.py:51-71.  P1/P2: fp64, `p_rows` x 4 row-major per sample
 * (3 or 4 rows; only the first three are read); p_batched = 0 shares one P pair across
 * all n_poses.  pts1/pts2 (n_poses,J,2) uint8 -> xyz (n_poses,J,3) fp64. */
int cdr_triangulate_u8(const double* P1, const double* P2, int p_rows, int p_batched,
                       const uint8_t* pts1, const uint8_t* pts2, long long n_poses, int joints,
                       double* xyz, void* stream);

/* calc_mpjpe partial sums — models/metrics.py:82-95.
 *   pred2d_l/r (n,J,2), pred3d (n,J,3) fp32 (pred_is_f64=0) or fp64 (=1); gt fp64;
 *   weight fp64 (n,J) if weight_batched else (J), or NULL; weight_f32_product = 1 rounds
 *   pred*weight to fp32 first (numpy's float32*float32 promotion in train_cdr.py:196-199).
 *   sums[0..2] = sum over (n,J) of ||.||_2 for 2D-left, 2D-right, 3D; sums[3] = n*J.
 *   Deterministic (fixed-order tree).  scratch: >= cdr_mpjpe_scratch_bytes(n) bytes. */
size_t cdr_mpjpe_scratch_bytes(long long n);
int cdr_mpjpe_partial(const void* pred2d_l, const void* pred2d_r, const void* pred3d,
                      int pred_is_f64, const double* gt3d, const double* gt2d_l,
                      const double* gt2d_r, const double* weight, int weight_batched,
                      int weight_f32_product, long long n, int joints, double* sums,
                      void* scratch, void* stream);
/* Reduce the (B,3) pose_err of cdr_softargmax_dlt into sums[4] (same meaning as above). */
int cdr_mpjpe_reduce(const double* pose_err, long long n, int joints, double* sums, void* scratch,
                     void* stream);

/* ---- SURVEY §8f rank 3 (first slice): backward passes of the non-conv operators — what train_cdr.py:105-127
 * back-propagates through (`loss.backward()` via process_heatmap and dlt).  fp32 in/out, fp64 internals.
 * The FTL is linear: its backward is cdr_ftl with the transposed matrices (no extra entry point). */

/* d/d heat of process_heatmap (+ scale), models/cdrnet.py:120-149,250.  heat (n_maps,H,W), grad_kp (n_maps,2)
 * -> grad_heat (n_maps,H,W) = scale * p * (gx (x - cx) + gy (y - cy)), p = softmax(heat).  W % 4 == 0, H*W <= 4096. */
int cdr_softargmax_backward(const float* heat, const float* grad_kp, long long n_maps, int H, int W,
                            float scale, float* grad_heat, void* stream);

/* d/d (kp_l, kp_r) of CDRNet.dlt, models/cdrnet.py:151-179 (the gradient torch.svd's backward gives for
 * X = V[:3,3] / V[3,3]; P carries no gradient in the reference).  grad_xyz (B,J,3) -> grad_kp_l/r (B,J,2). */
int cdr_dlt_backward(const float* P_l, const float* P_r, const float* kp_l, const float* kp_r,
                     const float* grad_xyz, int batch, int joints, float* grad_kp_l, float* grad_kp_r,
                     void* stream);

/* ---- SURVEY §8f rank 3, second slice: what a training step of the head needs besides the differentiable operators
 * above (train_cdr.py:82-143) — BatchNorm2d in TRAINING mode and the three losses of models/loss.py — forward and
 * backward on the reference's layouts.  (The convolutions of a training step stay library GEMMs: cuDNN through torch.)
 *
 * nn.BatchNorm2d(train) on x (n, c, h*w) fp32 NCHW — models/cdrnet.py:19,25,28,36,41, models/decoder.py:34 — with the
 * ReLU that follows it fused when relu != 0: batch mean / biased variance over (n, h, w), running_mean / running_var
 * updated in place (momentum; unbiased variance), save_mean / save_invstd (c) kept for the backward. */
int cdr_bn_train_forward(const float* x, int n, int c, int hw, const float* gamma, const float* beta, double eps,
                         double momentum, float* running_mean, float* running_var, int relu, float* y,
                         float* save_mean, float* save_invstd, void* stream);
int cdr_bn_train_backward(const float* x, const float* dy, int n, int c, int hw, const float* gamma, const float* beta,
                          const float* save_mean, const float* save_invstd, int relu, float* dx, float* dgamma,
                          float* dbeta, void* stream);
/* The reference's losses on (rows = B*J, d) tensors, weight = target_weight as (rows) or NULL:
 *   kind 0 JointsMSELoss (models/loss.py:5-32), 1 JointsMSESmoothLoss (:35-66, `threshold`), 2 MPJPELoss (:69-98).
 * loss: 1 float; scratch: cdr_joint_loss_scratch_bytes() bytes, 8-byte aligned; fixed-order fp64 sums (deterministic). */
size_t cdr_joint_loss_scratch_bytes(void);
int cdr_joint_loss_forward(int kind, const float* pred, const float* target, const float* weight, long long rows, int d,
                           double threshold, float* loss, void* scratch, void* stream);
int cdr_joint_loss_backward(int kind, const float* pred, const float* target, const float* weight, long long rows, int d,
                            double threshold, const float* grad_loss, float* grad_pred, void* stream);

/* ---- Training the decoder's transposed convolutions: ConvTranspose2d(Cin, Cout, 4, stride 2, padding 1, bias=False) at
 * fp32 accuracy on the tensor cores (scaled fp16 hi/lo operands, 3 kind::f16 MMAs per product), forward and backward.
 * x (n, Cin, h, w), weight (Cin, Cout, 4, 4), y / dy (n, Cout, 2h, 2w), all fp32 NCHW, 16-byte aligned.
 * Supported: Cin and Cout multiples of 64, h == w in {8, 16, 32}, n >= 1 (CDR_ERR_UNSUPPORTED otherwise).
 * The forward leaves x, re-encoded for the weight gradient, in `saved` (saved_bytes, 256-byte aligned; as large as
 * an fp16 copy of x plus 1 KB); the backward reads it back.  One workspace (workspace_bytes, 256-byte aligned) serves
 * both calls.  The backward writes dx (n, Cin, h, w) and / or dweight (Cin, Cout, 4, 4); a NULL pointer skips that
 * GEMM.  dweight is bitwise deterministic (fixed-order reduction of its K slices, no atomics). */
int cdr_deconv_train_workspace_bytes(int n, int cin, int cout, int h, int w, size_t* saved_bytes,
                                     size_t* workspace_bytes);
int cdr_deconv_train_forward(const float* x, const float* weight, int n, int cin, int cout, int h, int w, float* y,
                             void* saved, size_t saved_bytes, void* workspace, size_t workspace_bytes, void* stream);
int cdr_deconv_train_backward(const void* saved, const float* weight, const float* dy, int n, int cin, int cout, int h,
                              int w, float* dx, float* dweight, void* workspace, size_t workspace_bytes, void* stream);

/* ---- Training 1x1 convolutions: Conv2d(Cin, Cout, 1), bias optional, at fp32 accuracy on the tensor cores (the same
 * scaled fp16 hi/lo operands), forward and backward.  x (n, Cin, h, w), weight (Cout, Cin, 1, 1), bias (Cout) or NULL,
 * y / dy (n, Cout, h, w), all fp32 NCHW; x, weight, y, dy, dx, dweight 16-byte aligned, bias / dbias 4-byte.
 * Supported: n >= 1, 1 <= Cin, Cout <= 4096, h*w a multiple of 64, n*h*w <= 2^22 (CDR_ERR_INVALID otherwise).
 * `saved` and the workspace work as for cdr_deconv_train_*.  The backward writes dx (n, Cin, h, w), dweight
 * (Cout, Cin, 1, 1) and / or dbias (Cout); a NULL pointer skips that output.  dweight and dbias are bitwise
 * deterministic (fixed-order reductions, no atomics). */
int cdr_conv1x1_train_workspace_bytes(int n, int cin, int cout, int h, int w, size_t* saved_bytes,
                                      size_t* workspace_bytes);
int cdr_conv1x1_train_forward(const float* x, const float* weight, const float* bias, int n, int cin, int cout, int h,
                              int w, float* y, void* saved, size_t saved_bytes, void* workspace, size_t workspace_bytes,
                              void* stream);
int cdr_conv1x1_train_backward(const void* saved, const float* weight, const float* dy, int n, int cin, int cout, int h,
                               int w, float* dx, float* dweight, float* dbias, void* workspace, size_t workspace_bytes,
                               void* stream);

/* ---- Training 3x3 convolutions: Conv2d(Cin, Cout, 3, stride, padding 1, bias=False) with stride 1 or 2, at fp32
 * accuracy on the tensor cores (the same scaled fp16 hi/lo operands), forward and backward.  x (n, Cin, h, w) with h x w
 * the INPUT map, weight (Cout, Cin, 3, 3), y / dy (n, Cout, h/stride, w/stride), all fp32 NCHW, 16-byte aligned.
 * Supported: n >= 1, Cin and Cout multiples of 64 in [64, 2048], h and w divisible by the stride, and for the output
 * map H x W: W a power of two in [8, 64], H*W = 64 or a multiple of 128, n*H*W <= 2^22 (CDR_ERR_INVALID otherwise).
 * `saved` and the workspace work as for cdr_deconv_train_*.  The backward writes dx (n, Cin, h, w) and / or dweight
 * (Cout, Cin, 3, 3); a NULL pointer skips that output.  dweight is bitwise deterministic (fixed-order reduction). */
int cdr_conv3x3_train_workspace_bytes(int n, int cin, int cout, int h, int w, int stride, size_t* saved_bytes,
                                      size_t* workspace_bytes);
int cdr_conv3x3_train_forward(const float* x, const float* weight, int n, int cin, int cout, int h, int w, int stride,
                              float* y, void* saved, size_t saved_bytes, void* workspace, size_t workspace_bytes,
                              void* stream);
int cdr_conv3x3_train_backward(const void* saved, const float* weight, const float* dy, int n, int cin, int cout, int h,
                               int w, int stride, float* dx, float* dweight, void* workspace, size_t workspace_bytes,
                               void* stream);

/* ---- Training the encoder's stem convolution: Conv2d(3, 64, 7, stride 2, padding 3, bias=False) at fp32 accuracy on
 * warp-level tensor-core MMAs (scaled fp16 hi/lo operands, 3 MMAs per product), forward and weight gradient.
 * x (n, 3, h, w), weight (64, 3, 7, 7), y / dy (n, 64, h/2, w/2), all fp32 NCHW, 16-byte aligned.
 * Supported: cin = 3, cout = 64, h % 16 == 0, w % 64 == 0, n*(h/2)*(w/2) <= 2^22 (CDR_ERR_INVALID otherwise).
 * There is NO input gradient: the stem's input is the image batch.  The backward returns CDR_ERR_INVALID unless dx is
 * NULL; a NULL dweight makes it a no-op.  `saved` and the workspace work as for cdr_deconv_train_*.  dweight is bitwise
 * deterministic (fixed-order reduction of its K slices, no atomics). */
int cdr_stem_train_workspace_bytes(int n, int cin, int cout, int h, int w, size_t* saved_bytes, size_t* workspace_bytes);
int cdr_stem_train_forward(const float* x, const float* weight, int n, int cin, int cout, int h, int w, float* y,
                           void* saved, size_t saved_bytes, void* workspace, size_t workspace_bytes, void* stream);
int cdr_stem_train_backward(const void* saved, const float* weight, const float* dy, int n, int cin, int cout, int h,
                            int w, float* dx, float* dweight, void* workspace, size_t workspace_bytes, void* stream);

/* ---- The stem's max-pool in training: MaxPool2d(3, stride 2, padding 1) on x (n, c, h, w) fp32 NCHW -> y (n, c, ho, wo),
 * ho = (h - 1) / 2 + 1, wo = (w - 1) / 2 + 1, equal to torch's CUDA kernel bit for bit, forward and backward.  The window
 * is scanned in row-major order from its first in-image element; an element replaces the maximum when it is larger or
 * NaN.  The forward writes y and `argmax`, n*c*ho*wo bytes: per output its window position ky*3 + kx.  The backward
 * writes dx (n, c, h, w): per input element the sum, from +0.0 in (oy, ox) order, of the dy of the windows whose argmax
 * it is.  Supported: every size >= 1, n*c*h*w < 2^31; fp32 tensors 4-byte aligned (CDR_ERR_INVALID otherwise). */
int cdr_maxpool3x3_train_forward(const float* x, int n, int c, int h, int w, float* y, uint8_t* argmax, void* stream);
int cdr_maxpool3x3_train_backward(const uint8_t* argmax, const float* dy, int n, int c, int h, int w, float* dx,
                                  void* stream);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif
#ifdef __cplusplus
}
#endif
#endif /* CDRHEAD_H_ */
