/* mrn_b200 -- C ABI of the B200-native MRN multiplexed-routing train / infer step.
 *
 * The reference (simplify23/MRN) is pure Python/PyTorch and has no FFI of its own; its boundary for this path
 * is the nn.Module / learner API of modules/model.py, modules/dm_router.py and il_modules/mrn.py.  Every entry
 * point below names the reference code (file:line, relative to the reference root) it replaces.  The Python
 * mirror of that API (mrn_b200/modules/*.py, mrn_b200/il_modules/mrn.py) binds these symbols through ctypes
 * (mrn_b200/_lib.py); INTEGRATION.md shows the stub a reference maintainer would add.
 *
 * Conventions
 *   - plain pointers and sizes only; every pointer is a DEVICE pointer unless it is documented as a host array
 *     (pointer tables `const T* const*`, `ld`, `Ci` arrays and the MrnbSvtrPack struct live on the host);
 *   - the caller owns all memory (inputs, outputs, workspace); nothing is allocated or freed, nothing
 *     synchronises; every kernel is enqueued on `stream` (a cudaStream_t passed as void*-compatible handle);
 *   - return value: 0 = MRNB_OK, negative = error; mrnb_last_error() returns a thread-local message;
 *   - there is no CPU fallback and no alternative backend: the library is sm_100a code only.
 */
#ifndef MRN_B200_H
#define MRN_B200_H

#include <stddef.h>

#ifdef __cplusplus
extern "C" {
#endif

#ifndef __CUDA_RUNTIME_H__
typedef struct CUstream_st* cudaStream_t;
#endif

#define MRNB_OK 0
#define MRNB_ERR_ARG (-1)
#define MRNB_ERR_WORKSPACE (-2)
#define MRNB_ERR_LAUNCH (-3)
#define MRNB_ERR_UNSUPPORTED (-4)

#define MRNB_MAX_EXPERTS 8
#define MRNB_PREC_FP32 0 /* CUDA-core fp32 contractions (parity mode, 1e-4 tolerance) */
#define MRNB_PREC_BF16 1 /* tcgen05 bf16 operands, fp32 accumulate in TMEM (2e-2 tolerance) */

int mrnb_version(void);
const char* mrnb_last_error(void);
/* kernels launched by this library since the last reset (bench.py "gpu_launches") */
long mrnb_launch_count(void);
void mrnb_reset_launch_count(void);

/* Optional per-kernel-family timing with CUDA events on the launching stream (bench.py roofline evidence).
 * Families: 0 tc_gemm_kernel (persistent tcgen05 GEMM), 1 sgemm_kernel (fp32), 2 attention, 3 LayerNorm, 4 patch embed,
 * 5 gated combine, 6 CTC lattice, 7 router elementwise, 8 optimiser, 9 misc, 10 mlp_tc_kernel, 11 tc_gemm2_kernel.  mrnb_profile_read synchronises on the recorded events. */
void mrnb_profile_enable(int on);
void mrnb_profile_reset(void);
int mrnb_profile_read(int family, double* ms, long* calls, double* flops, double* bytes);

/* ---------------------------------------------------------------------------------------------------------
 * SVTR expert recognisers, grouped over experts.
 * Replaces  modules/model.py:82-101 (Model_Extractor.forward), :133-148 (Model.forward),
 *           modules/svtr.py:500-528 (SVTR.forward_features) and everything below it,
 *           torch.stack(features, 1) at modules/model.py:400 / :369.
 *
 * Parameter slots (MrnbSvtrPack.p[slot]): fp32 device tensors STACKED over experts, [I, ...reference shape...],
 * except the two layouts marked (*) which are re-laid once at load time (kh,kw before Cin):
 */
enum {
  MRNB_P_POS_EMBED = 0, /* [I,512,64]        ConvNet.pos_embed */
  MRNB_P_CONV0_W,       /* [I,32,4,3,3]      patch_embed.proj.0.weight */
  MRNB_P_CONV0_B,       /* [I,32] */
  MRNB_P_BN0_W, MRNB_P_BN0_B, MRNB_P_BN0_MEAN, MRNB_P_BN0_VAR, /* [I,32] patch_embed.proj.1.* (mean/var are updated in train mode) */
  MRNB_P_CONV1_W,       /* [I,64,3,3,32] (*) patch_embed.proj.3.weight permuted (0,2,3,1) */
  MRNB_P_CONV1_B,       /* [I,64] */
  MRNB_P_BN1_W, MRNB_P_BN1_B, MRNB_P_BN1_MEAN, MRNB_P_BN1_VAR, /* [I,64] patch_embed.proj.4.* */
  MRNB_P_BLOCK0 = 13,   /* 12 blocks x MRNB_PB_COUNT slots: blocks1.0-2, blocks2.0-5, blocks3.0-2 */
  MRNB_P_SUB0 = 13 + 12 * 12, /* 3 merges x MRNB_PS_COUNT slots: sub_sample1..3 */
  MRNB_P_SEQ_W = 13 + 12 * 12 + 3 * 4, /* [I,256,512] model.SequenceModeling.0.weight */
  MRNB_P_SEQ_B,         /* [I,256] */
  MRNB_P_COUNT
};
enum { /* per block, d = 64/128/256 */
  MRNB_PB_NORM1_W = 0, MRNB_PB_NORM1_B, /* [I,d] */
  MRNB_PB_QKV_W, MRNB_PB_QKV_B,         /* [I,3d,d], [I,3d] */
  MRNB_PB_PROJ_W, MRNB_PB_PROJ_B,       /* [I,d,d], [I,d] */
  MRNB_PB_NORM2_W, MRNB_PB_NORM2_B,
  MRNB_PB_FC1_W, MRNB_PB_FC1_B,         /* [I,4d,d], [I,4d] */
  MRNB_PB_FC2_W, MRNB_PB_FC2_B,         /* [I,d,4d], [I,d] */
  MRNB_PB_COUNT
};
enum { /* per merge, Cin -> Cout = 64->128, 128->256, 256->512 */
  MRNB_PS_CONV_W = 0, /* [I,Cout,3,3,Cin] (*) sub_sampleK.conv.weight permuted (0,2,3,1) */
  MRNB_PS_CONV_B,     /* [I,Cout] */
  MRNB_PS_NORM_W, MRNB_PS_NORM_B, /* [I,Cout] */
  MRNB_PS_COUNT
};

typedef struct MrnbSvtrPack {
  int n_experts;
  const float* p[MRNB_P_COUNT]; /* fp32 parameters (always required) */
  const void* h[MRNB_P_COUNT];  /* 16-bit copies of the GEMM weight slots, MRNB_PREC_BF16 only: bf16 for qkv/proj/fc1/conv/seq
                                   (conv1 in its implicit-GEMM layout [I,64,384]), f16 for mlp.fc2 (fused MLP second GEMM) */
  const float* fc_w[MRNB_MAX_EXPERTS];  /* [C_i,256] model.{i}.fc.weight (ragged over experts) */
  const void* fc_w16[MRNB_MAX_EXPERTS]; /* bf16 copy; MRNB_PREC_BF16 only */
  const float* fc_b[MRNB_MAX_EXPERTS];  /* [C_i] */
  int n_class[MRNB_MAX_EXPERTS];
} MrnbSvtrPack;

#define MRNB_ALL_EXPERTS (-1)
size_t mrnb_svtr_workspace_bytes(int n_experts, int B, int chunk, int prec);

/* image [B,4,32,256] fp32 NCHW.  chunk: samples processed together after the patch embedding (0 = all).
 * bn_batch_stats / update_running are per-expert BIT MASKS (bit e = expert e; MRNB_ALL_EXPERTS = every expert, 0 = none):
 * bit set in bn_batch_stats: that expert's nn.BatchNorm2d runs as in .train() (batch statistics; the same bit in
 * update_running also applies the momentum update, reference quirk il_modules/mrn.py:401); clear: running statistics.
 * (The reference can hold experts in different modes: after update_step1 the newest expert is .eval() while the frozen
 * older ones are still in .train(), il_modules/mrn.py:284-287 vs :107.)
 * drop_scales: NULL or [I,12,2,B] DropPath multipliers (modules/svtr.py:7-22).
 * features: NULL or [B,I,64,256] fp32 (router input).  logits: host array of I device pointers (NULL entries are
 * skipped), logits[i] is [B,64,ld_logits[i]] fp32 with the first C_i columns written (model.{i} "predict"). */
int mrnb_svtr_experts_forward(const MrnbSvtrPack* pack, const float* image, int B, int chunk, int prec,
                              int bn_batch_stats, int update_running, const float* drop_scales, float* features,
                              float* const* logits, const long* ld_logits, void* workspace, size_t workspace_bytes,
                              cudaStream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * Stage-0 expert training: one SVTR expert, activation-keeping forward + full backward.
 * Replaces il_modules/mrn.py:225-279 (_init_train: model(image, cross=False)['logits'] -> loss.backward()), i.e. the
 * autograd graph of modules/model.py:351-353 -> :133-148 -> modules/svtr.py:500-528 in train mode.
 *
 * `pack` holds exactly ONE expert (n_experts == 1) in the slot layout above; `grads` has the same slots pointing into a
 * flat fp32 gradient arena [n_arena] (BN running-stat slots unused) that the backward zeroes and fills -- the same arena
 * layout serves mrnb_clip_adam and the NCCL all-reduce.  The workspace carries the saved activations from the forward
 * to the backward call (same pointer, same B).  drop_scales: NULL or [12,2,B] DropPath multipliers.
 * MRNB_PREC_BF16: pack->h[] / fc_w16[0] must hold bf16 copies of the GEMM weights (qkv, proj, fc1, fc2, merge convs,
 * seq, fc) refreshed after every optimiser step; the patch embedding and all statistics stay fp32.
 * logits / dlogits: [B,64,ld] fp32, first n_class[0] columns valid (dlogits from mrnb_ctc_dense_grad). */
size_t mrnb_svtr_train_workspace_bytes(int B, int n_class, int prec);
int mrnb_svtr_train_forward(const MrnbSvtrPack* pack, const float* image, int B, int prec, int bn_batch_stats,
                            int update_running, const float* drop_scales, float* logits, long ld_logits, void* workspace,
                            size_t workspace_bytes, cudaStream_t stream);
int mrnb_svtr_train_backward(const MrnbSvtrPack* pack, const MrnbSvtrPack* grads, const float* image, const float* dlogits,
                             long ld_dlogits, int B, int prec, int bn_batch_stats, const float* drop_scales,
                             float* grad_arena, long n_arena, void* workspace, size_t workspace_bytes, cudaStream_t stream);

/* The same two calls with the expert's feature exposed, for joint expert + router training through MRNNet's soft route
 * (modules/model.py:397-423 with nothing detached between the experts and the DM-Router; the two entries above are these
 * with NULL).  features: NULL or [B,64,256] fp32 (dense), the SequenceModeling Linear's output f (modules/model.py:141);
 * in bf16 mode the bf16 value the classifier head reads, widened.  dfeatures: NULL or [B,64,256] fp32 (dense), a
 * gradient dL/df from outside the expert (the DM-Router's input gradient), added to dlogits . W_fc before anything
 * downstream reads it. */
int mrnb_svtr_train_forward_features(const MrnbSvtrPack* pack, const float* image, int B, int prec, int bn_batch_stats,
                                     int update_running, const float* drop_scales, float* logits, long ld_logits,
                                     float* features, void* workspace, size_t workspace_bytes, cudaStream_t stream);
int mrnb_svtr_train_backward_features(const MrnbSvtrPack* pack, const MrnbSvtrPack* grads, const float* image,
                                      const float* dlogits, long ld_dlogits, const float* dfeatures, int B, int prec,
                                      int bn_batch_stats, const float* drop_scales, float* grad_arena, long n_arena,
                                      void* workspace, size_t workspace_bytes, cudaStream_t stream);

/* The backward with the gradient with respect to the input image, for any differentiable module in front of the
 * recogniser (a rectification front end such as the reference's Transformation="TPS" stage, modules/transformation.py:9-216;
 * learned augmentation; inversion of a frozen expert; saliency maps).  Arguments as mrnb_svtr_train_backward_features
 * (which is this call with dimage = NULL), plus:
 *   dimage: NULL or [B,4,32,256] fp32 NCHW (dense), overwritten with dL/dimage -- the input gradient of the patch
 *           embedding's conv0 (modules/svtr.py PatchEmbed.proj[0], Conv2d(4, 32, 3, 2, 1)), read from the fp32 gradient
 *           at conv0's output in both precision modes.
 *   grads / grad_arena: both NULL selects the input-only backward of a frozen expert -- no parameter gradient is
 *           computed (every launch whose only product is one is skipped); the BatchNorm batch statistics the input
 *           gradient needs are kept.  At least one of grad_arena and dimage must be non-NULL (else MRNB_ERR_ARG). */
int mrnb_svtr_train_backward_input(const MrnbSvtrPack* pack, const MrnbSvtrPack* grads, const float* image,
                                   const float* dlogits, long ld_dlogits, const float* dfeatures, int B, int prec,
                                   int bn_batch_stats, const float* drop_scales, float* grad_arena, long n_arena,
                                   float* dimage, void* workspace, size_t workspace_bytes, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * CRNN expert recognisers (VGG + 2 x BidirectionalLSTM + CTC head), T = 63 frames.
 * Replaces modules/feature_extraction.py:19-47 (VGG_FeatureExtractor.forward), modules/sequence_modeling.py:12-22
 * (BidirectionalLSTM.forward, x2), modules/model.py:82-101 (Model_Extractor.forward) and :133-148 (Model.forward),
 * called once per expert by MRNNet.forward (modules/model.py:366-368,397-399).
 *
 * Parameter slots are stacked over experts (leading dimension I).  Convolution weights are re-laid once at load
 * time as [Cout, kh, kw, Cin] (kh, kw before Cin), except conv0 which keeps nn.Conv2d's layout.  LSTM slots:
 * W_ih of both directions concatenated along the gate axis, b_ih + b_hh pre-summed.
 */
enum {
  MRNB_C_CONV0_W = 0,   /* [I,64,4,3,3]     ConvNet.0.weight */
  MRNB_C_CONV0_B,       /* [I,64] */
  MRNB_C_CONV1_W,       /* [I,128,3,3,64]   (*) ConvNet.3.weight permuted (0,2,3,1) */
  MRNB_C_CONV1_B,       /* [I,128] */
  MRNB_C_CONV2_W,       /* [I,256,3,3,128]  (*) ConvNet.6 */
  MRNB_C_CONV2_B,
  MRNB_C_CONV3_W,       /* [I,256,3,3,256]  (*) ConvNet.8 */
  MRNB_C_CONV3_B,
  MRNB_C_CONV4_W,       /* [I,512,3,3,256]  (*) ConvNet.11 (bias=False) */
  MRNB_C_BN4_W, MRNB_C_BN4_B, MRNB_C_BN4_MEAN, MRNB_C_BN4_VAR, /* [I,512] ConvNet.12.* (mean/var updated in train mode) */
  MRNB_C_CONV5_W,       /* [I,512,3,3,512]  (*) ConvNet.14 (bias=False) */
  MRNB_C_BN5_W, MRNB_C_BN5_B, MRNB_C_BN5_MEAN, MRNB_C_BN5_VAR, /* [I,512] ConvNet.15.* */
  MRNB_C_CONV6_W,       /* [I,512,2,2,512]  (*) ConvNet.18 */
  MRNB_C_CONV6_B,       /* [I,512] */
  MRNB_C_LSTM0 = 20,    /* 2 layers x MRNB_CL_COUNT slots: SequenceModeling.0, SequenceModeling.1 */
  MRNB_C_COUNT = 20 + 2 * 5
};
enum { /* per BidirectionalLSTM, Kin = 512 (layer 0) / 256 (layer 1).  The gate axis is INTERLEAVED per hidden unit:
          packed row 4*j + k holds nn.LSTM row k*256 + j (k = i,f,g,o), so the four gates of a unit are adjacent columns
          of the recurrent GEMM and its epilogue can apply the cell */
  MRNB_CL_WIH = 0, /* [I,2048,Kin]   rows 0..1023 rnn.weight_ih_l0 (interleaved), 1024..2047 rnn.weight_ih_l0_reverse */
  MRNB_CL_WHH,     /* [I,2,1024,256] rnn.weight_hh_l0, rnn.weight_hh_l0_reverse (interleaved rows) */
  MRNB_CL_BIAS,    /* [I,2048]       bias_ih + bias_hh (interleaved), forward then reverse */
  MRNB_CL_LIN_W,   /* [I,256,512]    linear.weight */
  MRNB_CL_LIN_B,   /* [I,256] */
  MRNB_CL_COUNT
};

typedef struct MrnbCrnnPack {
  int n_experts;
  const float* p[MRNB_C_COUNT]; /* fp32 parameters (always required) */
  const void* h[MRNB_C_COUNT];  /* bf16 copies of the GEMM weight slots (conv1..6, W_ih, W_hh, linear) and conv0 as
                                   [I,64,64] = 36 taps (c,kh,kw) zero-padded to 64; MRNB_PREC_BF16 only */
  const float* fc_w[MRNB_MAX_EXPERTS];  /* [C_i,256] model.{i}.fc.weight */
  const void* fc_w16[MRNB_MAX_EXPERTS]; /* bf16 copy; MRNB_PREC_BF16 only */
  const float* fc_b[MRNB_MAX_EXPERTS];  /* [C_i] */
  int n_class[MRNB_MAX_EXPERTS];
} MrnbCrnnPack;

/* Classifier heads fc_i (modules/model.py:164,181) on the features left in `workspace` by the last
 * mrnb_svtr_experts_forward call (chunk = 0, same pack / B / prec; logits = NULL there).  route_index = NULL: every
 * expert for every sample.  route_index = device int32 [B] (the hard route of modules/model.py:383-393): only the
 * routed expert's head is evaluated per sample -- 1 / I of the classifier FLOPs and of the logits traffic; logits rows
 * of the other (expert, sample) pairs are left untouched, and mrnb_gate_combine never reads them for a one-hot gate.
 * Tensor-core mode runs all heads (ragged C_i) as ONE grouped launch when the bf16 weights fc_w16[i] are slices of one
 * allocation in expert order. */
int mrnb_svtr_heads(const MrnbSvtrPack* pack, int B, int prec, const int* route_index, float* const* logits,
                    const long* ld_logits, void* workspace, size_t workspace_bytes, cudaStream_t stream);
size_t mrnb_crnn_workspace_bytes(int n_experts, int B, int prec);

/* image [B,4,32,256] fp32 NCHW.  bn_batch_stats / update_running as in mrnb_svtr_experts_forward.
 * features: NULL or [B,I,63,256] fp32 (router input).  logits[i]: NULL or [B,63,ld_logits[i]] fp32 (model.{i} "predict"). */
int mrnb_crnn_experts_forward(const MrnbCrnnPack* pack, const float* image, int B, int prec, int bn_batch_stats,
                              int update_running, float* features, float* const* logits, const long* ld_logits,
                              void* workspace, size_t workspace_bytes, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * Stage-0 expert training: one CRNN expert (VGG + 2 x BidirectionalLSTM + CTC head), forward keeping activations +
 * full backward (convolution / pooling / BatchNorm gradients, BPTT through both LSTM layers).
 * Replaces il_modules/mrn.py:225-279 for FeatureExtraction="VGG", SequenceModeling="BiLSTM": the autograd graph of
 * modules/feature_extraction.py:19-47, modules/sequence_modeling.py:12-22, modules/model.py:82-101,133-148.
 *
 * Slots point into one flat fp32 arena (gradients: same slots in a second arena).  Convolution weights are
 * [Cout,kh,kw,Cin] (conv0 included); LSTM tensors keep nn.LSTM's gate order (i,f,g,o) with the forward direction
 * followed by the reverse direction IN THE SAME SLOT (adjacent in the arena). */
enum {
  MRNB_T_CONV0_W = 0, MRNB_T_CONV0_B, /* [64,3,3,4], [64]        ConvNet.0 */
  MRNB_T_CONV1_W, MRNB_T_CONV1_B,     /* [128,3,3,64]            ConvNet.3 */
  MRNB_T_CONV2_W, MRNB_T_CONV2_B,     /* [256,3,3,128]           ConvNet.6 */
  MRNB_T_CONV3_W, MRNB_T_CONV3_B,     /* [256,3,3,256]           ConvNet.8 */
  MRNB_T_CONV4_W, MRNB_T_BN4_W, MRNB_T_BN4_B, /* [512,3,3,256] (no bias), ConvNet.12 weight / bias */
  MRNB_T_CONV5_W, MRNB_T_BN5_W, MRNB_T_BN5_B, /* [512,3,3,512] (no bias), ConvNet.15 weight / bias */
  MRNB_T_CONV6_W, MRNB_T_CONV6_B,     /* [512,2,2,512]           ConvNet.18 */
  MRNB_T_LSTM0 = 16,                  /* 2 layers x MRNB_TL_COUNT slots: SequenceModeling.0, SequenceModeling.1 */
  MRNB_T_FC_W = 16 + 2 * 6, MRNB_T_FC_B, /* [C,256], [C]         fc */
  MRNB_T_COUNT
};
enum { /* per BidirectionalLSTM, Kin = 512 / 256 */
  MRNB_TL_WIH = 0, /* [2,1024,Kin]  rnn.weight_ih_l0, rnn.weight_ih_l0_reverse */
  MRNB_TL_WHH,     /* [2,1024,256]  rnn.weight_hh_l0, rnn.weight_hh_l0_reverse */
  MRNB_TL_BIH,     /* [2,1024]      rnn.bias_ih_l0, rnn.bias_ih_l0_reverse */
  MRNB_TL_BHH,     /* [2,1024]      rnn.bias_hh_l0, rnn.bias_hh_l0_reverse */
  MRNB_TL_LIN_W,   /* [256,512]     linear.weight */
  MRNB_TL_LIN_B,   /* [256] */
  MRNB_TL_COUNT
};
typedef struct MrnbCrnnTrainPack {
  const float* p[MRNB_T_COUNT]; /* fp32 parameters (or gradients) */
  const void* h[MRNB_T_COUNT];  /* bf16 copies of the GEMM weights at the same element offsets; MRNB_PREC_BF16 only */
  float* bn_mean[2];            /* ConvNet.12 / ConvNet.15 running_mean [512] (updated in train mode) */
  float* bn_var[2];
  int n_class;
} MrnbCrnnTrainPack;

size_t mrnb_crnn_train_workspace_bytes(int B, int n_class, int prec);
/* logits / dlogits: [B,63,ld] fp32. */
int mrnb_crnn_train_forward(const MrnbCrnnTrainPack* pack, const float* image, int B, int prec, int bn_batch_stats,
                            int update_running, float* logits, long ld_logits, void* workspace, size_t workspace_bytes,
                            cudaStream_t stream);
int mrnb_crnn_train_backward(const MrnbCrnnTrainPack* pack, const MrnbCrnnTrainPack* grads, const float* dlogits,
                             long ld_dlogits, int B, int prec, int bn_batch_stats, float* grad_arena, long n_arena,
                             void* workspace, size_t workspace_bytes, cudaStream_t stream);
/* As for SVTR: features / dfeatures NULL or [B,63,256] fp32 (dense), the second BiLSTM's output (modules/model.py:141). */
int mrnb_crnn_train_forward_features(const MrnbCrnnTrainPack* pack, const float* image, int B, int prec, int bn_batch_stats,
                                     int update_running, float* logits, long ld_logits, float* features, void* workspace,
                                     size_t workspace_bytes, cudaStream_t stream);
int mrnb_crnn_train_backward_features(const MrnbCrnnTrainPack* pack, const MrnbCrnnTrainPack* grads, const float* dlogits,
                                      long ld_dlogits, const float* dfeatures, int B, int prec, int bn_batch_stats,
                                      float* grad_arena, long n_arena, void* workspace, size_t workspace_bytes,
                                      cudaStream_t stream);
/* As mrnb_svtr_train_backward_input: the image gradient dimage (NULL or [B,4,32,256] fp32 NCHW, overwritten) is the input
 * gradient of VGG's conv0 (modules/feature_extraction.py:27, Conv2d(4, 64, 3, 1, 1)), returned in the caller's NCHW
 * layout although the forward runs on an NHWC copy of the image; grads = grad_arena = NULL: input-only backward. */
int mrnb_crnn_train_backward_input(const MrnbCrnnTrainPack* pack, const MrnbCrnnTrainPack* grads, const float* dlogits,
                                   long ld_dlogits, const float* dfeatures, int B, int prec, int bn_batch_stats,
                                   float* grad_arena, long n_arena, float* dimage, void* workspace, size_t workspace_bytes,
                                   cudaStream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * DM-Router + gate head.   Replaces modules/dm_router.py:50-67 (DM_Router.forward, both gating blocks) and
 * modules/model.py:402-406 (train) / :371-377 (eval): rearrange -> channel_route -> route -> softmax / argmax.
 *
 * Router parameters live in ONE fp32 arena (also the gradient / Adam / NCCL all-reduce layout); offsets in floats
 * are returned by mrnb_router_param_offsets in nn.Module.parameters() order (modules/model.py:437-452):
 *   0 route.weight[T] 1 route.bias[1] 2 channel_route.weight[I,I*D] 3 channel_route.bias[I]
 *   4 norm.weight[D] 5 norm.bias[D] 6 proj_1.weight[2D,D] 7 proj_1.bias[2D]
 *   8 spatial_gating.norm.weight[D] 9 .bias[D] 10 spatial_gating.proj.weight[IT,IT] 11 .bias[IT]
 *   12 channel_gating.norm.weight[T] 13 .bias[T] 14 channel_gating.proj.weight[ID,ID] 15 .bias[ID]
 *   16 proj_2.weight[D,D] 17 proj_2.bias[D] 18 proj_3.weight[D,D] 19 proj_3.bias[D]
 */
#define MRNB_ROUTER_NPARAMS 20
long mrnb_router_param_offsets(int n_experts, int T, int D, long* offsets /* host, [MRNB_ROUTER_NPARAMS+1] */);
size_t mrnb_router_workspace_bytes(int B, int n_experts, int T, int D, int with_backward);

/* x [B,I,T,D] fp32 -> out [B,I,T,D], scores r [B,I] (pre-softmax), gate = softmax(r) [B,I], index = argmax_j r (first max).
 * The workspace keeps the activations the backward needs. */
int mrnb_router_forward(const float* params, const float* x, int B, int n_experts, int T, int D, int prec,
                        float* out, float* scores, float* gate, int* index, void* workspace, size_t workspace_bytes,
                        cudaStream_t stream);

/* Backward of the stage-1 objective w.r.t. every router parameter (il_modules/mrn.py:342,360,362):
 *   loss = pi * CTC + CrossEntropy(gate, domain)   -- CE applied to the already softmaxed gate (reference quirk).
 * dgate_ctc [B,I] is d(pi*CTC)/dgate from mrnb_ctc_lattice; domain [B] int64.  Writes grads (same arena layout,
 * overwritten) and taski_loss (scalar, the CE term).  Must follow mrnb_router_forward with the same workspace.
 * domain == NULL: dgate_ctc (required) is the complete dL/dgate of an arbitrary loss, no CE term is added and
 * taski_loss may be NULL (autograd through MRNNet). */
int mrnb_router_backward(const float* params, const float* x, const float* gate, const float* dgate_ctc,
                         const long long* domain, int B, int n_experts, int T, int D, int prec, float* grads,
                         float* taski_loss, void* workspace, size_t workspace_bytes, cudaStream_t stream);

/* mrnb_router_backward plus the input gradient dx [B,I,T,D] fp32 = dL/dx through the gate head and the DM-Router (both
 * residuals included): the gradient reaching the experts' features when they are trained with the router
 * (modules/model.py:400-406 with nothing detached).  Parameter gradients as mrnb_router_backward's; in bf16 mode they
 * come from the materialised d_out (the generic DM-Router backward), not the rank-one gate-head path, so they agree
 * with mrnb_router_backward's within the bf16 budget rather than bitwise. */
int mrnb_router_backward_dx(const float* params, const float* x, const float* gate, const float* dgate_ctc,
                            const long long* domain, int B, int n_experts, int T, int D, int prec, float* grads, float* dx,
                            float* taski_loss, void* workspace, size_t workspace_bytes, cudaStream_t stream);

/* DM_Router alone with an explicit upstream gradient (tests): d_out [B,I,T,D] -> grads of the dm_router.0.*
 * slots (4..19) and, if dx != NULL, the input gradient. */
int mrnb_dm_router_backward(const float* params, const float* x, const float* d_out, int B, int n_experts, int T, int D,
                            int prec, float* grads, float* dx, void* workspace, size_t workspace_bytes, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * Gated combine + log-softmax + CTC + greedy decode.
 * Replaces modules/model.py:361-364,410-423 (pad with ONES, stack, gate-mul, sum), :383-393 (hard route = one-hot gate),
 *          il_modules/mrn.py:251-252,345-346 + il_modules/base.py:131 (log_softmax + CTCLoss(mean, zero_infinity)),
 *          test.py:211-221,257 + tools/utils.py:62-76 (argmax, collapse, confidence).
 *
 * mrnb_gate_combine: z[i] [B,T,ld[i]] (first Ci[i] columns valid; z, ld, Ci are HOST arrays), gate [B,I].
 *   Always writes lse [B,T].  Optional outputs (NULL to skip): logits [B,T,ldo] (the combined union-charset
 *   logits), E [B,T,I] = sum_c softmax(logits)[c] * pad_i[c], amax [B,T] (first maximal class), maxprob [B,T],
 *   lpe [B,T,Lmax+1] log-probs of blank + each target label, zlab [B,T,Lmax+1,I] per-expert values at those columns.
 *   targets [B,Lmax] int64 padded with 1, tlen [B] int32 (tools/utils.py:45-60). */
int mrnb_gate_combine(const float* const* z, const long* ld, const int* Ci, int n_experts, const float* gate, int B,
                      int T, float* logits, long ldo, float* lse, float* E, int* amax, float* maxprob,
                      const long long* targets, const int* tlen, int Lmax, float* lpe, float* zlab, cudaStream_t stream);

/* Backward of mrnb_gate_combine for a dense upstream gradient (autograd through MRNNet's soft route): dY [B,T,ldy] fp32
 * = dL/dlogits over the union charset C = Ci[n_experts-1] ->
 *   dgate [B,I],  dgate[b,i] = sum_{t, c<C} dY[b,t,c] * (c < Ci[i] ? z_i[b,t,c] : 1.0)   (pad with ones, quirk 1).
 * The gate is not an input: the combined logits are linear in it.  Every expert is read, a zero-gate one too.  Same
 * expert table as mrnb_gate_combine (z, ld, Ci host arrays; Ci[i] <= C); z[i] and dY 16-byte aligned, ld[i] and ldy
 * multiples of 4.  Deterministic (fixed reduction order, no atomics).
 * workspace: >= mrnb_gate_combine_backward_workspace_bytes(B, T, n_experts) (per-row partials). */
size_t mrnb_gate_combine_backward_workspace_bytes(int B, int T, int n_experts);
int mrnb_gate_combine_backward(const float* const* z, const long* ld, const int* Ci, int n_experts, int B, int T,
                               const float* dY, long ldy, float* dgate, void* workspace, size_t workspace_bytes,
                               cudaStream_t stream);
/* mrnb_gate_combine_backward plus the per-expert logit gradients in the same pass (trainable experts,
 * modules/model.py:410-423 differentiated w.r.t. z_i):  dz_i[b,t,c] = gate[b,i] * dY[b,t,c] for c < Ci[i].
 * gate [B,I]; dz, ldz HOST arrays [n_experts]: dz[i] = NULL skips expert i (frozen), otherwise [B,T,ldz[i]] fp32,
 * 16-byte aligned, ldz[i] >= Ci[i] a multiple of 4; columns Ci[i]..ldz[i] are never written.  dgate is bitwise the
 * value mrnb_gate_combine_backward returns. */
int mrnb_gate_combine_backward_experts(const float* const* z, const long* ld, const int* Ci, int n_experts, int B, int T,
                                       const float* dY, long ldy, const float* gate, float* const* dz, const long* ldz,
                                       float* dgate, void* workspace, size_t workspace_bytes, cudaStream_t stream);

/* CTC alpha-beta over all T frames, blank 0.  nll [B] (0 where infeasible: zero_infinity), loss_mean = mean_b(nll_b /
 * max(len_b,1)).  Optional: dgate [B,I] = grad_scale/max(len,1) * sum_t(E_i - sum_s occ_s * zlab_i[ext_s])  (pass
 * grad_scale = pi / B), occ_col [B,T,Lmax+1] posterior mass per label column (for mrnb_ctc_dense_grad). */
int mrnb_ctc_lattice(const float* lpe, const float* zlab, const float* E, const long long* targets, const int* tlen,
                     int Lmax, int B, int T, int n_experts, float grad_scale, float* nll, float* loss_mean, float* dgate,
                     float* occ_col, cudaStream_t stream);

/* Dense gradient of the mean CTC loss w.r.t. logits [B,T,C] (expert-training stage, il_modules/mrn.py:251-260). */
int mrnb_ctc_dense_grad(const float* logits, long ldl, const float* lse, const float* occ_col, const float* nll,
                        const long long* targets, const int* tlen, int Lmax, int B, int T, int C, float grad_scale,
                        float* grad, long ldg, cudaStream_t stream);

/* ids [B,T] compacted (collapse repeats, drop blank 0; -1 padded), len [B], conf [B] = prod_t maxprob[b,t]. */
int mrnb_greedy_decode(const int* amax, const float* maxprob, int B, int T, int* out_ids, int* out_len, float* conf,
                       cudaStream_t stream);

/* CTC prefix beam search (N-best decoding).  No counterpart in the reference: an addition to its greedy decode,
 * test.py:211-221.  Opt-in; the default decode stays mrnb_greedy_decode.
 *
 * mrnb_ctc_topk: per-frame candidate pruning on the same expert table and gate as mrnb_gate_combine (z, ld, Ci are HOST
 *   arrays; experts with a zero gate are not read) and the lse [B,T] it wrote.  The combined value is recomputed with
 *   the combine's expression, so top_ids[...,0] equals its amax wherever amax != 0.  Writes top_ids [B,T,K] int32 (the K
 *   non-blank classes with the highest combined value, ties to the smaller class; -1 past the C-1 real classes),
 *   top_lp [B,T,K] = value - lse (-inf in unused slots) and blank_lp [B,T].  1 <= K <= 32.
 * mrnb_ctc_beam_search: CTC prefix beam search in log space over blank + the K candidates of every frame, beam width W,
 *   the n_best best labelings out: ids [B,n_best,T] compact (-1 padded), len [B,n_best], score [B,n_best] = log p of
 *   the labeling over the kept alignments.  Ties: stay before extension, then the parent's rank, then the class index
 *   (class indices < 2^26).  1 <= K <= 32, 1 <= W <= 32, 1 <= n_best <= W, 1 <= T <= 128.  No workspace. */
int mrnb_ctc_topk(const float* const* z, const long* ld, const int* Ci, int n_experts, const float* gate, const float* lse,
                  int B, int T, int K, int* top_ids, float* top_lp, float* blank_lp, cudaStream_t stream);
int mrnb_ctc_beam_search(const int* top_ids, const float* top_lp, const float* blank_lp, int B, int T, int K, int W,
                         int n_best, int* out_ids, int* out_len, float* out_score, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * Image preparation on the device.  Replaces data/dataset.py:235-246 (ResizeNormalize: PIL Image.resize((imgW, imgH),
 * BICUBIC) on the RGBA crop -> torchvision ToTensor -> sub_(0.5).div_(0.5)) as applied per image by AlignCollate
 * (data/dataset.py:169-197); output bytes are identical to Pillow's (premultiplied-alpha two-pass fixed-point resampling).
 * pixels: packed RGBA rows of all images (device); offsets [B] (bytes, multiples of 4), widths / heights [B]: DEVICE
 * arrays.  max_w / max_h: the largest width / height in the batch (host values; bound the tap count and the
 * intermediate).  out: [B,4,out_h,out_w] fp32.  workspace: >= mrnb_resize_workspace_bytes(B, max_h, out_w). */
size_t mrnb_resize_workspace_bytes(int B, int max_h, int out_w);
int mrnb_resize_normalize_rgba(const unsigned char* pixels, const long long* offsets, const int* widths, const int* heights,
                               int B, int max_w, int max_h, int out_h, int out_w, float* out, void* workspace,
                               size_t workspace_bytes, cudaStream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * clip_grad_norm_(5) + Adam on a flat arena.  Replaces il_modules/mrn.py:364-367 (torch foreach kernels).
 * state: exp_avg, exp_avg_sq [n]; norm_out: device scalar receiving the pre-clip L2 norm.  step is 1-based. */
int mrnb_clip_adam(float* params, const float* grads, float* exp_avg, float* exp_avg_sq, long n, float lr, float beta1,
                   float beta2, float eps, float max_norm, int step, float* norm_out, void* workspace /* >= 4 KiB */,
                   cudaStream_t stream);

/* ---------------------------------------------------------------------------------------------------------
 * Building blocks (used by the entry points above; exported for the parity tests). */
int mrnb_linear_f32(const float* A, const float* W, const float* bias, const float* residual, float* out, int M, int N,
                    int K, int act_gelu, cudaStream_t stream);
/* tcgen05 / TMEM / TMA GEMM: A [M,K] bf16, W [N,K] bf16, out fp32 or bf16 [M,N]; K % 64 == 0. */
int mrnb_linear_bf16(const void* A, const void* W, const float* bias, const float* residual, void* out, int out_is_f32,
                     int M, int N, int K, int act_gelu, cudaStream_t stream);
/* General tcgen05 GEMM used by the router (MN-major operands, split-K): out[M,N] = A . B with A stored [M,K] (a_mn=0)
 * or [K,M] (a_mn=1), B stored [N,K] (b_mn=0) or [K,N] (b_mn=1), bf16; K % 64 == 0; out must be zeroed when splitk > 1. */
int mrnb_tc_gemm_general(const void* A, int a_mn, const void* B, int b_mn, float* out, int M, int N, int K, int splitk,
                         cudaStream_t stream);
/* Fused MLP branch (bf16 mode): x <- x + rs * (GELU(A W1^T + b1) W2^T + b2), A = LN2(x) and W1 bf16, W2 f16 (the GELU
 * output is an f16 tensor-core operand); optional
 * LayerNorm of the new x into ln_out (bf16 [M,D], D <= 128, may alias A).  Replaces modules/svtr.py:61-67,203. */
int mrnb_mlp_bf16(const void* A, const void* W1, const float* b1, const void* W2, const float* b2, float* x,
                  const float* rowscale, int rows_per_scale, void* ln_out, const float* ln_gamma, const float* ln_beta,
                  float ln_eps, int M, int D, cudaStream_t stream);
/* Fused SVTR mixer branch of one Block on the tensor cores (bf16 mode), one group of `units` samples:
 *   x <- x + rowscale[u] * ( proj( softmax(q k^T [+ Local 7x11 window]) v ) + bproj ),  q|k|v = A Wqkv^T + bqkv (q * 32^-0.5)
 * A = LN1(x) bf16 [units, N, D] with N = 32768 / D tokens on an (N/64) x 64 grid, head_dim 32; Wqkv bf16 [3D, D], Wproj
 * bf16 [D, D]; x fp32 [units, N, D] updated in place; optional ln_out = LN(x) (bf16, D <= 128, may alias A).
 * q, k, v, scores and probabilities stay on chip.  Replaces modules/svtr.py:133-152 + :201-203 (first branch). */
int mrnb_mixer_bf16(const void* A, const void* Wqkv, const float* bqkv, const void* Wproj, const float* bproj, float* x,
                    const float* rowscale, void* ln_out, const float* ln_gamma, const float* ln_beta, float ln_eps,
                    int units, int D, int local, cudaStream_t stream);
int mrnb_layernorm_f32(const float* x, float* y, const float* gamma, const float* beta, long rows, int D, float eps,
                       cudaStream_t stream);
int mrnb_svtr_attention_f32(const float* qkv, float* out, int groups, int N, int d, int heads, int H, int W, int local,
                            cudaStream_t stream);
/* tcgen05 attention (bf16 mode): qkv [groups*N, 3d] bf16 -> out [groups*N, d] bf16; N % 128 == 0, head_dim 32. */
int mrnb_svtr_attention_bf16(const void* qkv, void* out, int groups, int N, int d, int heads, int H, int W, int local,
                             cudaStream_t stream);
/* Training attention of one SVTR stage on the tensor cores (bf16 mode of the stage-0 step), head_dim 32, d = 32 * heads,
 * N in {128, 256, 512} tokens on an (N / W) x W grid, W a power of two >= 32.
 *   forward : qkv [B*N, 3d] bf16 -> P [B*heads, N, N] bf16 = softmax(32^-0.5 q k^T [+ Local 7x11 window]), O [B*N, d] bf16 = P v
 *   backward: dO fp32 and its bf16 copy dO16 [B*N, d], with the forward's qkv, O and P -> dS [B*heads, N, N] bf16 =
 *             P (dO v^T - dO.O), dqkv [B*N, 3d] bf16 = (dQ | dK | dV). */
int mrnb_attn_tc_train_forward(const void* qkv, void* P, void* O, int B, int N, int d, int heads, int W, int local,
                               cudaStream_t stream);
int mrnb_attn_tc_train_backward(const void* qkv, const void* O, const float* dO, const void* dO16, const void* P, void* dS,
                                void* dqkv, int B, int N, int d, int heads, cudaStream_t stream);
/* conv0 input-gradient kernels of the two backwards above, on their own: d = the fp32 gradient at conv0's output, NHWC
 * ([B,16,128,32] SVTR / [B,32,256,64] CRNN); w = the training pack's conv0 weight ([32,4,3,3] nn.Conv2d layout / [64,3,3,4]);
 * dimage [B,4,32,256] fp32 NCHW, every element overwritten.  One thread per pixel sums its taps and channels in a fixed
 * order: bitwise repeatable.  B <= 65535. */
int mrnb_svtr_conv0_dimage(const float* d, const float* w, float* dimage, int B, cudaStream_t stream);
int mrnb_crnn_conv0_dimage(const float* d, const float* w, float* dimage, int B, cudaStream_t stream);
int mrnb_cast_f32_to_bf16(const float* x, void* y, long n, cudaStream_t stream);
int mrnb_cast_f32_to_f16(const float* x, void* y, long n, cudaStream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* MRN_B200_H */
