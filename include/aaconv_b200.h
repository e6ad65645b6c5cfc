/*
 * aaconv_b200.h -- C ABI of the B200-native AAConv2d hot path (libaaconv_b200.so).
 *
 * The reference (kamenbliznashki/chexpert) has no FFI layer: the boundary it exposes for this path is
 * the nn.Module contract of AAConv2d (models/attn_aug_conv.py:19-100) and the loss callable
 * (chexpert.py:530,160).  This header is what a Python/ctypes (or any FFI) host binds instead of the
 * ATen ops those lines call.  Every entry point
 *   - takes plain device pointers, ints and a CUDA stream handle (void* == cudaStream_t); no torch types;
 *   - returns 0 on success, a negative AACONV_E_* code otherwise (aaconv_last_error() has the text);
 *   - never allocates persistent device memory: outputs, the saved-for-backward block and scratch are
 *     caller-owned buffers sized by the *_bytes() queries;
 *   - is asynchronous on `stream` and holds no global mutable state (safe from the autograd worker thread).
 *
 * Tensor layouts at the boundary are the reference's: x (B,Cin,Hin,Win) and y (B,Cout,H,W) contiguous
 * NCHW, parameters in their state_dict shapes (attn_aug_conv.py:34-41).  fp32 everywhere at the boundary;
 * `precision` selects the arithmetic inside (AACONV_FP32: fp32 FFMA path, rtol 1e-4 parity;
 * AACONV_BF16: bf16 tcgen05 tensor-core path with fp32 accumulation and fp32 softmax statistics).
 */
#ifndef AACONV_B200_H_
#define AACONV_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AACONV_ABI_VERSION 2

enum { AACONV_FP32 = 0, AACONV_BF16 = 1 };

enum {
  AACONV_OK = 0,
  AACONV_E_ARG = -1,       /* bad dimension / null pointer / unsupported configuration */
  AACONV_E_CUDA = -2,      /* a CUDA runtime call or launch failed */
  AACONV_E_UNSUPPORTED = -3
};

/* Static description of one AAConv2d call.  Mirrors the constructor arguments of
 * attn_aug_conv.py:20 plus the input extent; H,W are the post-stride map == input_dims when relative. */
typedef struct aaconv_dims {
  int32_t B, Cin, Hin, Win;
  int32_t Cout;            /* out_channels of the module (conv branch gets Cout-dv, attention dv) */
  int32_t H, W;            /* output map: floor((Hin-1)/stride)+1, ... (attn_aug_conv.py:35,70)      */
  int32_t ksize, stride, pad, dil;
  int32_t dk, dv, nh;
  int32_t relative;        /* attn_aug_conv.py:76 */
} aaconv_dims;

/* Parameter block, state_dict order of attn_aug_conv.py:34-41.  conv_w may be NULL iff Cout <= dv
 * (attn_aug_conv.py:34 -> self.conv is None); key_rel_* are ignored when !relative. */
typedef struct aaconv_params {
  const float* conv_w;     /* (Cout-dv, Cin, k, k) */
  const float* qkv_w;      /* (2dk+dv, Cin, 1, 1)  */
  const float* out_w;      /* (dv, dv, 1, 1)       */
  const float* key_rel_h;  /* (dk/nh, 2H-1)        */
  const float* key_rel_w;  /* (dk/nh, 2W-1)        */
} aaconv_params;

typedef struct aaconv_param_grads {   /* any member may be NULL: that gradient is skipped */
  float* conv_w;
  float* qkv_w;
  float* out_w;
  float* key_rel_h;
  float* key_rel_w;
} aaconv_param_grads;

/* Optional I/O description of one call (NULL = the defaults: fp32 x / y, dense y, no fused prologue).  It lets the module sit
 * inside the DenseNet the way north_star (4) and SURVEY.md section 8 rows f1 / f3 ask:
 *   x_dtype / y_dtype   element type of x (and dx) / of y: AACONV_FP32 or AACONV_BF16 (bf16 activations under autocast);
 *                        dy and the parameters stay fp32.
 *   y_batch_stride      elements between consecutive samples of y; 0 = Cout*H*W.  With Ctot*H*W the call writes the first Cout
 *                        channels of a wider (B,Ctot,H,W) feature buffer -- the pre-allocated DenseBlock buffer that replaces
 *                        torch.cat (torchvision densenet.py:48,120-124; attn_aug_conv.py:479-482) -- straight from the epilogues.
 *   fuse_in_relu        1: x is the INPUT of the Transition's InstanceNorm2d (affine=False, eps) + ReLU (attn_aug_conv.py:438-439);
 *                        forward computes the per-(b,c) mean / rstd and applies relu((x-mean)*rstd) while packing the GEMM operand,
 *                        backward returns the gradient with respect to that raw x (ReLU mask + InstanceNorm adjoint fused). */
typedef struct aaconv_io {
  int32_t x_dtype, y_dtype;
  int64_t y_batch_stride;
  int32_t fuse_in_relu;
  float in_eps;
} aaconv_io;

int aaconv_abi_version(void);
const char* aaconv_last_error(void);          /* thread-local text of the last failing call */
int aaconv_validate(const aaconv_dims* d, int precision);

/* Sizes of the caller-owned work buffers (bytes; multiples of 256). */
size_t aaconv_saved_bytes(const aaconv_dims* d, int precision);     /* forward -> backward state       */
size_t aaconv_scratch_bytes(const aaconv_dims* d, int precision, int want_weights);  /* transient, either direction;
                                                           want_weights: forward will also fill `weights` */
size_t aaconv_saved_bytes_io(const aaconv_dims* d, int precision, const aaconv_io* io);
size_t aaconv_scratch_bytes_io(const aaconv_dims* d, int precision, const aaconv_io* io);

/* Byte offsets of the named blocks inside the saved buffer (for tests and the visualise path).
 * names: "q","k","v","o","lse" (fp32 path: q,k (B,nh,L,dkh) with q pre-scaled; v,o (B,nh,L,dvh);
 * lse (B,nh,L)).  Returns -1 for an unknown name. */
int64_t aaconv_saved_offset(const aaconv_dims* d, int precision, const char* name);

/* Forward: replaces AAConv2d.forward (attn_aug_conv.py:65-97).
 *   y        (B,Cout,H,W)   conv channels first, attention channels last (attn_aug_conv.py:95)
 *   weights  optional (B,nh,HW,HW) softmax probabilities -- the tensor the reference stashes as
 *            self.weights (attn_aug_conv.py:87); NULL = do not materialise it.                       */
int aaconv_forward(const aaconv_dims* d, int precision, const float* x, const aaconv_params* p,
                   float* y, float* weights, void* saved, void* scratch, void* stream);

/* Backward: the adjoint autograd derives from attn_aug_conv.py:65-97 (SURVEY.md section 8a).
 *   dy (B,Cout,H,W); dx (B,Cin,Hin,Win) or NULL; parameter grads are WRITTEN (not accumulated).
 *   `saved` is the block forward filled; the bf16 path completes its backward-only columns in place (idempotent:
 *   backward may be called again on the same block, e.g. under retain_graph).                        */
int aaconv_backward(const aaconv_dims* d, int precision, const float* x, const aaconv_params* p,
                    const float* dy, void* saved, void* scratch,
                    float* dx, const aaconv_param_grads* g, void* stream);

/* The same two calls with an I/O description (see aaconv_io): x / dx in io->x_dtype, y in io->y_dtype at io->y_batch_stride,
 * optional fused InstanceNorm + ReLU prologue.  dy stays fp32 dense (B,Cout,H,W).  Buffers sized by the *_bytes_io() queries. */
int aaconv_forward_io(const aaconv_dims* d, int precision, const aaconv_io* io, const void* x, const aaconv_params* p,
                      void* y, float* weights, void* saved, void* scratch, void* stream);
int aaconv_backward_io(const aaconv_dims* d, int precision, const aaconv_io* io, const void* x, const aaconv_params* p,
                       const float* dy, void* saved, void* scratch, void* dx, const aaconv_param_grads* g, void* stream);

/* Loss: replaces nn.BCEWithLogitsLoss(reduction='none')(z,t) [.sum(1).mean(0)]  (chexpert.py:530,160,205).
 *   z (B,C) logits.  Targets are either
 *     targets (B,C) floats in {0,1} (already U-Ones'd, dataset.py:139,142), with cols == NULL, or
 *     raw labels (B,ld) in {nan,-1,0,1} with cols[C] the selected columns (dataset.py:25): the kernel
 *     applies blank->0 and -1->1 itself.
 *   element_loss (B,C) or NULL; loss scalar (sum over classes, mean over batch) or NULL;
 *   dz (B,C) or NULL = d loss / d z * grad_scale[0] (grad_scale NULL = 1).                           */
int aaconv_bce_forward_backward(const float* z, const float* targets, int ld, const int32_t* cols,
                                int B, int C, float* element_loss, float* loss, float* dz,
                                const float* grad_scale, void* stream);

/* Ensemble evaluation (SURVEY.md section 8 row f4): replaces torch.stack(outputs, 2).mean(2) (chexpert.py:233) and the
 * per-class sklearn roc_curve + auc on raw logits (chexpert.py:130-135).
 *   aaconv_ensemble_mean  logits (n_models, N, C) -> mean (N, C), summed in checkpoint order.
 *   aaconv_auroc          logits (N, C), targets (N, C) in {0,1} -> auroc (C): tie-corrected pair counting in integers
 *                         (== area under sklearn's ROC polygon); NaN for a class with a single label value.
 *                         workspace: aaconv_auroc_workspace_bytes(C) bytes of device memory.                  */
int aaconv_ensemble_mean(const float* logits, int n_models, int N, int C, float* mean, void* stream);
size_t aaconv_auroc_workspace_bytes(int C);
int aaconv_auroc(const float* logits, const float* targets, int N, int C, float* auroc, void* workspace, void* stream);

/* Dense-block side of the feature buffer (SURVEY.md section 8 row f3): BatchNorm2d in TRAINING mode (batch statistics, as
 * nn.BatchNorm2d does under model.train(): torchvision densenet.py:36,40 inside models/attn_aug_conv.py:479-482) fused with the
 * ReLU that follows it, reading its input THROUGH a batch stride -- layer i of a block normalises channels [0, c_i) of the
 * (B, C_total, H, W) feature buffer in place of torch.cat's copy.  x: (B, C, HW) elements of `dtype` (AACONV_FP32 | AACONV_BF16)
 * with x_batch_stride >= C*HW elements between samples; y, dy, dx dense (B, C, HW) of the same dtype; weight, bias,
 * running_mean, running_var (C) fp32 (running_* may both be NULL; updated with `momentum`, unbiased variance);
 * saved: (C) x (mean, rstd) fp32 written by forward for backward; workspace: aaconv_bn_relu_workspace_bytes(B, C) bytes.
 * forward keeps the per-(channel, sample) plane statistics in the first 8*B*C bytes of `workspace`, channel-major; with
 * stats_valid_channels = n > 0 the caller asserts that the entries of channels [0, n) already hold the statistics of THIS input
 * (a dense block passes the same buffer from layer to layer: channels [0, c_{i-1}) were reduced by the previous layer), and only
 * channels [n, C) are reduced.
 * backward: dx may be NULL; dweight / dbias (C) are WRITTEN (may be NULL).  All reductions run in a fixed order. */
size_t aaconv_bn_relu_workspace_bytes(int B, int C);
int aaconv_bn_relu_forward(const void* x, int dtype, int B, int C, int HW, int64_t x_batch_stride, const float* weight, const float* bias,
                           float* running_mean, float* running_var, float momentum, float eps, void* y, float* saved, void* workspace,
                           int stats_valid_channels, void* stream);
int aaconv_bn_relu_backward(const void* x, int dtype, int B, int C, int HW, int64_t x_batch_stride, const void* dy, const float* saved,
                            const float* weight, const float* bias, void* dx, float* dweight, float* dbias, void* workspace, void* stream);
/* The same with dx ACCUMULATED onto a gradient that is already in memory: gacc (B, C, HW) elements of `dtype` with g_batch_stride >= C*HW
 * elements between samples -- the gradient of the dense block's feature buffer, of which this layer's input is a channel prefix
 * (replaces the dense dx + the add autograd would run for the two consumers of the concatenated features, tv densenet.py:48,120-124). */
int aaconv_bn_relu_backward_acc(const void* x, int dtype, int B, int C, int HW, int64_t x_batch_stride, const void* dy, const float* saved,
                                const float* weight, const float* bias, void* gacc, int64_t g_batch_stride, float* dweight, float* dbias,
                                void* workspace, void* stream);

/* Channels-last side of the dense layers (chexpert_b200/csrc/bn_cl.cu): cuDNN's tensor-core convolutions are NHWC kernels, so the
 * BatchNorm + ReLU passes hand them NHWC tensors and take NHWC gradients back instead of leaving ~10 layout transposes per layer
 * to cuDNN.  C and HW multiples of 4, tensors aligned for four-element accesses, C <= 4096 when x is NHWC.
 *   aaconv_bn_stats_nchw        group statistics of channels [stats_valid_channels, C) of an NCHW (batch-strided) input into the
 *                               shared per-block buffer (layout of aaconv_bn_relu_forward); returns the group geometry
 *   aaconv_bn_relu_cl_forward   y (NHWC) = relu(bn(x)); x NHWC dense (x_is_cl = 1: statistics computed here) or NCHW with a batch
 *                               stride (x_is_cl = 0: statistics from aaconv_bn_stats_nchw in nchw_stats)
 *   aaconv_bn_relu_cl_backward  dy NHWC; dx NHWC dense (x_is_cl = 1) or NCHW through dx_batch_stride, ADDED when dx_accumulate
 *   aaconv_slice_layout         a channel slice between NHWC dense and NCHW with a batch stride (the block's concatenation)
 *   workspace: aaconv_bn_relu_cl_workspace_bytes(B, C, HW) bytes. */
size_t aaconv_bn_relu_cl_workspace_bytes(int B, int C, int HW);
int aaconv_bn_stats_nchw(const void* x, int dtype, int B, int C, int HW, int64_t x_batch_stride, void* workspace, int stats_valid_channels,
                         int* groups, int* planes_per_group, void* stream);
int aaconv_bn_relu_cl_forward(const void* x, int dtype, int B, int C, int HW, int x_is_cl, int64_t x_batch_stride, const float* weight,
                              const float* bias, float* running_mean, float* running_var, float momentum, float eps, void* y_cl, float* saved,
                              void* workspace, const void* nchw_stats, int stats_groups, int planes_per_group, void* stream);
int aaconv_bn_relu_cl_backward(const void* x, int dtype, int B, int C, int HW, int x_is_cl, int64_t x_batch_stride, const void* dy_cl,
                               const float* saved, const float* weight, const float* bias, void* dx, int64_t dx_batch_stride,
                               int dx_accumulate, float* dweight, float* dbias, void* workspace, void* stream);
int aaconv_slice_layout(const void* src, void* dst, int dtype, int B, int C, int HW, int64_t nchw_batch_stride, int to_nchw, void* stream);

/* relu(BatchNorm2d in EVAL mode): y = max(x * s_c + t_c, 0), s_c = weight_c / sqrt(running_var_c + eps), t_c = bias_c - running_mean_c * s_c.
 * x: (B, C, HW) NCHW with x_batch_stride >= C*HW (a channel prefix of the feature buffer), or NHWC dense (x_is_cl = 1).
 * y: dense, NCHW (y_is_cl = 0) or NHWC (y_is_cl = 1), same dtype as x (AACONV_FP32 | AACONV_BF16).  Supported pairs:
 * NCHW -> NCHW (any C, HW, alignment), NCHW -> NHWC and NHWC -> NHWC (C, HW multiples of 4, four-element aligned, NHWC C <= 4096).
 * Reads the running statistics, never writes them; no workspace. */
int aaconv_bn_relu_eval(const void* x, int dtype, int B, int C, int HW, int x_is_cl, int64_t x_batch_stride,
                        const float* weight, const float* bias, const float* running_mean, const float* running_var,
                        float eps, void* y, int y_is_cl, void* stream);

/* The Transition of torchvision's DenseNet (BatchNorm2d -> ReLU -> Conv2d 1x1 -> AvgPool2d(2), tv densenet.py:98-104) with the pool
 * moved ahead of the 1x1 convolution, which it commutes with: P = avgpool2(relu(bn(x))), the caller convolves P.
 * x: (B, C, H, W) NCHW of `dtype` (AACONV_FP32 | AACONV_BF16) with x_batch_stride >= C*H*W elements between samples (the finished
 * feature buffer of a dense block).  P, dP: (B, H/2, W/2, C) NHWC dense, floor mode (an odd last row / column is in no window).
 * C a multiple of 4, H and W >= 2, B <= 65535, every tensor and batch stride aligned for four-element accesses.
 *   aaconv_bn_relu_pool_forward   training != 0: batch statistics over ALL H*W pixels from the group statistics of
 *                                 aaconv_bn_stats_nchw in nchw_stats (stats_groups, planes_per_group as it returns them; a dense block's
 *                                 shared buffer with only the channels it has not reduced added); writes saved (C) x (mean, rstd) and
 *                                 updates running_mean / running_var (may both be NULL) as nn.BatchNorm2d does (momentum, unbiased
 *                                 variance).  training == 0: BatchNorm2d in eval mode from the running statistics, which are read,
 *                                 never written (saved, nchw_stats unused).
 *   aaconv_bn_relu_pool_backward  (training mode) dP -> dx for EVERY pixel of x (the dropped row / column gets the mean terms),
 *                                 through dx_batch_stride, ADDED onto what is there when dx_accumulate; dx may be NULL.  dweight / dbias
 *                                 (C) are WRITTEN (may be NULL).  Fixed-order reductions.
 *   workspace: aaconv_bn_relu_pool_workspace_bytes(B, C, H, W) bytes (backward only). */
size_t aaconv_bn_relu_pool_workspace_bytes(int B, int C, int H, int W);
int aaconv_bn_relu_pool_forward(const void* x, int dtype, int B, int C, int H, int W, int64_t x_batch_stride, int training,
                                const float* weight, const float* bias, float* running_mean, float* running_var, float momentum, float eps,
                                void* y_cl, float* saved, const void* nchw_stats, int stats_groups, int planes_per_group, void* stream);
int aaconv_bn_relu_pool_backward(const void* x, int dtype, int B, int C, int H, int W, int64_t x_batch_stride, const void* dP_cl,
                                 const float* saved, const float* weight, const float* bias, void* dx, int64_t dx_batch_stride,
                                 int dx_accumulate, float* dweight, float* dbias, void* workspace, void* stream);

/* Accounting / measurement helpers used by bench.py (no reference counterpart).
 *   aaconv_launch_count   kernels launched by this library since it was loaded (all threads).
 *   aaconv_profile_begin  start recording a (start, stop) CUDA-event pair around every launch (`stream` is unused, kept for ABI).
 *   aaconv_profile_end    stop; fills ms[i] = device time of launch i (its own start -> stop event) and the
 *                         '\n'-joined kernel names; returns the number of entries written (<= max_entries). */
long long aaconv_launch_count(void);
/* Debug hooks of the attention kernels (tools/attn_timeline.py, tools/attn_ablate.py); both default to off.
 *   aaconv_debug_set_timeline  device buffer of 16 x 96 int64: clock64 stamps of one persistent CTA of the dQa kernel (NULL = off)
 *   aaconv_debug_set_mode      ablation bits: 1 no MUFU, 2 no global traffic after the first tiles, 4 no gradient MMAs,
 *                              8 no math, 32 dQa drain without the bulk store -- results are WRONG when bits 1-8 are set; 16 = soft
 *                              mbarrier timeouts (see aaconv_debug_read_mbar_log)                                          */
void aaconv_debug_set_timeline(void* device_buffer);
void aaconv_debug_set_mode(int mode);
/*   aaconv_debug_read_mbar_log  with mode bit 16 set, a timed-out mbarrier wait in the small-value-width attention kernels is
 *                              logged instead of trapping; returns how many were logged, out[i] = smem barrier address << 32 |
 *                              parity << 31 | block << 12 | thread                                                    */
int aaconv_debug_read_mbar_log(unsigned long long* out, int max_entries);
int aaconv_profile_begin(void* stream);
int aaconv_profile_end(char* names_buf, size_t names_len, float* ms, int max_entries);

#ifdef __cplusplus
}
#endif
#endif  /* AACONV_B200_H_ */
