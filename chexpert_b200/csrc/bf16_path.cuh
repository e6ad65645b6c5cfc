// Internal interface of the bf16 tcgen05 path.
#pragma once
#include "common.cuh"

namespace aaconv {

// Column layout of the augmented attention operands (see attn_tc_bwd.cu).
struct AugLayout {
  int KD;   // dkh (+ W + H when relative): columns that form the logit
  int C1;   // start of the V block = roundup16(KD + 2)
  int KP;   // padded row length (multiple of 64)
  int NQ;   // roundup16(KD): width of the dQa accumulator
};

AugLayout aug_layout(const Dims& d);
int aug_supported(const Dims& d);
// aug_ops.cu
int aug_build_fwd(const Dims& d, const float* q, const float* k, const float* v, const float* krw, const float* krh,
                  void* qa, void* ka, cudaStream_t st);
// aug_tc.cu: the same operands from a tcgen05 (kind::tf32) product + per-row window; square maps of 10/20/40/64, dk/nh = 20
int aug_build_tc_supported(const Dims& d);
int aug_build_tc(const Dims& d, const float* q, const float* k, const float* v, const float* krw, const float* krh,
                 void* qa, void* ka, cudaStream_t st);
// aug_tc.cu: tcgen05 version of rel_bwd (bf16 packed output only); partials in rel_bwd's layout, summed by rel_bwd_reduce
int rel_bwd_tc_supported(const Dims& d, int KPq);
int rel_bwd_tc(const Dims& d, const float* dqa, const float* q, const float* krw, const float* krh, void* dqkvh, int KPq,
               float* partial, int RP, int DK8, int* nparts, cudaStream_t st);
int rel_bwd_reduce(const Dims& d, const float* partial, int nparts, int RP, int DK8, float* dkrw, float* dkrh, cudaStream_t st);
// (B,nh,L,L) softmax map from the bf16 operands and the bf16 forward kernel's lse (visualise path)
int aug_weights(const Dims& d, const void* qa, const void* ka, const float* lse, float* weights, cudaStream_t st);
// out_proj adjoint (dO, dWout) + the backward-only columns of Qa (-lse, dO, -delta) in one pass (nh = 8, dv/nh <= 2); partial: out_bwd_patch_partial_floats
int out_bwd_patch_supported(const Dims& d);
size_t out_bwd_patch_partial_floats(const Dims& d);
int out_bwd_patch(const Dims& d, const float* dy, const float* o, const float* lse, const float* wout, float* d_o, float* delta,
                  void* qa, float* dw, float* partial, cudaStream_t st);
int out_proj_fwd(const Dims& d, const float* o, const float* wout, void* y, cudaStream_t st);   // attention channels of y
// any value width: data part of the out_proj adjoint + the patch (dWout: f32_out_bwd_weight)
int out_bwd_data_patch(const Dims& d, const float* dy, const float* o, const float* lse, const float* wout, float* d_o, float* delta,
                       void* qa, cudaStream_t st);
int rel_bwd_supported(const Dims& d);
size_t rel_bwd_partial_floats(const Dims& d);
int rel_bwd(const Dims& d, const float* dqa, const float* q, const float* krw, const float* krh, float* dq, void* dqkvh,
            int KPq, float* dkrw, float* dkrh, float* partial, cudaStream_t st);
// dk/dv go to fp32 head-split tensors, or (dqkvh != NULL) as bf16 straight into the packed (B*L, KPq) projection-gradient operand
int tc_attn_bwd(const Dims& d, const void* qa, const void* ka, float* dqa, float* dk, float* dv, void* dqkvh, int KPq,
                cudaStream_t st);
int aug_bwd_dq(const Dims& d, const float* dqa, const float* krw, const float* krh, float* dq, cudaStream_t st);

// attn_cc.cu: value width <= 2 -- value terms on the CUDA cores, score/gradient contractions on tcgen05
int cc_attn_supported(const Dims& d);
int cc_attn_fwd(const Dims& d, const void* qa, const void* ka, const float* v, float* o, float* lse, cudaStream_t st);
int cc_attn_bwd(const Dims& d, const void* qa, const void* ka, const float* v, const float* d_o, const float* delta, float* dqa,
                float* dk, float* dv, void* dqkvh, int KPq, cudaStream_t st);

// attn_tc.cu (forward)
int tc_attn_supported(const Dims& d);
int tc_attn_fwd(const Dims& d, const void* qa, const void* ka, float* o, float* lse, cudaStream_t st);

// gemm_tc.cu (tcgen05 implicit GEMMs)
struct TcGemmBufs {
  void *xh, *dyh, *dqkvh, *wf, *wd, *wq;
  int NPc, NPq, CinP, CinK, KPc, KPq;
  size_t bytes;
};
int tc_gemm_supported(const Dims& d);
TcGemmBufs tc_gemm_bufs(const Dims& d, void* base);
int pack_nhwc_bf16(const float* in, void* out, int B, int C, int Cp, int HW, cudaStream_t st);
// t.xh must hold the packed (optionally normalised) x of this call (pack_x); y: d.y_bf16 / d.y_bs
int tc_fprop(const Dims& d, const TcGemmBufs& t, const float* conv_w, const float* qkv_w, void* y,
             float* q, float* k, float* v, cudaStream_t st);
int tc_pack_grads(const Dims& d, const TcGemmBufs& t, const float* dy, const float* dq, const float* dk, const float* dv,
                  cudaStream_t st);   // dq == NULL: dqkvh was already written by the attention backward kernels
int tc_dgrad(const Dims& d, const TcGemmBufs& t, const float* conv_w, const float* qkv_w, void* dx, int dx_bf16, cudaStream_t st);
int tc_zero_class(const Dims& d, void* dx, int dx_bf16, int rh, int rw, cudaStream_t st);
int tc_wgrad_supported(const Dims& d);
size_t tc_wgrad_partial_floats(const Dims& d);
int tc_wgrad(const Dims& d, const TcGemmBufs& t, float* dwc, float* dwq, float* partial, cudaStream_t st);

// prologue.cu: fused InstanceNorm + ReLU prologue of the Transition (attn_aug_conv.py:438-439) and the typed x / dx boundary
int in_stats(const Dims& d, const void* x, float* stats, cudaStream_t st);                      // stats: (B*Cin) x (mean, rstd)
int pack_x(const void* in, int in_bf16, const float* stats, void* out, int B, int C, int Cp, int HW, cudaStream_t st);
int in_relu_apply(const Dims& d, const void* x, const float* stats, float* out, cudaStream_t st);
int in_relu_bwd(const Dims& d, const void* x, const void* g, int g_bf16, const float* stats, void* dx, cudaStream_t st);

// fp32_gemms.cu
int aug_rel_weight_grad(const Dims& d, const float* q, const float* dqa, int KD, int axis, float* dkr, float* partial,
                        cudaStream_t st);

// bf16_path.cu
size_t bf16_saved_bytes(const Dims& d);
size_t bf16_scratch_bytes(const Dims& d, int want_weights);
int64_t bf16_saved_offset(const Dims& d, const char* name);
int bf16_forward(const Dims& d, const void* x, const aaconv_params* p, void* y, float* weights, void* saved,
                 void* scratch, cudaStream_t st);
int bf16_backward(const Dims& d, const void* x, const aaconv_params* p, const float* dy, void* saved,
                  void* scratch, void* dx, const aaconv_param_grads* g, cudaStream_t st);
}  // namespace aaconv
