// Shared host/device helpers for libaaconv_b200 (sm_100a only).
#pragma once

#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cstdint>
#include <cstdio>
#include <cstdarg>
#include <string>

#include "../../include/aaconv_b200.h"

namespace aaconv {

// ---- error plumbing (thread-local text, int codes across the ABI) ------------------------------
std::string& last_error_ref();
int fail(int code, const char* fmt, ...);

// A failed runtime call also leaves its error in the thread's last-error slot; it is consumed here, so that it is reported
// once, by this call, and not again by the next launch check (AACONV_LAUNCH_OK) of a later, unrelated call.
#define AACONV_CUDA_OK(expr)                                                                       \
  do {                                                                                             \
    cudaError_t e__ = (expr);                                                                      \
    if (e__ != cudaSuccess) {                                                                      \
      (void)cudaGetLastError();                                                                    \
      return ::aaconv::fail(AACONV_E_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #expr,          \
                            cudaGetErrorString(e__));                                              \
    }                                                                                              \
  } while (0)

// Called right after every kernel launch of this library: error check + launch accounting (+ optional
// per-launch CUDA-event profile, see aaconv_profile_begin/end).
void note_launch(const char* name, cudaStream_t st);
// Wraps the stream argument of every <<<...>>> launch: when the per-launch profile is on it records the launch's START event
// (so host-side gaps between launches are not charged to the next kernel); returns `st` unchanged.
cudaStream_t pre_launch(cudaStream_t st);
#define AACONV_ST(stream__) ::aaconv::pre_launch(stream__)
#define AACONV_LAUNCH_OK_ON(name, stream__)                                                        \
  do {                                                                                             \
    cudaError_t e__ = cudaGetLastError();                                                          \
    if (e__ != cudaSuccess)                                                                        \
      return ::aaconv::fail(AACONV_E_CUDA, "%s:%d launch %s -> %s", __FILE__, __LINE__, name,     \
                            cudaGetErrorString(e__));                                              \
    ::aaconv::note_launch(name, stream__);                                                         \
  } while (0)
#define AACONV_LAUNCH_OK(name) AACONV_LAUNCH_OK_ON(name, st)

// NVTX range around one stage of a forward / backward call (header-only NVTX v3: no extra library; a no-op unless a tool such
// as nsys / ncu --nvtx is attached).  Stage names: aaconv.prologue, .fprop, .aug_build, .attention, .epilogue, .out_bwd,
// .attention_bwd, .rel_bwd, .dgrad, .wgrad, .prologue_bwd
struct NvtxRange {
  explicit NvtxRange(const char* name);
  ~NvtxRange();
};

#define AACONV_TRY(expr)                                                                           \
  do {                                                                                             \
    int r__ = (expr);                                                                              \
    if (r__ != 0) return r__;                                                                      \
  } while (0)

// ---- derived dimensions ------------------------------------------------------------------------
struct Dims {
  int B, Cin, Hin, Win, Cout, H, W, ks, stride, pad, dil, dk, dv, nh, relative;
  int dkh, dvh, L, Cc /*conv-branch channels*/, Nqkv, BN /*B*nh*/, RW, RH;
  float qscale;
  // I/O description (aaconv_io): element types of x / y, batch stride of y, fused InstanceNorm + ReLU prologue
  int x_bf16 = 0, y_bf16 = 0, fuse_in = 0;
  long long y_bs = 0;
  float in_eps = 1e-5f;
  __host__ Dims(const aaconv_dims& d, const aaconv_io* io) : Dims(d) {
    if (io) {
      x_bf16 = io->x_dtype == AACONV_BF16;
      y_bf16 = io->y_dtype == AACONV_BF16;
      fuse_in = io->fuse_in_relu != 0;
      in_eps = io->in_eps > 0.f ? io->in_eps : 1e-5f;
      if (io->y_batch_stride > 0) y_bs = io->y_batch_stride;
    }
  }
  __host__ explicit Dims(const aaconv_dims& d)
      : B(d.B), Cin(d.Cin), Hin(d.Hin), Win(d.Win), Cout(d.Cout), H(d.H), W(d.W), ks(d.ksize),
        stride(d.stride), pad(d.pad), dil(d.dil), dk(d.dk), dv(d.dv), nh(d.nh), relative(d.relative) {
    dkh = nh > 0 ? dk / nh : 0;
    dvh = nh > 0 ? dv / nh : 0;
    L = H * W;
    Cc = Cout > dv ? Cout - dv : 0;
    Nqkv = 2 * dk + dv;
    BN = B * nh;
    RW = 2 * W - 1;
    RH = 2 * H - 1;
    qscale = dkh > 0 ? 1.0f / sqrtf((float)dkh) : 0.f;
    y_bs = (long long)Cout * L;
  }
};

// y element store: fp32 or bf16 destination selected at run time (the y tensor is small; the branch is uniform)
#ifdef __CUDACC__
__device__ __forceinline__ void store_y(void* y, size_t idx, float v, int bf16_out) {
  if (bf16_out) static_cast<__nv_bfloat16*>(y)[idx] = __float2bfloat16(v);
  else static_cast<float*>(y)[idx] = v;
}
// BatchNorm2d in eval mode as one affine map per channel: (s_c, t_c) with y = x s_c + t_c, s_c = weight_c / sqrt(running_var_c + eps)
// (IEEE division and square root), t_c = bias_c - running_mean_c s_c
__device__ __forceinline__ float2 bn_eval_affine(const float* __restrict__ weight, const float* __restrict__ bias,
                                                 const float* __restrict__ running_mean, const float* __restrict__ running_var, float eps,
                                                 int c) {
  const float s = weight[c] / sqrtf(running_var[c] + eps);
  return make_float2(s, bias[c] - running_mean[c] * s);
}
#endif

inline size_t align256(size_t n) { return (n + 255) & ~size_t(255); }

// Bump allocator over a caller-owned buffer.
struct Carver {
  char* base;
  size_t off = 0;
  explicit Carver(void* b) : base(static_cast<char*>(b)) {}
  template <class T>
  T* take(size_t count) {
    T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
    off += align256(count * sizeof(T));
    return p;
  }
};

inline int cdiv(int a, int b) { return (a + b - 1) / b; }

// relu(BatchNorm2d eval) NCHW (batch stride xbs) -> dense NCHW, any C / HW / alignment (bn_relu.cu; aaconv_bn_relu_eval dispatches)
int bn_relu_eval_nchw(const void* x, int dtype, int B, int C, int HW, long long xbs, const float* weight, const float* bias,
                      const float* running_mean, const float* running_var, float eps, void* y, cudaStream_t st);

}  // namespace aaconv
