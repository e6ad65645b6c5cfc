// Grad-CAM at features.norm5 of the DenseNets (the data part of chexpert.py:260-361: grad_cam / visualize), from the tensors the
// fused eval step already holds.  The head is norm5 -> relu -> global average pool -> Linear, so the gradient of logit c with
// respect to norm5's output A has a closed form and no backward pass runs:
//   A_k[p]  = fmaf(X_k[p], s_k, t_k)                  X = norm5's input (the last dense block's buffer), (s, t) = bn_eval_affine
//   dz_c / dA_k[p] = W[c,k] / n * [A_k[p] > 0]        n = h * w; strict >, as torch's threshold_backward
//   alpha[c,k] = W[c,k] m_k / n^2                     m_k = #{p : A_k[p] > 0}
//   cam_c[p]   = max(0, sum_k alpha[c,k] A_k[p])      the classifier bias does not enter
//   up_c       = F.interpolate(cam_c, (S, S), mode='bilinear', align_corners=False)
// A is computed with the fmaf and the affine of the eval-mode apply kernels (bn_relu.cu, bn_cl.cu), so A > 0 holds at exactly the
// pixels where the logits' relu(norm5) is non-zero.
//
// Three launches, every reduction in a fixed order and no atomics (bit-reproducible; an image's maps do not depend on its batch-mates):
//   grad_cam_count     grid (C / 8, B): one warp per (image, channel) counts m_k into the caller's int32 workspace
//   grad_cam_map       grid (n / 32, K / 8, B): 32 pixels x 8 classes per CTA; its 8 warps sum interleaved eighths of the channels,
//                      then one thread per (class, pixel) adds the 8 partial sums in slice order
//   grad_cam_upsample  grid (S / 8, K, B): 8 output rows of one map per CTA, coalesced stores (only when `up` is asked for)
#include "common.cuh"

namespace aaconv {
namespace {

typedef __nv_bfloat16 bf16;

constexpr int kThreads = 256;
constexpr int kMaxC = 4096;          // the map kernel keeps norm5's affine, (s, t) per channel, in 32 KB of shared memory
constexpr int kMaxHW = 4096;         // 64 x 64 (a 2048-px input): n^2 <= 2^24 is exact in fp32, and m_k fits any int
constexpr int kMaxK = 64;
constexpr int kMaxS = 4096;
constexpr int kTile = 32;                      // pixels of a map CTA (one per lane)
constexpr int kSlices = kThreads / kTile;      // channel slices of a map CTA (one per warp)
constexpr int kGroup = 8;                      // classes of a map CTA
constexpr int kRows = 8;                       // output rows of an upsample CTA

__device__ __forceinline__ float ld(const float* p) { return __ldg(p); }
__device__ __forceinline__ float ld(const bf16* p) { return __bfloat162float(*p); }

template <class T>
__global__ void __launch_bounds__(kThreads) grad_cam_count_kernel(const T* __restrict__ x, long long xbs, int C, int n,
                                                                  const float* __restrict__ weight, const float* __restrict__ bias,
                                                                  const float* __restrict__ running_mean,
                                                                  const float* __restrict__ running_var, float eps, int* __restrict__ m) {
  const int lane = threadIdx.x & 31, k = blockIdx.x * (kThreads / 32) + (threadIdx.x >> 5), b = blockIdx.y;
  if (k >= C) return;
  const float2 a = bn_eval_affine(weight, bias, running_mean, running_var, eps, k);
  const T* px = x + (size_t)b * xbs + (size_t)k * n;
  int cnt = 0;
  for (int p = lane; p < n; p += 32) cnt += fmaf(ld(px + p), a.x, a.y) > 0.f;
  cnt = __reduce_add_sync(0xffffffffu, cnt);
  if (lane == 0) m[(size_t)b * C + k] = cnt;
}

template <class T>
__global__ void __launch_bounds__(kThreads) grad_cam_map_kernel(const T* __restrict__ x, long long xbs, int C, int n,
                                                                const float* __restrict__ weight, const float* __restrict__ bias,
                                                                const float* __restrict__ running_mean,
                                                                const float* __restrict__ running_var, float eps,
                                                                const float* __restrict__ cls_w, int K, const int* __restrict__ m,
                                                                float* __restrict__ cam) {
  extern __shared__ float2 affine[];                       // (C)
  __shared__ float part[kSlices][kGroup][kTile];
  const int b = blockIdx.z, c0 = blockIdx.y * kGroup, p0 = blockIdx.x * kTile;
  const int nc = min(kGroup, K - c0);
  for (int k = threadIdx.x; k < C; k += kThreads) affine[k] = bn_eval_affine(weight, bias, running_mean, running_var, eps, k);
  __syncthreads();

  const int lane = threadIdx.x & 31, slice = threadIdx.x >> 5, p = p0 + lane;
  float acc[kGroup];
#pragma unroll
  for (int c = 0; c < kGroup; ++c) acc[c] = 0.f;
  if (p < n) {
    const T* px = x + (size_t)b * xbs + p;
    const int* mb = m + (size_t)b * C;
    const float* wc = cls_w + (size_t)c0 * C;
    for (int k = slice; k < C; k += kSlices) {
      const float2 a = affine[k];
      const float v = fmaf(ld(px + (size_t)k * n), a.x, a.y);
      const float mk = (float)__ldg(mb + k);
#pragma unroll
      for (int c = 0; c < kGroup; ++c)
        if (c < nc) acc[c] = fmaf(__ldg(wc + (size_t)c * C + k) * mk, v, acc[c]);
    }
  }
#pragma unroll
  for (int c = 0; c < kGroup; ++c) part[slice][c][lane] = acc[c];
  __syncthreads();

  const int c = threadIdx.x / kTile, q = threadIdx.x % kTile;     // kThreads == kGroup * kTile: one (class, pixel) per thread
  if (c < nc && p0 + q < n) {
    float s = 0.f;
#pragma unroll
    for (int j = 0; j < kSlices; ++j) s += part[j][c][q];
    cam[((size_t)b * K + c0 + c) * n + p0 + q] = fmaxf(s / ((float)n * (float)n), 0.f);
  }
}

// torch's upsample_bilinear2d (align_corners=False, no scale factor): source index scale * (dst + 0.5) - 0.5 clamped at 0,
// scale = (float)in / out
__global__ void __launch_bounds__(kThreads) grad_cam_upsample_kernel(const float* __restrict__ cam, int h, int w, int S, float scale_h,
                                                                     float scale_w, float* __restrict__ up) {
  const int b = blockIdx.z, c = blockIdx.y, K = gridDim.y, y0 = blockIdx.x * kRows;
  const int rows = min(kRows, S - y0);
  const float* src = cam + ((size_t)b * K + c) * h * w;
  float* dst = up + ((size_t)b * K + c) * S * S;
  for (int i = threadIdx.x; i < rows * S; i += kThreads) {
    const int oy = y0 + i / S, ox = i % S;
    const float sy = fmaxf(scale_h * (oy + 0.5f) - 0.5f, 0.f), sx = fmaxf(scale_w * (ox + 0.5f) - 0.5f, 0.f);
    const int iy = (int)sy, ix = (int)sx;
    const int dy = iy < h - 1 ? w : 0, dx = ix < w - 1 ? 1 : 0;
    const float ly1 = sy - iy, ly0 = 1.f - ly1, lx1 = sx - ix, lx0 = 1.f - lx1;
    const float* s0 = src + (size_t)iy * w + ix;
    dst[(size_t)oy * S + ox] = ly0 * (lx0 * __ldg(s0) + lx1 * __ldg(s0 + dx)) + ly1 * (lx0 * __ldg(s0 + dy) + lx1 * __ldg(s0 + dy + dx));
  }
}

template <class T>
int grad_cam_t(const T* x, int B, int C, int h, int w, long long xbs, const float* weight, const float* bias, const float* rm,
               const float* rv, float eps, const float* cls_w, int K, float* cam, float* up, int S, int* m, cudaStream_t st) {
  const int n = h * w;
  grad_cam_count_kernel<T><<<dim3(cdiv(C, kThreads / 32), B), kThreads, 0, AACONV_ST(st)>>>(x, xbs, C, n, weight, bias, rm, rv, eps, m);
  AACONV_LAUNCH_OK("grad_cam_count");
  grad_cam_map_kernel<T><<<dim3(cdiv(n, kTile), cdiv(K, kGroup), B), kThreads, (size_t)C * sizeof(float2), AACONV_ST(st)>>>(
      x, xbs, C, n, weight, bias, rm, rv, eps, cls_w, K, m, cam);
  AACONV_LAUNCH_OK("grad_cam_map");
  if (up) {
    grad_cam_upsample_kernel<<<dim3(cdiv(S, kRows), K, B), kThreads, 0, AACONV_ST(st)>>>(cam, h, w, S, (float)h / S, (float)w / S, up);
    AACONV_LAUNCH_OK("grad_cam_upsample");
  }
  return 0;
}

bool misaligned(const void* p, size_t bytes) { return reinterpret_cast<uintptr_t>(p) % bytes != 0; }

}  // namespace

extern "C" {

int aaconv_grad_cam(const void* x, int dtype, int B, int C, int h, int w, int64_t x_batch_stride, const float* weight,
                    const float* bias, const float* running_mean, const float* running_var, float eps, const float* cls_weight, int K,
                    float* cam, float* up, int S, int32_t* workspace, void* stream) {
  if (!x || !weight || !bias || !running_mean || !running_var || !cls_weight || !cam || !workspace)
    return fail(AACONV_E_ARG, "grad_cam: null pointer (only up may be NULL)");
  if (dtype != AACONV_FP32 && dtype != AACONV_BF16) return fail(AACONV_E_ARG, "grad_cam: dtype %d is neither fp32 nor bf16", dtype);
  if (B < 1 || B > 65535) return fail(AACONV_E_ARG, "grad_cam: B %d outside [1, 65535]", B);
  if (C < 1 || C > kMaxC) return fail(AACONV_E_ARG, "grad_cam: C %d outside [1, %d]", C, kMaxC);
  if (h < 1 || w < 1 || (long long)h * w > kMaxHW)
    return fail(AACONV_E_ARG, "grad_cam: map %d x %d, h and w must be >= 1 and h*w at most %d (64 x 64)", h, w, kMaxHW);
  if (K < 1 || K > kMaxK) return fail(AACONV_E_ARG, "grad_cam: K %d outside [1, %d] classes", K, kMaxK);
  if (up && (S < 1 || S > kMaxS)) return fail(AACONV_E_ARG, "grad_cam: S %d outside [1, %d]", S, kMaxS);
  if (x_batch_stride < (int64_t)C * h * w)
    return fail(AACONV_E_ARG, "grad_cam: x_batch_stride %lld below C*h*w = %lld", (long long)x_batch_stride, (long long)C * h * w);
  const size_t esz = dtype == AACONV_BF16 ? 2 : 4;
  if (misaligned(x, esz)) return fail(AACONV_E_ARG, "grad_cam: x must be aligned to its %zu-byte element", esz);
  if (misaligned(weight, 4) || misaligned(bias, 4) || misaligned(running_mean, 4) || misaligned(running_var, 4) ||
      misaligned(cls_weight, 4) || misaligned(cam, 4) || (up && misaligned(up, 4)) || misaligned(workspace, 4))
    return fail(AACONV_E_ARG, "grad_cam: fp32 / int32 arrays must be aligned to 4 bytes");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return dtype == AACONV_BF16
             ? grad_cam_t(static_cast<const bf16*>(x), B, C, h, w, x_batch_stride, weight, bias, running_mean, running_var, eps, cls_weight, K,
                          cam, up, S, workspace, st)
             : grad_cam_t(static_cast<const float*>(x), B, C, h, w, x_batch_stride, weight, bias, running_mean, running_var, eps, cls_weight,
                          K, cam, up, S, workspace, st);
}

}  // extern "C"

}  // namespace aaconv
