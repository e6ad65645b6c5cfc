// Channels-last side of the dense-block BatchNorm2d (training) + ReLU kernels (SURVEY.md section 8 row f3).
//
// cuDNN's tensor-core convolutions are NHWC kernels: with NCHW activations it transposes every operand of every fprop / dgrad /
// wgrad itself (21 % of the aadensenet121 step in the round-2 profile), and leaving the conversion to torch (`.contiguous(
// channels_last)` + torch's NHWC BatchNorm) measured SLOWER (1074 vs 1376 images/s: generic strided copies at 14 us each, 22 us
// NHWC reductions).  Here the layout change is folded into passes that exist anyway:
//
//   norm1 -> relu1   x = channels [0, C) of the NCHW feature buffer (batch stride), y = NHWC:   stats (bn_relu.cu) -> finalize ->
//                    t_apply (64 channel x 64 pixel tiles through shared memory);  backward: dy NHWC, dx ADDED into the NCHW
//                    gradient of the buffer:  t_bwd_reduce -> finalize -> t_bwd_dx
//   norm2 -> relu2   x, y NHWC (the 128-channel bottleneck):  cl_stats -> finalize -> cl_apply;  cl_bwd_reduce -> finalize -> cl_bwd_dx
//   append           new features NHWC -> their channel slice of the NCHW buffer, and the slice of the buffer gradient -> NHWC
//   eval mode        t_apply / cl_apply alone (EVAL instantiations), their per-channel affine maps from the running statistics
//                    (aaconv_bn_relu_eval; inference only, no backward)
//   Transition       densenet121's BatchNorm -> ReLU -> 1x1 conv -> AvgPool2d(2), the pool moved ahead of the conv: NCHW block buffer
//                    -> pooled NHWC operand (pool_apply, training or EVAL); backward pool_bwd_reduce -> finalize -> pool_bwd_dx
//                    (aaconv_bn_relu_pool_*)
//
// All reductions run in a fixed order (bit-reproducible).  Reference: torchvision densenet.py:31-95,120-124 under
// models/attn_aug_conv.py:479-482.
#include <algorithm>
#include <cuda_bf16.h>
#include "common.cuh"

namespace aaconv {

typedef __nv_bfloat16 bf16;

namespace {

__device__ __forceinline__ float4 ldv(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ldv(const bf16* p) {
  const uint2 u = *reinterpret_cast<const uint2*>(p);
  const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
  const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
  return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ void stv(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void stv(bf16* p, float4 v) {
  const __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
  uint2 u;
  u.x = *reinterpret_cast<const uint32_t*>(&a);
  u.y = *reinterpret_cast<const uint32_t*>(&b);
  *reinterpret_cast<uint2*>(p) = u;
}
__device__ __forceinline__ float ld1v(const float* p) { return *p; }
__device__ __forceinline__ float ld1v(const bf16* p) { return __bfloat162float(*p); }
__device__ __forceinline__ void st1v(float* p, float v) { *p = v; }
__device__ __forceinline__ void st1v(bf16* p, float v) { *p = __float2bfloat16(v); }

// ------------------------------------------------------------------------------------------------
// finalize kernels: one thread per channel, partials at partial[c * sc + g * sg]
// ------------------------------------------------------------------------------------------------
// One warp per channel (8 channels per CTA): lanes stride over the G partials, then a shuffle tree in a fixed order.  (A serial
// loop per channel thread measured 35 us per call at G = 600: two divides per dependent step.)
struct Chan { float n, mean, m2; };
__device__ __forceinline__ Chan chan_merge(Chan a, Chan b) {          // a (+) b; either side may be empty
  if (b.n == 0.f) return a;
  if (a.n == 0.f) return b;
  const float tot = a.n + b.n, d = b.mean - a.mean, bf = __fdividef(b.n, tot);   // IEEE division: ~100 cycles per dependent step
  Chan r;
  r.n = tot;
  r.mean = a.mean + d * bf;
  r.m2 = a.m2 + b.m2 + d * d * (a.n * bf);
  return r;
}
// Chan merge of G (mean, M2) partials (n_each elements each, n_last for the last one) -> saved (mean, rstd), running statistics
__global__ void __launch_bounds__(256) bn_fin_fwd_kernel(const float2* __restrict__ partial, int C, int G, long long sc, long long sg,
                                                         float n_each, float n_last, float eps, float momentum, float2* __restrict__ saved,
                                                         float* __restrict__ running_mean, float* __restrict__ running_var) {
  const int c = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (c >= C) return;
  Chan acc = {0.f, 0.f, 0.f};
  // the partials of a lane are fetched in batches of 8 independent loads (ncu: with load -> merge -> load in sequence this kernel took
  // 18 us at G = 582, every iteration a dependent L2 round trip)
  for (int g0 = lane; g0 < G; g0 += 32 * 8) {
    float2 p[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) { const int g = g0 + 32 * k; p[k] = g < G ? partial[c * sc + g * sg] : make_float2(0.f, 0.f); }
#pragma unroll
    for (int k = 0; k < 8; ++k) {
      const int g = g0 + 32 * k;
      if (g < G) { const Chan b = {g == G - 1 ? n_last : n_each, p[k].x, p[k].y}; acc = chan_merge(acc, b); }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    Chan b;
    b.n = __shfl_down_sync(0xffffffffu, acc.n, o);
    b.mean = __shfl_down_sync(0xffffffffu, acc.mean, o);
    b.m2 = __shfl_down_sync(0xffffffffu, acc.m2, o);
    if (lane < o) acc = chan_merge(acc, b);
  }
  if (lane == 0) {
    const float var = acc.m2 / acc.n;
    saved[c] = make_float2(acc.mean, rsqrtf(var + eps));
    if (running_mean) {
      running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * acc.mean;
      running_var[c] = (1.f - momentum) * running_var[c] + momentum * var * (acc.n / fmaxf(acc.n - 1.f, 1.f));
    }
  }
}
// plain sums of G (sum g, sum g x^) partials -> sums[c], dweight, dbias
__global__ void __launch_bounds__(256) bn_fin_bwd_kernel(const float2* __restrict__ partial, int C, int G, long long sc, long long sg,
                                                         float2* __restrict__ sums, float* __restrict__ dweight, float* __restrict__ dbias) {
  const int c = blockIdx.x * 8 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (c >= C) return;
  float s1 = 0.f, s2 = 0.f;
  for (int g0 = lane; g0 < G; g0 += 32 * 8) {          // batches of 8 independent loads, summed in index order
    float2 p[8];
#pragma unroll
    for (int k = 0; k < 8; ++k) { const int g = g0 + 32 * k; p[k] = g < G ? partial[c * sc + g * sg] : make_float2(0.f, 0.f); }
#pragma unroll
    for (int k = 0; k < 8; ++k) { s1 += p[k].x; s2 += p[k].y; }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s1 += __shfl_down_sync(0xffffffffu, s1, o);
    s2 += __shfl_down_sync(0xffffffffu, s2, o);
  }
  if (lane == 0) {
    sums[c] = make_float2(s1, s2);
    if (dweight) dweight[c] = s2;
    if (dbias) dbias[c] = s1;
  }
}

// ------------------------------------------------------------------------------------------------
// NHWC -> NHWC (x, y: (rows = B*HW, C) dense, C % 4 == 0)
// thread layout: TPR = threads per row (power of two <= 256 covering C / 4 quads when possible), 256 / TPR rows side by side
// ------------------------------------------------------------------------------------------------
// CTAs the NCHW-side reduction aims for: each loops over its pixel chunks serially with two barriers per chunk, so the latency is
// hidden by CTAs, not inside one (300 CTAs: 19 us per call on average; see profiles/r02_b_scaling.md)
constexpr int T_RED_CTAS = 2368;
constexpr int CL_ROWS = 256;   // most rows per CTA of the reduction kernels (the host picks 32..256 so that every SM gets a few CTAs)
// most channels of an NHWC input: cl_stats keeps a thread's segment means in registers, 4 quads of at most 256 threads per row
constexpr int CL_MAX_C = 4 * 4 * 256;

// red[slot][c] -> fixed-order sum over the 256 / TPR row slots for channel c (c < C), result broadcast through red[0][c]
__device__ __forceinline__ void reduce_slots(float* red, int C, int nslot) {
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += 256) {
    float s = 0.f;
    for (int k = 0; k < nslot; ++k) s += red[k * C + c];
    red[c] = s;                         // slot 0 is only read by this thread for this c
  }
  __syncthreads();
}

template <class T>
__global__ void __launch_bounds__(256) cl_stats_kernel(const T* __restrict__ x, long long rows, int rpc, int C, int tprl, float2* __restrict__ partial) {
  extern __shared__ __align__(16) float red[];           // [256 / TPR][C]
  const int TPR = 1 << tprl, nslot = 256 >> tprl, q0 = threadIdx.x & (TPR - 1), slot = threadIdx.x >> tprl, Q = C >> 2;
  const long long r0 = (long long)blockIdx.x * rpc;
  const int nr = (int)min((long long)rpc, rows - r0);
  const T* px = x + r0 * C;
  // pass 1: per-channel sums of the segment
  for (int q = q0; q < Q; q += TPR) {
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int r = slot; r < nr; r += nslot) { const float4 v = ldv(px + (size_t)r * C + 4 * q); s.x += v.x; s.y += v.y; s.z += v.z; s.w += v.w; }
    *reinterpret_cast<float4*>(red + slot * C + 4 * q) = s;
  }
  reduce_slots(red, C, nslot);
  float4 mean[4];                                         // up to 4 quads per thread (C <= 4 * 4 * TPR <= CL_MAX_C)
  const float inv = 1.f / (float)nr;
  int k = 0;
  for (int q = q0; q < Q; q += TPR, ++k) {
    const float4 s = *reinterpret_cast<const float4*>(red + 4 * q);
    mean[k & 3] = make_float4(s.x * inv, s.y * inv, s.z * inv, s.w * inv);
  }
  __syncthreads();
  // pass 2: M2 around the segment mean
  k = 0;
  for (int q = q0; q < Q; q += TPR, ++k) {
    const float4 m = mean[k & 3];
    float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
    for (int r = slot; r < nr; r += nslot) {
      const float4 v = ldv(px + (size_t)r * C + 4 * q);
      const float a = v.x - m.x, b = v.y - m.y, c = v.z - m.z, d = v.w - m.w;
      s.x += a * a; s.y += b * b; s.z += c * c; s.w += d * d;
    }
    *reinterpret_cast<float4*>(red + slot * C + 4 * q) = s;
  }
  reduce_slots(red, C, nslot);
  k = 0;
  float2* out = partial + (size_t)blockIdx.x * C;          // [segment][channel]
  if (slot == 0)
    for (int q = q0; q < Q; q += TPR, ++k) {
      const float4 m = mean[k & 3];
      const float4 s = *reinterpret_cast<const float4*>(red + 4 * q);
      out[4 * q] = make_float2(m.x, s.x); out[4 * q + 1] = make_float2(m.y, s.y);
      out[4 * q + 2] = make_float2(m.z, s.z); out[4 * q + 3] = make_float2(m.w, s.w);
    }
}

// EVAL: BatchNorm2d in eval mode, the channel's affine map from the running statistics (`saved` unused); else from saved (mean, rstd)
template <class T, bool EVAL>
__global__ void __launch_bounds__(256) cl_apply_kernel(const T* __restrict__ x, long long nquads, int C, const float2* __restrict__ saved,
                                                       const float* __restrict__ weight, const float* __restrict__ bias, T* __restrict__ y,
                                                       const float* __restrict__ running_mean, const float* __restrict__ running_var,
                                                       float eps) {
  // the quad's channels repeat with period C / 4: a grid-stride loop with a stride that is a multiple of C / 4 keeps them fixed
  const int Q = C >> 2;
  const long long stride = ((long long)gridDim.x * 256 / Q) * Q;
  long long i = (long long)blockIdx.x * 256 + threadIdx.x;
  if (i >= stride) return;
  const int c = (int)(i % Q) * 4;
  float sc[4], sh[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    if constexpr (EVAL) {
      const float2 a = bn_eval_affine(weight, bias, running_mean, running_var, eps, c + u);
      sc[u] = a.x; sh[u] = a.y;
    } else {
      const float2 st = saved[c + u]; sc[u] = weight[c + u] * st.y; sh[u] = bias[c + u] - st.x * sc[u];
    }
  }
  for (; i < nquads; i += stride) {
    const float4 v = ldv(x + 4 * i);
    stv(y + 4 * i, make_float4(fmaxf(fmaf(v.x, sc[0], sh[0]), 0.f), fmaxf(fmaf(v.y, sc[1], sh[1]), 0.f), fmaxf(fmaf(v.z, sc[2], sh[2]), 0.f),
                               fmaxf(fmaf(v.w, sc[3], sh[3]), 0.f)));
  }
}

template <class T>
__global__ void __launch_bounds__(256) cl_bwd_reduce_kernel(const T* __restrict__ x, const T* __restrict__ dy, long long rows, int rpc, int C, int tprl,
                                                            const float2* __restrict__ saved, const float* __restrict__ weight,
                                                            const float* __restrict__ bias, float2* __restrict__ partial) {
  extern __shared__ __align__(16) float red[];           // [2][256 / TPR][C]
  const int TPR = 1 << tprl, nslot = 256 >> tprl, q0 = threadIdx.x & (TPR - 1), slot = threadIdx.x >> tprl, Q = C >> 2;
  const long long r0 = (long long)blockIdx.x * rpc;
  const int nr = (int)min((long long)rpc, rows - r0);
  const T* px = x + r0 * C;
  const T* pg = dy + r0 * C;
  float* red2 = red + nslot * C;
  for (int q = q0; q < Q; q += TPR) {
    float mu[4], rs[4], w[4], bb[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) { const float2 st = saved[4 * q + u]; mu[u] = st.x; rs[u] = st.y; w[u] = weight[4 * q + u]; bb[u] = bias[4 * q + u]; }
    float s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
    for (int r = slot; r < nr; r += nslot) {
      const float4 xv = ldv(px + (size_t)r * C + 4 * q), gv = ldv(pg + (size_t)r * C + 4 * q);
      const float xs[4] = {xv.x, xv.y, xv.z, xv.w}, gs[4] = {gv.x, gv.y, gv.z, gv.w};
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float xh = (xs[u] - mu[u]) * rs[u];
        const float g = fmaf(w[u], xh, bb[u]) > 0.f ? gs[u] : 0.f;
        s1[u] += g;
        s2[u] = fmaf(g, xh, s2[u]);
      }
    }
    *reinterpret_cast<float4*>(red + slot * C + 4 * q) = make_float4(s1[0], s1[1], s1[2], s1[3]);
    *reinterpret_cast<float4*>(red2 + slot * C + 4 * q) = make_float4(s2[0], s2[1], s2[2], s2[3]);
  }
  __syncthreads();
  float2* out = partial + (size_t)blockIdx.x * C;
  for (int c = threadIdx.x; c < C; c += 256) {
    float a = 0.f, b = 0.f;
    for (int k = 0; k < nslot; ++k) { a += red[k * C + c]; b += red2[k * C + c]; }
    out[c] = make_float2(a, b);
  }
}

template <class T>
__global__ void __launch_bounds__(256) cl_bwd_dx_kernel(const T* __restrict__ x, const T* __restrict__ dy, long long nquads, int C,
                                                        const float2* __restrict__ saved, const float* __restrict__ weight,
                                                        const float* __restrict__ bias, const float2* __restrict__ sums, float inv_n,
                                                        T* __restrict__ dx) {
  const int Q = C >> 2;
  const long long stride = ((long long)gridDim.x * 256 / Q) * Q;
  long long i = (long long)blockIdx.x * 256 + threadIdx.x;
  if (i >= stride) return;
  const int c = (int)(i % Q) * 4;
  float mu[4], rs[4], w[4], bb[4], m1[4], m2[4];
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const float2 st = saved[c + u], sm = sums[c + u];
    mu[u] = st.x; rs[u] = st.y; w[u] = weight[c + u]; bb[u] = bias[c + u]; m1[u] = sm.x * inv_n; m2[u] = sm.y * inv_n;
  }
  for (; i < nquads; i += stride) {
    const float4 xv = ldv(x + 4 * i), gv = ldv(dy + 4 * i);
    const float xs[4] = {xv.x, xv.y, xv.z, xv.w}, gs[4] = {gv.x, gv.y, gv.z, gv.w};
    float o[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const float xh = (xs[u] - mu[u]) * rs[u];
      const float g = fmaf(w[u], xh, bb[u]) > 0.f ? gs[u] : 0.f;
      o[u] = w[u] * rs[u] * (g - m1[u] - xh * m2[u]);
    }
    stv(dx + 4 * i, make_float4(o[0], o[1], o[2], o[3]));
  }
}

// ------------------------------------------------------------------------------------------------
// NCHW (batch stride) <-> NHWC tile kernels: 64 channels x 64 pixels through shared memory.
// NCHW side: a warp covers 2 channels x 16 pixel quads (coalesced along pixels); NHWC side: 2 pixels x 16 channel quads.
// HW % 4 == 0 and C % 4 == 0; the last channel tile may be partial.
// ------------------------------------------------------------------------------------------------
template <class T, class F>
__device__ __forceinline__ void tile_load_nchw(const T* __restrict__ src /* plane (b, c0) */, int C, int c0, int HW, int p0,
                                               float (*t)[65], F f) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int px = p0 + (lane & 15) * 4, pl = (lane & 15) * 4;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int cl = warp * 8 + i * 2 + (lane >> 4), c = c0 + cl;
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c < C && px < HW) v = f(c, ldv(src + (size_t)cl * HW + px));
    t[pl][cl] = v.x; t[pl + 1][cl] = v.y; t[pl + 2][cl] = v.z; t[pl + 3][cl] = v.w;
  }
}

// The per-channel affine maps (ssc, ssh) of the CTA's 64 channels [c0, c0 + 64), y = relu(x ssc + ssh).  The G group statistics of
// a channel (NCHW layout of aaconv_bn_stats_nchw) are merged here (the separate finalize launch cost 5 us per layer); the CTAs of
// pixel tile 0 / sample 0 (blockIdx.x == 0, blockIdx.z == 0) also write saved (mean, rstd) and the running statistics.
// EVAL: BatchNorm2d in eval mode instead -- the affine maps come from the running statistics, which are only read (partial, G,
// n_*, momentum and saved unused).  The caller synchronises before reading ssc / ssh.
template <bool EVAL>
__device__ __forceinline__ void tile_affine(int c0, int C, const float2* __restrict__ partial, int G, float n_each, float n_last, float eps,
                                            float momentum, float2* __restrict__ saved, float* __restrict__ running_mean,
                                            float* __restrict__ running_var, const float* __restrict__ weight,
                                            const float* __restrict__ bias, float* ssc, float* ssh) {
  const int b = blockIdx.z;
  if constexpr (EVAL) {
    if (threadIdx.x < 64 && c0 + (int)threadIdx.x < C) {
      const float2 a = bn_eval_affine(weight, bias, running_mean, running_var, eps, c0 + threadIdx.x);
      ssc[threadIdx.x] = a.x;
      ssh[threadIdx.x] = a.y;
    }
  } else {   // four threads per channel, then two shuffle steps (fixed order); measured: with 64 threads merging serially through IEEE
      // divisions half of the kernel's samples sat in the barrier below
    const int ch = threadIdx.x >> 2, sub = threadIdx.x & 3, c = min(c0 + ch, C - 1);
    Chan acc = {0.f, 0.f, 0.f};
    for (int g = sub; g < G; g += 4) {
      const float2 p = partial[(size_t)c * G + g];
      const Chan q = {g == G - 1 ? n_last : n_each, p.x, p.y};
      acc = chan_merge(acc, q);
    }
#pragma unroll
    for (int o = 1; o <= 2; o <<= 1) {
      Chan q;
      q.n = __shfl_down_sync(0xffffffffu, acc.n, o);
      q.mean = __shfl_down_sync(0xffffffffu, acc.mean, o);
      q.m2 = __shfl_down_sync(0xffffffffu, acc.m2, o);
      if ((sub & (2 * o - 1)) == 0) acc = chan_merge(acc, q);
    }
    if (sub == 0 && c0 + ch < C) {
    const float var = __fdividef(acc.m2, acc.n), rstd = rsqrtf(var + eps);
    const float sc = weight[c] * rstd;
    ssc[ch] = sc;
    ssh[ch] = bias[c] - acc.mean * sc;
    if (blockIdx.x == 0 && b == 0) {
      saved[c] = make_float2(acc.mean, rstd);
      if (running_mean) {
        running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * acc.mean;
        running_var[c] = (1.f - momentum) * running_var[c] + momentum * var * (acc.n / fmaxf(acc.n - 1.f, 1.f));
      }
    }
    }
  }
}

// y (NHWC) = relu(bn(x (NCHW, batch stride))), the affine maps from tile_affine.
template <class T, bool EVAL>
__global__ void __launch_bounds__(256) t_apply_kernel(const T* __restrict__ x, long long xbs, int C, int HW, const float2* __restrict__ partial,
                                                      int G, float n_each, float n_last, float eps, float momentum,
                                                      float2* __restrict__ saved, float* __restrict__ running_mean,
                                                      float* __restrict__ running_var, const float* __restrict__ weight,
                                                      const float* __restrict__ bias, T* __restrict__ y) {
  __shared__ float t[64][65];                                   // [pixel][channel]
  __shared__ float ssc[64], ssh[64];
  const int b = blockIdx.z, c0 = blockIdx.y * 64, p0 = blockIdx.x * 64;
  tile_affine<EVAL>(c0, C, partial, G, n_each, n_last, eps, momentum, saved, running_mean, running_var, weight, bias, ssc, ssh);
  __syncthreads();
  tile_load_nchw(x + (size_t)b * xbs + (size_t)c0 * HW, C, c0, HW, p0, t, [&](int c, float4 v) {
    const float sc = ssc[c - c0], sh = ssh[c - c0];
    return make_float4(fmaxf(fmaf(v.x, sc, sh), 0.f), fmaxf(fmaf(v.y, sc, sh), 0.f), fmaxf(fmaf(v.z, sc, sh), 0.f), fmaxf(fmaf(v.w, sc, sh), 0.f));
  });
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, cl = (lane & 15) * 4;
  T* dst = y + (size_t)b * HW * C;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int pl = warp * 8 + i * 2 + (lane >> 4), px = p0 + pl;
    if (px < HW && c0 + cl < C) stv(dst + (size_t)px * C + c0 + cl, make_float4(t[pl][cl], t[pl][cl + 1], t[pl][cl + 2], t[pl][cl + 3]));
  }
}

// partial[(c) * (B * nseg) + b * nseg + seg] = (sum g, sum g x^) over the segment's pixels; dy NHWC, x NCHW
template <class T>
__global__ void __launch_bounds__(256) t_bwd_reduce_kernel(const T* __restrict__ x, long long xbs, int C, int HW, const T* __restrict__ dy,
                                                           const float2* __restrict__ saved, const float* __restrict__ weight,
                                                           const float* __restrict__ bias, int chunks_per_seg, float2* __restrict__ partial) {
  __shared__ float t[64][65];                                   // x^ tile, [pixel][channel]
  __shared__ float red[2][16][64];
  const int seg = blockIdx.x, nseg = gridDim.x, c0 = blockIdx.y * 64, b = blockIdx.z, B = gridDim.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, cl = (lane & 15) * 4;
  float w[4], bb[4], s1[4] = {0.f, 0.f, 0.f, 0.f}, s2[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
  for (int u = 0; u < 4; ++u) { const int c = min(c0 + cl + u, C - 1); w[u] = weight[c]; bb[u] = bias[c]; }
  const int nchunks = (HW + 63) / 64;
  for (int ch = seg * chunks_per_seg; ch < min(nchunks, (seg + 1) * chunks_per_seg); ++ch) {
    const int p0 = ch * 64;
    // dy first: its latency runs under the x tile's (ncu: 61 % of the samples sat on the long scoreboard with the loads in sequence)
    float4 gq[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int px = p0 + warp * 8 + i * 2 + (lane >> 4);
      gq[i] = (px < HW && c0 + cl < C) ? ldv(dy + ((size_t)b * HW + px) * C + c0 + cl) : make_float4(0.f, 0.f, 0.f, 0.f);
    }
    __syncthreads();                                            // the previous chunk's tile has been consumed
    tile_load_nchw(x + (size_t)b * xbs + (size_t)c0 * HW, C, c0, HW, p0, t, [&](int c, float4 v) {
      const float2 st = saved[c];
      return make_float4((v.x - st.x) * st.y, (v.y - st.x) * st.y, (v.z - st.x) * st.y, (v.w - st.x) * st.y);
    });
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int pl = warp * 8 + i * 2 + (lane >> 4), px = p0 + pl;
      if (px < HW && c0 + cl < C) {
        const float4 gv = gq[i];
        const float gs[4] = {gv.x, gv.y, gv.z, gv.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float xh = t[pl][cl + u];
          const float g = fmaf(w[u], xh, bb[u]) > 0.f ? gs[u] : 0.f;
          s1[u] += g;
          s2[u] = fmaf(g, xh, s2[u]);
        }
      }
    }
  }
  // the 16 threads that share a channel quad (8 warps x 2 half-warps), summed in a fixed order
  const int slot = warp * 2 + (lane >> 4);
#pragma unroll
  for (int u = 0; u < 4; ++u) { red[0][slot][cl + u] = s1[u]; red[1][slot][cl + u] = s2[u]; }
  __syncthreads();
  if (threadIdx.x < 64 && c0 + threadIdx.x < C) {
    float a = 0.f, d = 0.f;
#pragma unroll
    for (int k = 0; k < 16; ++k) { a += red[0][k][threadIdx.x]; d += red[1][k][threadIdx.x]; }
    partial[(size_t)(c0 + threadIdx.x) * ((size_t)B * nseg) + (size_t)b * nseg + seg] = make_float2(a, d);
  }
}

// gacc (NCHW, batch stride gbs) (+)= dx; dy NHWC, x NCHW
template <class T, bool ACC>
__global__ void __launch_bounds__(256) t_bwd_dx_kernel(const T* __restrict__ x, long long xbs, int C, int HW, const T* __restrict__ dy,
                                                       const float2* __restrict__ saved, const float* __restrict__ weight,
                                                       const float* __restrict__ bias, const float2* __restrict__ sums, float inv_n,
                                                       T* __restrict__ gacc, long long gbs) {
  __shared__ float t[64][65];
  const int b = blockIdx.z, c0 = blockIdx.y * 64, p0 = blockIdx.x * 64;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // every global read of the CTA is issued before the first barrier: dy (NHWC mapping), the accumulation target (NCHW mapping), x
  float4 gq[4], ga[4];
  T* const dstp = gacc + (size_t)b * gbs + (size_t)c0 * HW;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int px = p0 + warp * 8 + i * 2 + (lane >> 4), cq = (lane & 15) * 4;
    gq[i] = (px < HW && c0 + cq < C) ? ldv(dy + ((size_t)b * HW + px) * C + c0 + cq) : make_float4(0.f, 0.f, 0.f, 0.f);
    const int cl2 = warp * 8 + i * 2 + (lane >> 4), px2 = p0 + (lane & 15) * 4;
    ga[i] = (ACC && c0 + cl2 < C && px2 < HW) ? ldv(static_cast<const T*>(dstp + (size_t)cl2 * HW + px2)) : make_float4(0.f, 0.f, 0.f, 0.f);
  }
  tile_load_nchw(x + (size_t)b * xbs + (size_t)c0 * HW, C, c0, HW, p0, t, [&](int c, float4 v) {
    const float2 st = saved[c];
    return make_float4((v.x - st.x) * st.y, (v.y - st.x) * st.y, (v.z - st.x) * st.y, (v.w - st.x) * st.y);
  });
  __syncthreads();
  {
    const int cl = (lane & 15) * 4;
    float w[4], bb[4], k[4], m1[4], m2[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int c = min(c0 + cl + u, C - 1);
      const float2 sm = sums[c];
      w[u] = weight[c]; bb[u] = bias[c]; k[u] = w[u] * saved[c].y; m1[u] = sm.x * inv_n; m2[u] = sm.y * inv_n;
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int pl = warp * 8 + i * 2 + (lane >> 4), px = p0 + pl;
      (void)px;
      const float4 gv = gq[i];
      const float gs[4] = {gv.x, gv.y, gv.z, gv.w};
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float xh = t[pl][cl + u];
        const float g = fmaf(w[u], xh, bb[u]) > 0.f ? gs[u] : 0.f;
        t[pl][cl + u] = k[u] * (g - m1[u] - xh * m2[u]);        // in place: this thread owns (pl, cl..cl+3) in this phase
      }
    }
  }
  __syncthreads();
  {
    const int px = p0 + (lane & 15) * 4, pl = (lane & 15) * 4;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int cl = warp * 8 + i * 2 + (lane >> 4), c = c0 + cl;
      if (c < C && px < HW) {
        float4 v = make_float4(t[pl][cl], t[pl + 1][cl], t[pl + 2][cl], t[pl + 3][cl]);
        if (ACC) { v.x += ga[i].x; v.y += ga[i].y; v.z += ga[i].z; v.w += ga[i].w; }
        stv(dstp + (size_t)cl * HW + px, v);
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// torchvision's Transition, BatchNorm2d -> ReLU -> Conv2d 1x1 -> AvgPool2d(2), with the pool moved ahead of the 1x1 convolution
// (the convolution is per pixel and linear, so the two commute): x NCHW (batch stride) -> P (B, H/2, W/2, C) NHWC dense, the 2x2
// window means of relu(bn(x)); the convolution then runs on a quarter of the pixels.  Floor mode: an odd last row / column is in
// no window, but it is part of the batch statistics, and backward gives it the mean terms of dx.
// A CTA covers 64 channels x 64 windows (flattened over the window grid); warp w owns channels c0 + 8w .. c0 + 8w + 7, lane l the
// windows l and l + 32 -- the four source pixels of a window are two pairs of neighbouring elements of two NCHW rows.
// ------------------------------------------------------------------------------------------------
// the 2 x 2 window (hq, wq) of a plane: v = rows 2 hq, 2 hq + 1 x columns 2 wq, 2 wq + 1; elements outside the plane read as 0
template <class T>
__device__ __forceinline__ void win_load(const T* __restrict__ plane, int H, int W, int hq, int wq, float v[4]) {
  const int h = 2 * hq, w = 2 * wq;
  const T* p = plane + (size_t)h * W + w;
  const bool r1 = h + 1 < H, c1 = w + 1 < W;
  v[0] = ld1v(p);
  v[1] = c1 ? ld1v(p + 1) : 0.f;
  v[2] = r1 ? ld1v(p + W) : 0.f;
  v[3] = r1 && c1 ? ld1v(p + W + 1) : 0.f;
}

// P = avgpool2(relu(bn(x))); the affine maps (and in training saved / running statistics) from tile_affine
template <class T, bool EVAL>
__global__ void __launch_bounds__(256) pool_apply_kernel(const T* __restrict__ x, long long xbs, int C, int H, int W,
                                                         const float2* __restrict__ partial, int G, float n_each, float n_last, float eps,
                                                         float momentum, float2* __restrict__ saved, float* __restrict__ running_mean,
                                                         float* __restrict__ running_var, const float* __restrict__ weight,
                                                         const float* __restrict__ bias, T* __restrict__ y) {
  __shared__ float t[64][65];                                   // [window][channel]
  __shared__ float ssc[64], ssh[64];
  const int b = blockIdx.z, c0 = blockIdx.y * 64, p0 = blockIdx.x * 64;
  const int Wp = W >> 1, P = (H >> 1) * Wp;
  tile_affine<EVAL>(c0, C, partial, G, n_each, n_last, eps, momentum, saved, running_mean, running_var, weight, bias, ssc, ssh);
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int cl = warp * 8 + i, c = c0 + cl;
    const T* plane = x + (size_t)b * xbs + (size_t)min(c, C - 1) * H * W;
#pragma unroll
    for (int k = 0; k < 2; ++k) {
      const int pl = lane + 32 * k, p = p0 + pl;
      float s = 0.f;
      if (c < C && p < P) {
        const int hq = p / Wp;
        float v[4];
        win_load(plane, H, W, hq, p - hq * Wp, v);
        const float sc = ssc[cl], sh = ssh[cl];
        s = 0.25f * ((fmaxf(fmaf(v[0], sc, sh), 0.f) + fmaxf(fmaf(v[1], sc, sh), 0.f)) +
                     (fmaxf(fmaf(v[2], sc, sh), 0.f) + fmaxf(fmaf(v[3], sc, sh), 0.f)));
      }
      t[pl][cl] = s;
    }
  }
  __syncthreads();
  const int cq = (lane & 15) * 4;
  T* dst = y + (size_t)b * P * C;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int pl = warp * 8 + i * 2 + (lane >> 4), p = p0 + pl;
    if (p < P && c0 + cq < C) stv(dst + (size_t)p * C + c0 + cq, make_float4(t[pl][cq], t[pl][cq + 1], t[pl][cq + 2], t[pl][cq + 3]));
  }
}

// the dP tile of windows [p0, p0 + 64) of the window grid (Hq, Wq) -> t[window][channel]; windows outside the pooled map
// (Hp, Wp) -- the odd last row / column -- get 0
template <class T>
__device__ __forceinline__ void dp_tile(const T* __restrict__ dP, int b, int C, int c0, int Hp, int Wp, int Wq, int nwin, int p0,
                                        float (*t)[65]) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, cq = (lane & 15) * 4;
  float4 gq[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {                                 // every load issued before the first store
    const int q = p0 + warp * 8 + i * 2 + (lane >> 4), hq = q / Wq, wq = q - hq * Wq;
    gq[i] = (q < nwin && hq < Hp && wq < Wp && c0 + cq < C) ? ldv(dP + (((size_t)b * Hp + hq) * Wp + wq) * C + c0 + cq)
                                                            : make_float4(0.f, 0.f, 0.f, 0.f);
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int pl = warp * 8 + i * 2 + (lane >> 4);
    t[pl][cq] = gq[i].x; t[pl][cq + 1] = gq[i].y; t[pl][cq + 2] = gq[i].z; t[pl][cq + 3] = gq[i].w;
  }
}

// partial[c * (B * nseg) + b * nseg + seg] = (sum g, sum g x^) over the source pixels of the segment's windows, g = dP / 4 where the
// pre-activation is positive (the dropped row / column has g = 0 and adds nothing)
template <class T>
__global__ void __launch_bounds__(256) pool_bwd_reduce_kernel(const T* __restrict__ x, long long xbs, int C, int H, int W,
                                                              const T* __restrict__ dP, const float2* __restrict__ saved,
                                                              const float* __restrict__ weight, const float* __restrict__ bias,
                                                              int chunks_per_seg, float2* __restrict__ partial) {
  __shared__ float t[64][65];                                   // dP tile, [window][channel]
  const int seg = blockIdx.x, nseg = gridDim.x, c0 = blockIdx.y * 64, b = blockIdx.z, B = gridDim.z;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int Hp = H >> 1, Wp = W >> 1, P = Hp * Wp;
  float mu[8], rs[8], w[8], bb[8], s1[8], s2[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    const int c = min(c0 + warp * 8 + i, C - 1);
    const float2 st = saved[c];
    mu[i] = st.x; rs[i] = st.y; w[i] = weight[c]; bb[i] = bias[c]; s1[i] = 0.f; s2[i] = 0.f;
  }
  const int nchunks = (P + 63) / 64;
  for (int ch = seg * chunks_per_seg; ch < min(nchunks, (seg + 1) * chunks_per_seg); ++ch) {
    const int p0 = ch * 64;
    __syncthreads();                                            // the previous chunk's tile has been consumed
    dp_tile(dP, b, C, c0, Hp, Wp, Wp, P, p0, t);
    __syncthreads();
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int cl = warp * 8 + i, c = c0 + cl;
      if (c >= C) continue;
      const T* plane = x + (size_t)b * xbs + (size_t)c * H * W;
#pragma unroll
      for (int k = 0; k < 2; ++k) {
        const int pl = lane + 32 * k, p = p0 + pl;
        if (p >= P) continue;
        const int hq = p / Wp;
        float v[4];
        win_load(plane, H, W, hq, p - hq * Wp, v);
        const float g = 0.25f * t[pl][cl];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float xh = (v[u] - mu[i]) * rs[i];
          const float gg = fmaf(w[i], xh, bb[i]) > 0.f ? g : 0.f;
          s1[i] += gg;
          s2[i] = fmaf(gg, xh, s2[i]);
        }
      }
    }
  }
  // the 32 lanes of a channel, summed in a fixed shuffle-tree order
#pragma unroll
  for (int i = 0; i < 8; ++i) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      s1[i] += __shfl_down_sync(0xffffffffu, s1[i], o);
      s2[i] += __shfl_down_sync(0xffffffffu, s2[i], o);
    }
    const int c = c0 + warp * 8 + i;
    if (lane == 0 && c < C) partial[(size_t)c * ((size_t)B * nseg) + (size_t)b * nseg + seg] = make_float2(s1[i], s2[i]);
  }
}

// dx (NCHW, batch stride dbs) (+)= w rstd (g - mean(g) - x^ mean(g x^)) for EVERY source pixel: the grid runs over the
// ceil(H/2) x ceil(W/2) windows, those past the pooled map covering the dropped row / column with g = 0
template <class T, bool ACC>
__global__ void __launch_bounds__(256) pool_bwd_dx_kernel(const T* __restrict__ x, long long xbs, int C, int H, int W,
                                                          const T* __restrict__ dP, const float2* __restrict__ saved,
                                                          const float* __restrict__ weight, const float* __restrict__ bias,
                                                          const float2* __restrict__ sums, float inv_n, T* __restrict__ dx, long long dbs) {
  __shared__ float t[64][65];
  const int b = blockIdx.z, c0 = blockIdx.y * 64, p0 = blockIdx.x * 64;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int Wq = (W + 1) >> 1, nwin = ((H + 1) >> 1) * Wq;
  dp_tile(dP, b, C, c0, H >> 1, W >> 1, Wq, nwin, p0, t);
  __syncthreads();
#pragma unroll 2
  for (int i = 0; i < 8; ++i) {
    const int c = c0 + warp * 8 + i;
    if (c >= C) continue;
    const float2 st = saved[c], sm = sums[c];
    const float mu = st.x, rs = st.y, w = weight[c], bb = bias[c], k = w * rs, m1 = sm.x * inv_n, m2 = sm.y * inv_n;
    const T* plane = x + (size_t)b * xbs + (size_t)c * H * W;
    T* dplane = dx + (size_t)b * dbs + (size_t)c * H * W;
#pragma unroll
    for (int kk = 0; kk < 2; ++kk) {
      const int pl = lane + 32 * kk, q = p0 + pl;
      if (q >= nwin) continue;
      const int hq = q / Wq, wq = q - hq * Wq;
      float v[4];
      win_load(plane, H, W, hq, wq, v);
      const float g = 0.25f * t[pl][warp * 8 + i];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int h = 2 * hq + (u >> 1), ww = 2 * wq + (u & 1);
        if (h >= H || ww >= W) continue;
        const float xh = (v[u] - mu) * rs;
        const float gg = fmaf(w, xh, bb) > 0.f ? g : 0.f;
        T* d = dplane + (size_t)h * W + ww;
        float o = k * (gg - m1 - xh * m2);
        if (ACC) o += ld1v(static_cast<const T*>(d));
        st1v(d, o);
      }
    }
  }
}

// plain layout changes of a channel slice: NHWC (B, HW, C) -> NCHW slice (batch stride dbs), and back
template <class T>
__global__ void __launch_bounds__(256) cl_to_nchw_kernel(const T* __restrict__ src, int C, int HW, T* __restrict__ dst, long long dbs) {
  __shared__ float t[64][65];
  const int b = blockIdx.z, c0 = blockIdx.y * 64, p0 = blockIdx.x * 64;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  {
    const int cl = (lane & 15) * 4;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const int pl = warp * 8 + i * 2 + (lane >> 4), px = p0 + pl;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (px < HW && c0 + cl < C) v = ldv(src + ((size_t)b * HW + px) * C + c0 + cl);
      t[pl][cl] = v.x; t[pl][cl + 1] = v.y; t[pl][cl + 2] = v.z; t[pl][cl + 3] = v.w;
    }
  }
  __syncthreads();
  const int px = p0 + (lane & 15) * 4, pl = (lane & 15) * 4;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int cl = warp * 8 + i * 2 + (lane >> 4), c = c0 + cl;
    if (c < C && px < HW) stv(dst + (size_t)b * dbs + (size_t)c * HW + px, make_float4(t[pl][cl], t[pl + 1][cl], t[pl + 2][cl], t[pl + 3][cl]));
  }
}
template <class T>
__global__ void __launch_bounds__(256) nchw_to_cl_kernel(const T* __restrict__ src, long long sbs, int C, int HW, T* __restrict__ dst) {
  __shared__ float t[64][65];
  const int b = blockIdx.z, c0 = blockIdx.y * 64, p0 = blockIdx.x * 64;
  tile_load_nchw(src + (size_t)b * sbs + (size_t)c0 * HW, C, c0, HW, p0, t, [](int, float4 v) { return v; });
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, cl = (lane & 15) * 4;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int pl = warp * 8 + i * 2 + (lane >> 4), px = p0 + pl;
    if (px < HW && c0 + cl < C) stv(dst + ((size_t)b * HW + px) * C + c0 + cl, make_float4(t[pl][cl], t[pl][cl + 1], t[pl][cl + 2], t[pl][cl + 3]));
  }
}

int tpr_log2(int C) {
  const int Q = C / 4;
  int l = 0;
  while ((1 << l) < Q && l < 8) ++l;
  return l;
}
int aligned4(const void* p, size_t elt) { return (reinterpret_cast<uintptr_t>(p) & (4 * elt - 1)) == 0; }

}  // namespace

// workspace layout of the channels-last calls (floats): [0, 2*C) sums / spare, then the partials
static int cl_rows_per_cta(long long rows) {   // ~4 CTAs per SM when the tensor allows it, 32..256 rows each
  const long long want = (rows + 591) / 592;
  return (int)std::max<long long>(32, std::min<long long>(CL_ROWS, (want + 7) / 8 * 8));
}
static size_t cl_partials(int B, int C, int HW, int x_is_cl) {
  if (x_is_cl) { const long long rows = (long long)B * HW; return (size_t)((rows + cl_rows_per_cta(rows) - 1) / cl_rows_per_cta(rows)) * C; }
  const int nchunks = cdiv(HW, 64), ctiles = cdiv(C, 64);
  const int nseg = std::max(1, std::min(nchunks, cdiv(T_RED_CTAS, ctiles * B)));
  return (size_t)C * B * nseg;
}

template <class T>
int cl_fwd(const T* x, int B, int C, int HW, int x_is_cl, long long xbs, const float* w, const float* b, float* rm, float* rv, float momentum,
           float eps, T* y, float* saved, float* ws, const float* nchw_partial, int G, float n_each, float n_last, cudaStream_t st) {
  if (x_is_cl) {
    const long long rows = (long long)B * HW;
    const int rpc = cl_rows_per_cta(rows), nseg = (int)((rows + rpc - 1) / rpc), l = tpr_log2(C);
    float2* part = reinterpret_cast<float2*>(ws) + C;
    cl_stats_kernel<T><<<nseg, 256, sizeof(float) * (256 >> l) * C, AACONV_ST(st)>>>(x, rows, rpc, C, l, part);
    AACONV_LAUNCH_OK("bn_cl_stats");
    const float last = (float)(rows - (long long)(nseg - 1) * rpc);
    bn_fin_fwd_kernel<<<cdiv(C, 8), 256, 0, AACONV_ST(st)>>>(part, C, nseg, 1, C, (float)rpc, last, eps, momentum,
                                                              reinterpret_cast<float2*>(saved), rm, rv);
    AACONV_LAUNCH_OK("bn_fin_fwd");
    const long long nquads = rows * (C / 4);
    const int grid = (int)std::min<long long>((nquads + 255) / 256, 148 * 16);
    cl_apply_kernel<T, false><<<std::max(grid, cdiv(C / 4, 256)), 256, 0, AACONV_ST(st)>>>(x, nquads, C, reinterpret_cast<const float2*>(saved),
                                                                                          w, b, y, nullptr, nullptr, 0.f);
    AACONV_LAUNCH_OK("bn_cl_apply");
    return 0;
  }
  t_apply_kernel<T, false><<<dim3(cdiv(HW, 64), cdiv(C, 64), B), 256, 0, AACONV_ST(st)>>>(x, xbs, C, HW, reinterpret_cast<const float2*>(nchw_partial),
                                                                                         G, n_each, n_last, eps, momentum,
                                                                                         reinterpret_cast<float2*>(saved), rm, rv, w, b, y);
  AACONV_LAUNCH_OK("bn_t_apply");
  return 0;
}

// eval mode: the apply passes alone, their affine maps from the running statistics (read only: the const_casts below feed a kernel
// parameter that the EVAL instantiation never writes through)
template <class T>
int cl_eval(const T* x, int B, int C, int HW, int x_is_cl, long long xbs, const float* w, const float* b, const float* rm, const float* rv,
            float eps, T* y, cudaStream_t st) {
  if (x_is_cl) {
    const long long nquads = (long long)B * HW * (C / 4);
    const int grid = (int)std::min<long long>((nquads + 255) / 256, 148 * 16);
    cl_apply_kernel<T, true><<<std::max(grid, cdiv(C / 4, 256)), 256, 0, AACONV_ST(st)>>>(x, nquads, C, nullptr, w, b, y, rm, rv, eps);
    AACONV_LAUNCH_OK("bn_cl_eval");
    return 0;
  }
  t_apply_kernel<T, true><<<dim3(cdiv(HW, 64), cdiv(C, 64), B), 256, 0, AACONV_ST(st)>>>(x, xbs, C, HW, nullptr, 0, 0.f, 0.f, eps, 0.f, nullptr,
                                                                                        const_cast<float*>(rm), const_cast<float*>(rv), w, b, y);
  AACONV_LAUNCH_OK("bn_t_eval");
  return 0;
}

template <class T>
int cl_bwd(const T* x, int B, int C, int HW, int x_is_cl, long long xbs, const T* dy, const float* saved, const float* w, const float* b, T* dx,
           long long dbs, int acc, float* dw, float* db, float* ws, cudaStream_t st) {
  float2* sums = reinterpret_cast<float2*>(ws);
  float2* part = sums + C;
  const float inv_n = 1.f / ((float)B * HW);
  if (x_is_cl) {
    const long long rows = (long long)B * HW;
    const int rpc = cl_rows_per_cta(rows), nseg = (int)((rows + rpc - 1) / rpc), l = tpr_log2(C);
    cl_bwd_reduce_kernel<T><<<nseg, 256, sizeof(float) * 2 * (256 >> l) * C, AACONV_ST(st)>>>(x, dy, rows, rpc, C, l, reinterpret_cast<const float2*>(saved),
                                                                                            w, b, part);
    AACONV_LAUNCH_OK("bn_cl_bwd_reduce");
    bn_fin_bwd_kernel<<<cdiv(C, 8), 256, 0, AACONV_ST(st)>>>(part, C, nseg, 1, C, sums, dw, db);
    AACONV_LAUNCH_OK("bn_fin_bwd");
    if (!dx) return 0;
    const long long nquads = rows * (C / 4);
    const int grid = (int)std::min<long long>((nquads + 255) / 256, 148 * 16);
    cl_bwd_dx_kernel<T><<<std::max(grid, cdiv(C / 4, 256)), 256, 0, AACONV_ST(st)>>>(x, dy, nquads, C, reinterpret_cast<const float2*>(saved), w, b, sums,
                                                                                    inv_n, dx);
    AACONV_LAUNCH_OK("bn_cl_bwd_dx");
    return 0;
  }
  const int nchunks = cdiv(HW, 64), ctiles = cdiv(C, 64);
  const int nseg0 = std::max(1, std::min(nchunks, cdiv(T_RED_CTAS, ctiles * B)));
  const int cps = cdiv(nchunks, nseg0), nseg = cdiv(nchunks, cps);
  t_bwd_reduce_kernel<T><<<dim3(nseg, ctiles, B), 256, 0, AACONV_ST(st)>>>(x, xbs, C, HW, dy, reinterpret_cast<const float2*>(saved), w, b, cps, part);
  AACONV_LAUNCH_OK("bn_t_bwd_reduce");
  bn_fin_bwd_kernel<<<cdiv(C, 8), 256, 0, AACONV_ST(st)>>>(part, C, B * nseg, (long long)B * nseg, 1, sums, dw, db);
  AACONV_LAUNCH_OK("bn_fin_bwd");
  if (!dx) return 0;
  dim3 grid(nchunks, ctiles, B);
  if (acc)
    t_bwd_dx_kernel<T, true><<<grid, 256, 0, AACONV_ST(st)>>>(x, xbs, C, HW, dy, reinterpret_cast<const float2*>(saved), w, b, sums, inv_n, dx, dbs);
  else
    t_bwd_dx_kernel<T, false><<<grid, 256, 0, AACONV_ST(st)>>>(x, xbs, C, HW, dy, reinterpret_cast<const float2*>(saved), w, b, sums, inv_n, dx, dbs);
  AACONV_LAUNCH_OK("bn_t_bwd_dx");
  return 0;
}

// BatchNorm + ReLU + AvgPool2d(2) of a Transition: the segments of the backward reduction (as t_bwd_reduce's, over windows)
static int pool_segments(int B, int C, int H, int W, int* chunks_per_seg) {
  const int nchunks = cdiv((H / 2) * (W / 2), 64), ctiles = cdiv(C, 64);
  const int nseg0 = std::max(1, std::min(nchunks, cdiv(T_RED_CTAS, ctiles * B)));
  const int cps = cdiv(nchunks, nseg0);
  if (chunks_per_seg) *chunks_per_seg = cps;
  return cdiv(nchunks, cps);
}

template <class T>
int pool_fwd(const T* x, int B, int C, int H, int W, long long xbs, int training, const float* w, const float* b, float* rm, float* rv,
             float momentum, float eps, T* y, float* saved, const float* nchw_partial, int G, float n_each, float n_last, cudaStream_t st) {
  const dim3 grid(cdiv((H / 2) * (W / 2), 64), cdiv(C, 64), B);
  const float2* part = reinterpret_cast<const float2*>(nchw_partial);
  if (training) {
    pool_apply_kernel<T, false><<<grid, 256, 0, AACONV_ST(st)>>>(x, xbs, C, H, W, part, G, n_each, n_last, eps, momentum,
                                                                 reinterpret_cast<float2*>(saved), rm, rv, w, b, y);
    AACONV_LAUNCH_OK("bn_pool_apply");
  } else {   // running statistics read only (the EVAL instantiation never writes through rm / rv)
    pool_apply_kernel<T, true><<<grid, 256, 0, AACONV_ST(st)>>>(x, xbs, C, H, W, nullptr, 0, 0.f, 0.f, eps, 0.f, nullptr, rm, rv, w, b, y);
    AACONV_LAUNCH_OK("bn_pool_eval");
  }
  return 0;
}

template <class T>
int pool_bwd(const T* x, int B, int C, int H, int W, long long xbs, const T* dP, const float* saved, const float* w, const float* b, T* dx,
             long long dbs, int acc, float* dw, float* db, float* ws, cudaStream_t st) {
  float2* sums = reinterpret_cast<float2*>(ws);
  float2* part = sums + C;
  const float2* sv = reinterpret_cast<const float2*>(saved);
  int cps = 0;
  const int nseg = pool_segments(B, C, H, W, &cps), ctiles = cdiv(C, 64);
  pool_bwd_reduce_kernel<T><<<dim3(nseg, ctiles, B), 256, 0, AACONV_ST(st)>>>(x, xbs, C, H, W, dP, sv, w, b, cps, part);
  AACONV_LAUNCH_OK("bn_pool_bwd_reduce");
  bn_fin_bwd_kernel<<<cdiv(C, 8), 256, 0, AACONV_ST(st)>>>(part, C, B * nseg, (long long)B * nseg, 1, sums, dw, db);
  AACONV_LAUNCH_OK("bn_fin_bwd");
  if (!dx) return 0;
  const dim3 grid(cdiv(((H + 1) / 2) * ((W + 1) / 2), 64), ctiles, B);
  const float inv_n = 1.f / ((float)B * H * W);
  if (acc)
    pool_bwd_dx_kernel<T, true><<<grid, 256, 0, AACONV_ST(st)>>>(x, xbs, C, H, W, dP, sv, w, b, sums, inv_n, dx, dbs);
  else
    pool_bwd_dx_kernel<T, false><<<grid, 256, 0, AACONV_ST(st)>>>(x, xbs, C, H, W, dP, sv, w, b, sums, inv_n, dx, dbs);
  AACONV_LAUNCH_OK("bn_pool_bwd_dx");
  return 0;
}

}  // namespace aaconv

using namespace aaconv;

extern "C" {

size_t aaconv_bn_relu_cl_workspace_bytes(int B, int C, int HW) {
  if (B <= 0 || C <= 0 || HW <= 0) return 0;
  const size_t p = std::max(cl_partials(B, C, HW, 0), cl_partials(B, C, HW, 1));
  return align256(sizeof(float) * 2 * ((size_t)C + p));
}

// NCHW group statistics of channels [stats_valid_channels, C) (the shared per-block buffer of aaconv_bn_relu_forward) are the caller's
// business when x is NCHW: this call expects them in nchw_stats ((C, G) float2, G and the group sizes as aaconv_bn_relu_forward lays
// them out) -- see chexpert_b200/fused_bn.py.
int aaconv_bn_relu_cl_forward(const void* x, int dtype, int B, int C, int HW, int x_is_cl, int64_t x_batch_stride, const float* weight,
                              const float* bias, float* running_mean, float* running_var, float momentum, float eps, void* y_cl, float* saved,
                              void* workspace, const void* nchw_stats, int stats_groups, int planes_per_group, void* stream) {
  if (!x || !weight || !bias || !y_cl || !saved || !workspace || B <= 0 || C <= 0 || HW <= 0 || (C & 3) || (HW & 3))
    return fail(AACONV_E_ARG, "bad bn_relu_cl_forward arguments (C and HW must be multiples of 4)");
  if (dtype != AACONV_FP32 && dtype != AACONV_BF16) return fail(AACONV_E_ARG, "bad bn_relu_cl dtype");
  if (x_is_cl && C > CL_MAX_C) return fail(AACONV_E_ARG, "bn_relu_cl_forward: an NHWC input has at most 4096 channels");
  if (!x_is_cl && (!nchw_stats || stats_groups <= 0 || planes_per_group <= 0 || x_batch_stride < (int64_t)C * HW))
    return fail(AACONV_E_ARG, "bn_relu_cl_forward: NCHW input needs its group statistics and batch stride");
  const size_t elt = dtype == AACONV_BF16 ? 2 : 4;
  if (!aligned4(x, elt) || !aligned4(y_cl, elt) || (!x_is_cl && ((size_t)x_batch_stride * elt) % (4 * elt)))
    return fail(AACONV_E_ARG, "bn_relu_cl_forward: tensors must be aligned for four-element accesses");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const float n_each = (float)planes_per_group * HW, n_last = (float)(B - (stats_groups - 1) * planes_per_group) * HW;
  return dtype == AACONV_BF16
             ? cl_fwd(static_cast<const bf16*>(x), B, C, HW, x_is_cl, x_batch_stride, weight, bias, running_mean, running_var, momentum, eps,
                      static_cast<bf16*>(y_cl), saved, static_cast<float*>(workspace), static_cast<const float*>(nchw_stats), stats_groups,
                      n_each, n_last, st)
             : cl_fwd(static_cast<const float*>(x), B, C, HW, x_is_cl, x_batch_stride, weight, bias, running_mean, running_var, momentum, eps,
                      static_cast<float*>(y_cl), saved, static_cast<float*>(workspace), static_cast<const float*>(nchw_stats), stats_groups,
                      n_each, n_last, st);
}

// dx: NHWC dense when x is NHWC; else NCHW through dx_batch_stride, added onto what is there when dx_accumulate != 0
int aaconv_bn_relu_cl_backward(const void* x, int dtype, int B, int C, int HW, int x_is_cl, int64_t x_batch_stride, const void* dy_cl,
                               const float* saved, const float* weight, const float* bias, void* dx, int64_t dx_batch_stride,
                               int dx_accumulate, float* dweight, float* dbias, void* workspace, void* stream) {
  if (!x || !dy_cl || !saved || !weight || !bias || !workspace || B <= 0 || C <= 0 || HW <= 0 || (C & 3) || (HW & 3))
    return fail(AACONV_E_ARG, "bad bn_relu_cl_backward arguments (C and HW must be multiples of 4)");
  if (dtype != AACONV_FP32 && dtype != AACONV_BF16) return fail(AACONV_E_ARG, "bad bn_relu_cl dtype");
  if (x_is_cl && C > CL_MAX_C) return fail(AACONV_E_ARG, "bn_relu_cl_backward: an NHWC input has at most 4096 channels");
  const size_t elt = dtype == AACONV_BF16 ? 2 : 4;
  if (!aligned4(x, elt) || !aligned4(dy_cl, elt) || (dx && !aligned4(dx, elt)) ||
      (!x_is_cl && (((size_t)x_batch_stride * elt) % (4 * elt) || (dx && ((size_t)dx_batch_stride * elt) % (4 * elt)))))
    return fail(AACONV_E_ARG, "bn_relu_cl_backward: tensors must be aligned for four-element accesses");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  return dtype == AACONV_BF16
             ? cl_bwd(static_cast<const bf16*>(x), B, C, HW, x_is_cl, x_batch_stride, static_cast<const bf16*>(dy_cl), saved, weight, bias,
                      static_cast<bf16*>(dx), dx_batch_stride, dx_accumulate, dweight, dbias, static_cast<float*>(workspace), st)
             : cl_bwd(static_cast<const float*>(x), B, C, HW, x_is_cl, x_batch_stride, static_cast<const float*>(dy_cl), saved, weight, bias,
                      static_cast<float*>(dx), dx_batch_stride, dx_accumulate, dweight, dbias, static_cast<float*>(workspace), st);
}

// layout change of a channel slice: to_nchw != 0: src NHWC (B, HW, C) dense -> dst NCHW with batch stride; else src NCHW (batch stride)
// -> dst NHWC dense
int aaconv_slice_layout(const void* src, void* dst, int dtype, int B, int C, int HW, int64_t nchw_batch_stride, int to_nchw, void* stream) {
  if (!src || !dst || B <= 0 || C <= 0 || HW <= 0 || (C & 3) || (HW & 3) || nchw_batch_stride < (int64_t)C * HW)
    return fail(AACONV_E_ARG, "bad slice_layout arguments (C and HW must be multiples of 4)");
  if (dtype != AACONV_FP32 && dtype != AACONV_BF16) return fail(AACONV_E_ARG, "bad slice_layout dtype");
  const size_t elt = dtype == AACONV_BF16 ? 2 : 4;
  if (!aligned4(src, elt) || !aligned4(dst, elt) || ((size_t)nchw_batch_stride * elt) % (4 * elt))
    return fail(AACONV_E_ARG, "slice_layout: tensors must be aligned for four-element accesses");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  dim3 grid(cdiv(HW, 64), cdiv(C, 64), B);
  if (dtype == AACONV_BF16) {
    if (to_nchw) cl_to_nchw_kernel<bf16><<<grid, 256, 0, AACONV_ST(st)>>>(static_cast<const bf16*>(src), C, HW, static_cast<bf16*>(dst), nchw_batch_stride);
    else nchw_to_cl_kernel<bf16><<<grid, 256, 0, AACONV_ST(st)>>>(static_cast<const bf16*>(src), nchw_batch_stride, C, HW, static_cast<bf16*>(dst));
  } else {
    if (to_nchw) cl_to_nchw_kernel<float><<<grid, 256, 0, AACONV_ST(st)>>>(static_cast<const float*>(src), C, HW, static_cast<float*>(dst), nchw_batch_stride);
    else nchw_to_cl_kernel<float><<<grid, 256, 0, AACONV_ST(st)>>>(static_cast<const float*>(src), nchw_batch_stride, C, HW, static_cast<float*>(dst));
  }
  AACONV_LAUNCH_OK(to_nchw ? "slice_cl_to_nchw" : "slice_nchw_to_cl");
  return 0;
}

// relu(BatchNorm2d in eval mode): NCHW (batch stride) -> NCHW (bn_relu.cu), NCHW (batch stride) -> NHWC (t_apply tiles), NHWC -> NHWC
int aaconv_bn_relu_eval(const void* x, int dtype, int B, int C, int HW, int x_is_cl, int64_t x_batch_stride, const float* weight,
                        const float* bias, const float* running_mean, const float* running_var, float eps, void* y, int y_is_cl,
                        void* stream) {
  if (!x || !weight || !bias || !running_mean || !running_var || !y || B <= 0 || C <= 0 || HW <= 0 || B > 65535)
    return fail(AACONV_E_ARG, "bad bn_relu_eval arguments");
  if (dtype != AACONV_FP32 && dtype != AACONV_BF16) return fail(AACONV_E_ARG, "bad bn_relu_eval dtype");
  if (x_is_cl && !y_is_cl)
    return fail(AACONV_E_ARG, "bn_relu_eval: an NHWC input needs an NHWC output (pairs: NCHW -> NCHW, NCHW -> NHWC, NHWC -> NHWC)");
  if (!x_is_cl && x_batch_stride < (int64_t)C * HW) return fail(AACONV_E_ARG, "bn_relu_eval: an NCHW input needs a batch stride >= C*HW");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  if (!y_is_cl)
    return bn_relu_eval_nchw(x, dtype, B, C, HW, x_batch_stride, weight, bias, running_mean, running_var, eps, y, st);
  if ((C & 3) || (HW & 3)) return fail(AACONV_E_ARG, "bn_relu_eval: an NHWC side needs C and HW multiples of 4");
  if (x_is_cl && C > CL_MAX_C) return fail(AACONV_E_ARG, "bn_relu_eval: an NHWC input has at most 4096 channels");
  const size_t elt = dtype == AACONV_BF16 ? 2 : 4;
  if (!aligned4(x, elt) || !aligned4(y, elt) || (!x_is_cl && ((size_t)x_batch_stride * elt) % (4 * elt)))
    return fail(AACONV_E_ARG, "bn_relu_eval: an NHWC side needs tensors aligned for four-element accesses");
  return dtype == AACONV_BF16
             ? cl_eval(static_cast<const bf16*>(x), B, C, HW, x_is_cl, x_batch_stride, weight, bias, running_mean, running_var, eps,
                       static_cast<bf16*>(y), st)
             : cl_eval(static_cast<const float*>(x), B, C, HW, x_is_cl, x_batch_stride, weight, bias, running_mean, running_var, eps,
                       static_cast<float*>(y), st);
}

// the limits the pooled kernels share: C % 4 == 0 (NHWC quads), at least one 2 x 2 window, four-element alignment of every tensor
// and batch stride (checked before the null pointers: the workspace query returns 0 for a shape past them)
static int pool_args_ok(const char* what, int dtype, int B, int C, int H, int W, int64_t xbs, const void* x, const void* p_cl,
                        const void* dx, int64_t dbs) {
  if (dtype != AACONV_FP32 && dtype != AACONV_BF16) return fail(AACONV_E_ARG, "%s: dtype must be fp32 or bf16", what);
  if (B <= 0 || B > 65535 || H < 2 || W < 2 || C <= 0 || (C & 3))
    return fail(AACONV_E_ARG, "%s: needs C a multiple of 4, H and W >= 2 and 1 <= B <= 65535 (got B=%d C=%d H=%d W=%d)", what, B, C, H, W);
  if (xbs < (int64_t)C * H * W || (dx && dbs < (int64_t)C * H * W))
    return fail(AACONV_E_ARG, "%s: batch strides must be >= C*H*W", what);
  const size_t elt = dtype == AACONV_BF16 ? 2 : 4;
  if (!aligned4(x, elt) || !aligned4(p_cl, elt) || (dx && !aligned4(dx, elt)) || ((size_t)xbs * elt) % (4 * elt) ||
      (dx && ((size_t)dbs * elt) % (4 * elt)))
    return fail(AACONV_E_ARG, "%s: tensors and batch strides must be aligned for four-element accesses", what);
  return 0;
}

size_t aaconv_bn_relu_pool_workspace_bytes(int B, int C, int H, int W) {
  if (B <= 0 || C <= 0 || H < 2 || W < 2) return 0;
  return align256(sizeof(float) * 2 * ((size_t)C + (size_t)C * B * pool_segments(B, C, H, W, nullptr)));
}

int aaconv_bn_relu_pool_forward(const void* x, int dtype, int B, int C, int H, int W, int64_t x_batch_stride, int training,
                                const float* weight, const float* bias, float* running_mean, float* running_var, float momentum, float eps,
                                void* y_cl, float* saved, const void* nchw_stats, int stats_groups, int planes_per_group, void* stream) {
  AACONV_TRY(pool_args_ok("bn_relu_pool_forward", dtype, B, C, H, W, x_batch_stride, x, y_cl, nullptr, 0));
  if (!x || !weight || !bias || !y_cl) return fail(AACONV_E_ARG, "bn_relu_pool_forward: null tensor");
  if (training && (!saved || !nchw_stats || stats_groups <= 0 || planes_per_group <= 0 ||
                   stats_groups != (B + planes_per_group - 1) / planes_per_group || (running_mean == nullptr) != (running_var == nullptr)))
    return fail(AACONV_E_ARG, "bn_relu_pool_forward: training needs saved and the group statistics of aaconv_bn_stats_nchw");
  if (!training && (!running_mean || !running_var)) return fail(AACONV_E_ARG, "bn_relu_pool_forward: eval mode needs the running statistics");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const int HW = H * W;
  const float n_each = (float)planes_per_group * HW, n_last = (float)(B - (stats_groups - 1) * planes_per_group) * HW;
  const float* part = static_cast<const float*>(nchw_stats);
  return dtype == AACONV_BF16
             ? pool_fwd(static_cast<const bf16*>(x), B, C, H, W, x_batch_stride, training, weight, bias, running_mean, running_var, momentum,
                        eps, static_cast<bf16*>(y_cl), saved, part, stats_groups, n_each, n_last, st)
             : pool_fwd(static_cast<const float*>(x), B, C, H, W, x_batch_stride, training, weight, bias, running_mean, running_var,
                        momentum, eps, static_cast<float*>(y_cl), saved, part, stats_groups, n_each, n_last, st);
}

int aaconv_bn_relu_pool_backward(const void* x, int dtype, int B, int C, int H, int W, int64_t x_batch_stride, const void* dP_cl,
                                 const float* saved, const float* weight, const float* bias, void* dx, int64_t dx_batch_stride,
                                 int dx_accumulate, float* dweight, float* dbias, void* workspace, void* stream) {
  AACONV_TRY(pool_args_ok("bn_relu_pool_backward", dtype, B, C, H, W, x_batch_stride, x, dP_cl, dx, dx_batch_stride));
  if (!x || !dP_cl || !saved || !weight || !bias || !workspace) return fail(AACONV_E_ARG, "bn_relu_pool_backward: null tensor");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* ws = static_cast<float*>(workspace);
  return dtype == AACONV_BF16
             ? pool_bwd(static_cast<const bf16*>(x), B, C, H, W, x_batch_stride, static_cast<const bf16*>(dP_cl), saved, weight, bias,
                        static_cast<bf16*>(dx), dx_batch_stride, dx_accumulate, dweight, dbias, ws, st)
             : pool_bwd(static_cast<const float*>(x), B, C, H, W, x_batch_stride, static_cast<const float*>(dP_cl), saved, weight, bias,
                        static_cast<float*>(dx), dx_batch_stride, dx_accumulate, dweight, dbias, ws, st);
}

}  // extern "C"
