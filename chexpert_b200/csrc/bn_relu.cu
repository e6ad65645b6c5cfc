// Fused BatchNorm2d (training mode, batch statistics) + ReLU over a channel slice of the pre-allocated DenseBlock feature buffer
// (SURVEY.md section 8 row f3; the reference runs torchvision's _DenseLayer: norm1 -> relu1 -> conv1 -> norm2 -> relu2 -> conv2,
// tv densenet.py:31-95 under models/attn_aug_conv.py:479-482).
//
// Why it exists: layer i of a dense block normalises channels [0, c_i) of ALL features so far.  With the feature buffer that
// input is a strided view (batch stride = C_total * H * W), for which PyTorch's batch_norm falls off its fast path (a generic
// Welford reduce_kernel + three elementwise kernels: the buffered block was 7 % slower than torch.cat), and even on the fast
// path BN + ReLU forward / backward are 4 + 8 passes over the activations with ONE CTA per channel for the reductions (64
// CTAs on 148 SMs at the first layers).  Here:
//   forward   bn_stats   grid (C, G) (G groups of batch planes, see Geo): per-group (mean, M2) partials, Chan-merged later -> no cancellation.
//                        In a dense block layer i normalises channels [0, c_i) of which [0, c_{i-1}) were already reduced by
//                        layer i-1 (same data, same statistics): the caller keeps ONE partial buffer per block and passes
//                        `stats_valid_channels`, so only the layer's 32 new channels are reduced (the pass shrinks ~5x)
//             bn_apply   grid (C, G): merges the G partials of its channel (fixed order; computes them itself when G == 1),
//                        y = relu(w (x - mean) rstd + b); the group-0 block also writes mean / rstd for backward and updates
//                        running_mean / running_var
//   backward  bn_bwd_red grid (C, G): g = dy * [y > 0], partial (sum g, sum g x^) per group (skipped when G == 1)
//             bn_bwd_dx  grid (C, G): merges the partials (fixed order), dx = w rstd (g - mean(g) - x^ mean(g x^)), optionally ADDED
//                        into the gradient of the feature buffer; the group-0 block writes dweight = sum g x^ and dbias = sum g
// 3 / 5 passes, all reductions in a fixed order (bit-reproducible), x read through its strides, y / dx dense.
//   eval      bn_eval    grid (C, G): BatchNorm2d in eval mode, relu(x s + t) from the running statistics, the apply loop of bn_apply
//                        (aaconv_bn_relu_eval's NCHW -> NCHW variant: stem norm0, norm5, layers the channels-last tiles cannot take)
#include <algorithm>
#include <cstdlib>
#include <cuda_bf16.h>
#include "common.cuh"

namespace aaconv {

typedef __nv_bfloat16 bf16;

namespace {

template <class T> __device__ __forceinline__ float ld1(const T* p);
template <> __device__ __forceinline__ float ld1<float>(const float* p) { return __ldg(p); }
template <> __device__ __forceinline__ float ld1<bf16>(const bf16* p) { return __bfloat162float(*p); }
template <class T> __device__ __forceinline__ void st1(T* p, float v);
template <> __device__ __forceinline__ void st1<float>(float* p, float v) { *p = v; }
template <> __device__ __forceinline__ void st1<bf16>(bf16* p, float v) { *p = __float2bfloat16(v); }
__device__ __forceinline__ float4 ld4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
__device__ __forceinline__ float4 ld4(const bf16* p) {
  const uint2 u = __ldg(reinterpret_cast<const uint2*>(p));
  const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
  const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
  return make_float4(a.x, a.y, b.x, b.y);
}
// plain (coherent) loads of data this kernel also writes
__device__ __forceinline__ float ld1_rw(const float* p) { return *p; }
__device__ __forceinline__ float ld1_rw(const bf16* p) { return __bfloat162float(*p); }
__device__ __forceinline__ float4 ld4_rw(const float* p) { return *reinterpret_cast<const float4*>(p); }
__device__ __forceinline__ float4 ld4_rw(const bf16* p) {
  const uint2 u = *reinterpret_cast<const uint2*>(p);
  const float2 a = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.x));
  const float2 b = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&u.y));
  return make_float4(a.x, a.y, b.x, b.y);
}
__device__ __forceinline__ void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
__device__ __forceinline__ void st4(bf16* p, float4 v) {
  const __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
  uint2 u;
  u.x = *reinterpret_cast<const uint32_t*>(&a);
  u.y = *reinterpret_cast<const uint32_t*>(&b);
  *reinterpret_cast<uint2*>(p) = u;
}

// fixed-order block sum of two values (256 threads)
__device__ __forceinline__ float2 block_sum2(float a, float b, float2* sh) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    a += __shfl_xor_sync(0xffffffffu, a, o);
    b += __shfl_xor_sync(0xffffffffu, b, o);
  }
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) sh[warp] = make_float2(a, b);
  __syncthreads();
  float2 t = make_float2(0.f, 0.f);
#pragma unroll
  for (int w = 0; w < 8; ++w) { t.x += sh[w].x; t.y += sh[w].y; }
  return t;
}

// Work decomposition.  One CTA handles channel c of a GROUP of `bpb` consecutive batch planes (grid (C, G), G = ceil(B / bpb)):
// bpb is chosen on the host so that a CTA touches ~8 k elements whatever the plane size.  With one CTA per (b, c) plane the
// 20x20 and 10x10 blocks of DenseNet121 launched 10-12 k CTAs of 100-400 elements each (25 active threads at 10x10): the four
// kernels averaged 4-16 us per call against 1-3 us of HBM time and were 31 % of the training step (round-2 profile).
// Inside a CTA the 256 threads form a (256 / tx) x tx grid, tx = the power of two covering a plane's vectors: ty planes are
// processed side by side; no integer division anywhere.
struct Geo {
  int B, HW, bpb, G;
  int unit;          // elements per access: 4 (vector path) or 1
  int n_unit;        // HW / unit
  int txl;           // log2(tx)
  long long xbs;
};
__device__ __forceinline__ int planes_of(const Geo& g, int grp) { return min(g.bpb, g.B - grp * g.bpb); }

// f(plane-in-group, element offset) over this thread's share of the group
template <class F>
__device__ __forceinline__ void for_each(const Geo& g, int nplanes, F f) {
  const int tx = 1 << g.txl, ox = threadIdx.x & (tx - 1), py = threadIdx.x >> g.txl, ty = 256 >> g.txl;
  for (int p = py; p < nplanes; p += ty)
    for (int o = ox; o < g.n_unit; o += tx) f(p, o * g.unit);
}

// partial[c * G + grp] = (mean, M2) of channel c over the planes of group grp: two passes (the data stays in L1 / L2 between them)
template <class T>
__global__ void __launch_bounds__(256) bn_stats_kernel(const T* __restrict__ x, const Geo g, float2* __restrict__ partial, int c_from) {
  __shared__ float2 sh[8];
  const int c = c_from + blockIdx.x, grp = blockIdx.y, np = planes_of(g, grp);
  const T* px = x + (size_t)(grp * g.bpb) * g.xbs + (size_t)c * g.HW;
  float s = 0.f;
  if (g.unit == 4) for_each(g, np, [&](int p, int o) { const float4 v = ld4(px + (size_t)p * g.xbs + o); s += (v.x + v.y) + (v.z + v.w); });
  else for_each(g, np, [&](int p, int o) { s += ld1(px + (size_t)p * g.xbs + o); });
  const float mean = block_sum2(s, 0.f, sh).x / ((float)np * g.HW);
  float q = 0.f;
  if (g.unit == 4) {
    for_each(g, np, [&](int p, int o) {
      const float4 v = ld4(px + (size_t)p * g.xbs + o);
      const float a0 = v.x - mean, a1 = v.y - mean, a2 = v.z - mean, a3 = v.w - mean;
      q += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
    });
  } else {
    for_each(g, np, [&](int p, int o) { const float a0 = ld1(px + (size_t)p * g.xbs + o) - mean; q += a0 * a0; });
  }
  const float m2 = block_sum2(q, 0.f, sh).x;
  if (threadIdx.x == 0) partial[(size_t)c * g.G + grp] = make_float2(mean, m2);
}

// Chan merge of the G group partials of channel c, in group order: -> (mean, biased var).  The partials are fetched by the
// block's threads in parallel (ONE memory latency, not G dependent ones), then combined by thread 0 in a fixed order.
__device__ __forceinline__ float2 merge_stats(const float2* __restrict__ partial, int c, const Geo& g, float2* sh /*[257]*/) {
  float n = 0.f, mean = 0.f, m2 = 0.f;
  for (int g0 = 0; g0 < g.G; g0 += 256) {
    const int ng = min(256, g.G - g0);
    __syncthreads();
    if ((int)threadIdx.x < ng) sh[threadIdx.x] = partial[(size_t)c * g.G + g0 + threadIdx.x];
    __syncthreads();
    if (threadIdx.x == 0) {
      for (int i = 0; i < ng; ++i) {
        const float2 p = sh[i];
        const float nb = (float)planes_of(g, g0 + i) * g.HW, tot = n + nb, d = p.x - mean, bf = __fdividef(nb, tot);
        mean += d * bf;                                  // (IEEE divisions made this serial loop ~100 cycles per step)
        m2 += p.y + d * d * (n * bf);
        n = tot;
      }
    }
  }
  if (threadIdx.x == 0) sh[256] = make_float2(mean, m2 / n);
  __syncthreads();
  return sh[256];
}
// plain sums of the G group partials of channel c, in group order
__device__ __forceinline__ float2 merge_sums(const float2* __restrict__ partial, int c, int G, float2* sh /*[257]*/) {
  float s1 = 0.f, s2 = 0.f;
  for (int g0 = 0; g0 < G; g0 += 256) {
    const int ng = min(256, G - g0);
    __syncthreads();
    if ((int)threadIdx.x < ng) sh[threadIdx.x] = partial[(size_t)c * G + g0 + threadIdx.x];
    __syncthreads();
    if (threadIdx.x == 0)
      for (int i = 0; i < ng; ++i) { s1 += sh[i].x; s2 += sh[i].y; }
  }
  if (threadIdx.x == 0) sh[256] = make_float2(s1, s2);
  __syncthreads();
  return sh[256];
}

// y (dense NCHW) = relu(x sc + sh) over channel c of group grp (this thread's share), x read through its batch stride
template <class T>
__device__ __forceinline__ void apply_relu_group(const T* __restrict__ x, T* __restrict__ y, const Geo& g, int c, int C, int grp, float sc,
                                                 float sh) {
  const int np = planes_of(g, grp), b0 = grp * g.bpb;
  const T* px = x + (size_t)b0 * g.xbs + (size_t)c * g.HW;
  T* py = y + ((size_t)b0 * C + c) * g.HW;
  const size_t ybs = (size_t)C * g.HW;
  if (g.unit == 4) {
    for_each(g, np, [&](int p, int o) {
      const float4 v = ld4(px + (size_t)p * g.xbs + o);
      st4(py + p * ybs + o, make_float4(fmaxf(fmaf(v.x, sc, sh), 0.f), fmaxf(fmaf(v.y, sc, sh), 0.f), fmaxf(fmaf(v.z, sc, sh), 0.f),
                                        fmaxf(fmaf(v.w, sc, sh), 0.f)));
    });
  } else {
    for_each(g, np, [&](int p, int o) { st1(py + p * ybs + o, fmaxf(fmaf(ld1(px + (size_t)p * g.xbs + o), sc, sh), 0.f)); });
  }
}

template <class T>
__global__ void __launch_bounds__(256) bn_apply_kernel(const T* __restrict__ x, const Geo g, const float2* __restrict__ partial,
                                                       const float* __restrict__ weight, const float* __restrict__ bias,
                                                       float* __restrict__ running_mean, float* __restrict__ running_var, float momentum,
                                                       float eps, T* __restrict__ y, float2* __restrict__ saved, int c_from,
                                                       float2* __restrict__ partial_out) {
  __shared__ float2 shm[257];
  const int c = blockIdx.x, grp = blockIdx.y, C = gridDim.x, np = planes_of(g, grp);
  float2 st;
  if (g.G == 1 && c >= c_from) {
    // one CTA owns the whole channel: its statistics are computed here (two more passes over data that stays in L1 / L2) and the
    // bn_stats launch is skipped; the partial is still written for the next layers of the dense block
    const T* px0 = x + (size_t)c * g.HW;
    float s = 0.f;
    if (g.unit == 4) for_each(g, np, [&](int p, int o) { const float4 v = ld4(px0 + (size_t)p * g.xbs + o); s += (v.x + v.y) + (v.z + v.w); });
    else for_each(g, np, [&](int p, int o) { s += ld1(px0 + (size_t)p * g.xbs + o); });
    const float mean = block_sum2(s, 0.f, shm).x / ((float)np * g.HW);
    float q = 0.f;
    if (g.unit == 4) {
      for_each(g, np, [&](int p, int o) {
        const float4 v = ld4(px0 + (size_t)p * g.xbs + o);
        const float a0 = v.x - mean, a1 = v.y - mean, a2 = v.z - mean, a3 = v.w - mean;
        q += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
      });
    } else {
      for_each(g, np, [&](int p, int o) { const float a0 = ld1(px0 + (size_t)p * g.xbs + o) - mean; q += a0 * a0; });
    }
    const float m2 = block_sum2(q, 0.f, shm).x;
    if (threadIdx.x == 0) partial_out[c] = make_float2(mean, m2);
    st = make_float2(mean, m2 / ((float)np * g.HW));
  } else {
    st = merge_stats(partial, c, g, shm);
  }
  const float rstd = rsqrtf(st.y + eps);
  if (grp == 0 && threadIdx.x == 0) {
    saved[c] = make_float2(st.x, rstd);
    if (running_mean) {                                    // nn.BatchNorm2d: unbiased variance in the running estimate
      const float n = (float)g.B * g.HW;
      running_mean[c] = (1.f - momentum) * running_mean[c] + momentum * st.x;
      running_var[c] = (1.f - momentum) * running_var[c] + momentum * st.y * (n / fmaxf(n - 1.f, 1.f));
    }
  }
  const float sc = weight[c] * rstd, sh = bias[c] - st.x * sc;
  apply_relu_group(x, y, g, c, C, grp, sc, sh);
}

// relu(BatchNorm2d eval) from the running statistics, NCHW -> NCHW: one pass, nothing to reduce.  Grid (C, G) as bn_apply.
template <class T>
__global__ void __launch_bounds__(256) bn_eval_kernel(const T* __restrict__ x, const Geo g, const float* __restrict__ weight,
                                                      const float* __restrict__ bias, const float* __restrict__ running_mean,
                                                      const float* __restrict__ running_var, float eps, T* __restrict__ y) {
  const float2 a = bn_eval_affine(weight, bias, running_mean, running_var, eps, blockIdx.x);
  apply_relu_group(x, y, g, blockIdx.x, gridDim.x, blockIdx.y, a.x, a.y);
}

// g = dy where the ReLU output is positive (recomputed from x and the saved statistics: y itself is not kept)
template <class T>
__global__ void __launch_bounds__(256) bn_bwd_reduce_kernel(const T* __restrict__ x, const Geo g, const T* __restrict__ dy,
                                                            const float2* __restrict__ saved, const float* __restrict__ weight,
                                                            const float* __restrict__ bias, float2* __restrict__ partial) {
  __shared__ float2 sh[8];
  const int c = blockIdx.x, grp = blockIdx.y, C = gridDim.x, np = planes_of(g, grp), b0 = grp * g.bpb;
  const float2 st = saved[c];
  const float w = weight[c], bb = bias[c];
  const T* px = x + (size_t)b0 * g.xbs + (size_t)c * g.HW;
  const T* pg = dy + ((size_t)b0 * C + c) * g.HW;
  const size_t ybs = (size_t)C * g.HW;
  float s1 = 0.f, s2 = 0.f;
  if (g.unit == 4) {
    for_each(g, np, [&](int p, int o) {
      const float4 xv = ld4(px + (size_t)p * g.xbs + o), gv = ld4(pg + p * ybs + o);
      const float xs[4] = {xv.x, xv.y, xv.z, xv.w}, gs[4] = {gv.x, gv.y, gv.z, gv.w};
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float xh = (xs[u] - st.x) * st.y;
        const float gg = fmaf(w, xh, bb) > 0.f ? gs[u] : 0.f;
        s1 += gg;
        s2 = fmaf(gg, xh, s2);
      }
    });
  } else {
    for_each(g, np, [&](int p, int o) {
      const float xh = (ld1(px + (size_t)p * g.xbs + o) - st.x) * st.y;
      const float gg = fmaf(w, xh, bb) > 0.f ? ld1(pg + p * ybs + o) : 0.f;
      s1 += gg;
      s2 = fmaf(gg, xh, s2);
    });
  }
  const float2 t = block_sum2(s1, s2, sh);
  if (threadIdx.x == 0) partial[(size_t)c * g.G + grp] = t;
}

// ACC: dx is ADDED onto a gradient that is already there, read and written through its own batch stride `dbs` -- the gradient of
// the dense block's feature buffer, of which this layer's input is a channel prefix (replaces a dense dx + autograd's add: two
// passes over the slice instead of five)
template <class T, bool ACC>
__global__ void __launch_bounds__(256) bn_bwd_dx_kernel(const T* __restrict__ x, const Geo g, const T* __restrict__ dy,
                                                        const float2* __restrict__ saved, const float* __restrict__ weight,
                                                        const float* __restrict__ bias, const float2* __restrict__ partial,
                                                        T* __restrict__ dx, long long dbs, float* __restrict__ dweight,
                                                        float* __restrict__ dbias) {
  __shared__ float2 shm[257];
  const int c = blockIdx.x, grp = blockIdx.y, C = gridDim.x, np = planes_of(g, grp), b0 = grp * g.bpb;
  float2 tot;
  if (g.G == 1) {     // one CTA owns the whole channel: the reduction pass runs here and the bn_bwd_reduce launch is skipped
    const float2 st0 = saved[c];
    const float w0 = weight[c], bb0 = bias[c];
    const T* px0 = x + (size_t)c * g.HW;
    const T* pg0 = dy + (size_t)c * g.HW;
    const size_t ybs0 = (size_t)C * g.HW;
    float a1 = 0.f, a2 = 0.f;
    if (g.unit == 4) {
      for_each(g, np, [&](int p, int o) {
        const float4 xv = ld4(px0 + (size_t)p * g.xbs + o), gv = ld4(pg0 + p * ybs0 + o);
        const float xs[4] = {xv.x, xv.y, xv.z, xv.w}, gs[4] = {gv.x, gv.y, gv.z, gv.w};
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const float xh = (xs[u] - st0.x) * st0.y;
          const float gg = fmaf(w0, xh, bb0) > 0.f ? gs[u] : 0.f;
          a1 += gg;
          a2 = fmaf(gg, xh, a2);
        }
      });
    } else {
      for_each(g, np, [&](int p, int o) {
        const float xh = (ld1(px0 + (size_t)p * g.xbs + o) - st0.x) * st0.y;
        const float gg = fmaf(w0, xh, bb0) > 0.f ? ld1(pg0 + p * ybs0 + o) : 0.f;
        a1 += gg;
        a2 = fmaf(gg, xh, a2);
      });
    }
    tot = block_sum2(a1, a2, reinterpret_cast<float2*>(shm));
  } else {
    tot = merge_sums(partial, c, g.G, shm);                              // group order
  }
  const float s1 = tot.x, s2 = tot.y;
  if (grp == 0 && threadIdx.x == 0) {
    if (dweight) dweight[c] = s2;
    if (dbias) dbias[c] = s1;
  }
  if (!dx) return;
  const float2 st = saved[c];
  const float w = weight[c], bb = bias[c], inv_n = 1.f / ((float)g.B * g.HW);
  const float m1 = s1 * inv_n, m2 = s2 * inv_n, k = w * st.y;
  const T* px = x + (size_t)b0 * g.xbs + (size_t)c * g.HW;
  const size_t ybs = (size_t)C * g.HW;
  const T* pg = dy + ((size_t)b0 * C + c) * g.HW;
  T* pd = dx + (size_t)b0 * dbs + (size_t)c * g.HW;
  if (g.unit == 4) {
    for_each(g, np, [&](int p, int o) {
      const float4 xv = ld4(px + (size_t)p * g.xbs + o), gv = ld4(pg + p * ybs + o);
      const float xs[4] = {xv.x, xv.y, xv.z, xv.w}, gs[4] = {gv.x, gv.y, gv.z, gv.w};
      float ov[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float xh = (xs[u] - st.x) * st.y;
        const float gg = fmaf(w, xh, bb) > 0.f ? gs[u] : 0.f;
        ov[u] = k * (gg - m1 - xh * m2);
      }
      T* q = pd + (size_t)p * dbs + o;
      if (ACC) { const float4 a = ld4_rw(q); ov[0] += a.x; ov[1] += a.y; ov[2] += a.z; ov[3] += a.w; }
      st4(q, make_float4(ov[0], ov[1], ov[2], ov[3]));
    });
  } else {
    for_each(g, np, [&](int p, int o) {
      const float xh = (ld1(px + (size_t)p * g.xbs + o) - st.x) * st.y;
      const float gg = fmaf(w, xh, bb) > 0.f ? ld1(pg + p * ybs + o) : 0.f;
      T* q = pd + (size_t)p * dbs + o;
      st1(q, k * (gg - m1 - xh * m2) + (ACC ? ld1_rw(q) : 0.f));
    });
  }
}

// host: group size, thread layout and whether every plane of every tensor can be accessed four elements at a time
template <class T>
Geo make_geo(int B, int C, int HW, long long xbs, const void* p0, const void* p1, const void* p2) {
  Geo g;
  g.B = B; g.HW = HW; g.xbs = xbs;
  static const int target = [] { const char* e = getenv("AACONV_BN_TARGET"); return e ? atoi(e) : 8192; }();   // elements per CTA (A/B)
  g.bpb = std::max(1, std::min(B, target / std::max(HW, 1)));
  g.G = (B + g.bpb - 1) / g.bpb;
  const size_t al = sizeof(T) * 4;                        // bytes of one four-element access (16 for fp32, 8 for bf16)
  const uintptr_t bits = reinterpret_cast<uintptr_t>(p0) | reinterpret_cast<uintptr_t>(p1) | reinterpret_cast<uintptr_t>(p2) |
                         (uintptr_t)((size_t)xbs * sizeof(T));
  (void)C;
  const bool vec = (HW & 3) == 0 && (bits & (al - 1)) == 0;
  g.unit = vec ? 4 : 1;
  g.n_unit = HW / g.unit;
  g.txl = 0;
  while ((1 << g.txl) < g.n_unit && g.txl < 8) ++g.txl;
  return g;
}

template <class T>
int fwd_t(const T* x, long long xbs, int B, int C, int HW, const float* w, const float* b, float* rm, float* rv, float momentum, float eps,
          T* y, float* saved, float* ws, int c_from, cudaStream_t st) {
  const Geo g = make_geo<T>(B, C, HW, xbs, x, y, nullptr);
  if (c_from < C && g.G > 1) {                            // group statistics of channels [c_from, C); the rest is already in `ws`
    bn_stats_kernel<T><<<dim3(C - c_from, g.G), 256, 0, AACONV_ST(st)>>>(x, g, reinterpret_cast<float2*>(ws), c_from);
    AACONV_LAUNCH_OK("bn_stats");
  }                                                       // (G == 1: the apply kernel reduces the new channels itself)
  bn_apply_kernel<T><<<dim3(C, g.G), 256, 0, AACONV_ST(st)>>>(x, g, reinterpret_cast<const float2*>(ws), w, b, rm, rv, momentum, eps, y,
                                                             reinterpret_cast<float2*>(saved), c_from, reinterpret_cast<float2*>(ws));
  AACONV_LAUNCH_OK("bn_relu_apply");
  return 0;
}
template <class T>
int bwd_t(const T* x, long long xbs, int B, int C, int HW, const T* dy, const float* saved, const float* w, const float* b, T* dx,
          long long dbs, int acc, float* dw, float* db, float* ws, cudaStream_t st) {
  Geo g = make_geo<T>(B, C, HW, xbs, x, dy, dx);
  if (g.unit == 4 && ((size_t)dbs * sizeof(T)) % (sizeof(T) * 4) != 0) { g.unit = 1; g.n_unit = HW; g.txl = 8; }
  dim3 grid(C, g.G);
  if (g.G > 1) {
    bn_bwd_reduce_kernel<T><<<grid, 256, 0, AACONV_ST(st)>>>(x, g, dy, reinterpret_cast<const float2*>(saved), w, b,
                                                             reinterpret_cast<float2*>(ws));
    AACONV_LAUNCH_OK("bn_relu_bwd_reduce");
  }
  if (acc)
    bn_bwd_dx_kernel<T, true><<<grid, 256, 0, AACONV_ST(st)>>>(x, g, dy, reinterpret_cast<const float2*>(saved), w, b,
                                                               reinterpret_cast<const float2*>(ws), dx, dbs, dw, db);
  else
    bn_bwd_dx_kernel<T, false><<<grid, 256, 0, AACONV_ST(st)>>>(x, g, dy, reinterpret_cast<const float2*>(saved), w, b,
                                                                reinterpret_cast<const float2*>(ws), dx, dbs, dw, db);
  AACONV_LAUNCH_OK("bn_relu_bwd_dx");
  return 0;
}

template <class T>
int eval_t(const T* x, long long xbs, int B, int C, int HW, const float* w, const float* b, const float* rm, const float* rv, float eps, T* y,
           cudaStream_t st) {
  const Geo g = make_geo<T>(B, C, HW, xbs, x, y, nullptr);
  bn_eval_kernel<T><<<dim3(C, g.G), 256, 0, AACONV_ST(st)>>>(x, g, w, b, rm, rv, eps, y);
  AACONV_LAUNCH_OK("bn_relu_eval");
  return 0;
}

}  // namespace

int bn_relu_eval_nchw(const void* x, int dtype, int B, int C, int HW, long long xbs, const float* weight, const float* bias,
                      const float* running_mean, const float* running_var, float eps, void* y, cudaStream_t st) {
  return dtype == AACONV_BF16 ? eval_t(static_cast<const bf16*>(x), xbs, B, C, HW, weight, bias, running_mean, running_var, eps,
                                       static_cast<bf16*>(y), st)
                              : eval_t(static_cast<const float*>(x), xbs, B, C, HW, weight, bias, running_mean, running_var, eps,
                                       static_cast<float*>(y), st);
}

}  // namespace aaconv

using namespace aaconv;

extern "C" {

size_t aaconv_bn_relu_workspace_bytes(int B, int C) { return (B > 0 && C > 0) ? align256(sizeof(float) * 2 * (size_t)B * C) : 0; }

int aaconv_bn_relu_forward(const void* x, int dtype, int B, int C, int HW, int64_t x_batch_stride, const float* weight, const float* bias,
                           float* running_mean, float* running_var, float momentum, float eps, void* y, float* saved, void* workspace,
                           int stats_valid_channels, void* stream) {
  if (!x || !weight || !bias || !y || !saved || !workspace || B <= 0 || C <= 0 || HW <= 0 || B > 65535 || stats_valid_channels < 0 ||
      stats_valid_channels > C)
    return fail(AACONV_E_ARG, "bad bn_relu_forward arguments");
  if ((dtype != AACONV_FP32 && dtype != AACONV_BF16) || x_batch_stride < (int64_t)C * HW) return fail(AACONV_E_ARG, "bad bn_relu dtype / stride");
  if ((running_mean == nullptr) != (running_var == nullptr)) return fail(AACONV_E_ARG, "running_mean and running_var come together");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* ws = static_cast<float*>(workspace);
  return dtype == AACONV_BF16
             ? fwd_t(static_cast<const bf16*>(x), x_batch_stride, B, C, HW, weight, bias, running_mean, running_var, momentum, eps,
                     static_cast<bf16*>(y), saved, ws, stats_valid_channels, st)
             : fwd_t(static_cast<const float*>(x), x_batch_stride, B, C, HW, weight, bias, running_mean, running_var, momentum, eps,
                     static_cast<float*>(y), saved, ws, stats_valid_channels, st);
}

// group statistics only (what aaconv_bn_relu_forward keeps in `workspace`), for callers that normalise with their own kernel
// (the channels-last path, bn_cl.cu): channels [stats_valid_channels, C) are reduced; *groups / *planes_per_group describe the layout
int aaconv_bn_stats_nchw(const void* x, int dtype, int B, int C, int HW, int64_t x_batch_stride, void* workspace, int stats_valid_channels,
                         int* groups, int* planes_per_group, void* stream) {
  if (!x || !workspace || !groups || !planes_per_group || B <= 0 || C <= 0 || HW <= 0 || B > 65535 || stats_valid_channels < 0 ||
      stats_valid_channels > C)
    return fail(AACONV_E_ARG, "bad bn_stats_nchw arguments");
  if ((dtype != AACONV_FP32 && dtype != AACONV_BF16) || x_batch_stride < (int64_t)C * HW) return fail(AACONV_E_ARG, "bad bn_stats dtype / stride");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  Geo g = dtype == AACONV_BF16 ? make_geo<bf16>(B, C, HW, x_batch_stride, x, nullptr, nullptr)
                               : make_geo<float>(B, C, HW, x_batch_stride, x, nullptr, nullptr);
  *groups = g.G;
  *planes_per_group = g.bpb;
  if (stats_valid_channels < C) {
    if (dtype == AACONV_BF16)
      bn_stats_kernel<bf16><<<dim3(C - stats_valid_channels, g.G), 256, 0, AACONV_ST(st)>>>(static_cast<const bf16*>(x), g,
                                                                                         static_cast<float2*>(workspace), stats_valid_channels);
    else
      bn_stats_kernel<float><<<dim3(C - stats_valid_channels, g.G), 256, 0, AACONV_ST(st)>>>(static_cast<const float*>(x), g,
                                                                                          static_cast<float2*>(workspace), stats_valid_channels);
    AACONV_LAUNCH_OK("bn_stats");
  }
  return 0;
}

int aaconv_bn_relu_backward(const void* x, int dtype, int B, int C, int HW, int64_t x_batch_stride, const void* dy, const float* saved,
                            const float* weight, const float* bias, void* dx, float* dweight, float* dbias, void* workspace, void* stream) {
  if (!x || !dy || !saved || !weight || !bias || !workspace || B <= 0 || C <= 0 || HW <= 0 || B > 65535)
    return fail(AACONV_E_ARG, "bad bn_relu_backward arguments");
  if ((dtype != AACONV_FP32 && dtype != AACONV_BF16) || x_batch_stride < (int64_t)C * HW) return fail(AACONV_E_ARG, "bad bn_relu dtype / stride");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* ws = static_cast<float*>(workspace);
  return dtype == AACONV_BF16 ? bwd_t(static_cast<const bf16*>(x), x_batch_stride, B, C, HW, static_cast<const bf16*>(dy), saved, weight, bias,
                                      static_cast<bf16*>(dx), (long long)C * HW, 0, dweight, dbias, ws, st)
                              : bwd_t(static_cast<const float*>(x), x_batch_stride, B, C, HW, static_cast<const float*>(dy), saved, weight,
                                      bias, static_cast<float*>(dx), (long long)C * HW, 0, dweight, dbias, ws, st);
}

int aaconv_bn_relu_backward_acc(const void* x, int dtype, int B, int C, int HW, int64_t x_batch_stride, const void* dy, const float* saved,
                                const float* weight, const float* bias, void* gacc, int64_t g_batch_stride, float* dweight, float* dbias,
                                void* workspace, void* stream) {
  if (!x || !dy || !saved || !weight || !bias || !workspace || !gacc || B <= 0 || C <= 0 || HW <= 0 || B > 65535)
    return fail(AACONV_E_ARG, "bad bn_relu_backward_acc arguments");
  if ((dtype != AACONV_FP32 && dtype != AACONV_BF16) || x_batch_stride < (int64_t)C * HW || g_batch_stride < (int64_t)C * HW)
    return fail(AACONV_E_ARG, "bad bn_relu dtype / stride");
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  float* ws = static_cast<float*>(workspace);
  return dtype == AACONV_BF16 ? bwd_t(static_cast<const bf16*>(x), x_batch_stride, B, C, HW, static_cast<const bf16*>(dy), saved, weight, bias,
                                      static_cast<bf16*>(gacc), g_batch_stride, 1, dweight, dbias, ws, st)
                              : bwd_t(static_cast<const float*>(x), x_batch_stride, B, C, HW, static_cast<const float*>(dy), saved, weight,
                                      bias, static_cast<float*>(gacc), g_batch_stride, 1, dweight, dbias, ws, st);
}

}  // extern "C"
