// Radiograph preprocessing on the device: the reference's transform (chexpert.py:64-79)
//   Resize(S) -> CenterCrop(S) -> ToTensor (/255) -> Normalize(0.5330, 0.0349) -> 3-channel expand
// for a ragged batch of 8-bit grayscale images, one launch, bit-identical to torchvision's PIL path followed by
// evaluate.normalise_u8 on the device.
//
// Resize is PIL's 8-bit bilinear resampling (Resample.c): two separable passes, horizontal first, each skipped when its
// dimension does not change; the horizontal result is rounded to uint8 before the vertical pass reads it.  Coefficients are
// PIL's precompute_coeffs in IEEE double, evaluated here with explicitly rounded intrinsics (__dadd_rn / __dmul_rn /
// __ddiv_rn) so that nvcc cannot contract them into FMAs the host C code does not use, then quantised to 22 fractional bits.
//
// One CTA per (image, band of output rows).  It computes the horizontal coefficients of the S cropped columns and the
// vertical ones of its band into shared memory, runs the horizontal pass over just the input rows the band needs (uint8 rows
// in shared memory), then the vertical pass, the normalisation and three coalesced plane stores.
#include "common.cuh"

#include <cmath>

namespace aaconv {
namespace {

constexpr int kThreads = 256;
constexpr int kPrecisionBits = 22;                  // PIL's PRECISION_BITS for 8-bit images
constexpr int kGeomCols = 8;                        // byte offset, h, w, resized h, resized w, crop top, crop left, unused
constexpr int kMaxSide = 8192, kMinSize = 16, kMaxSize = 2048;
constexpr int kSmemTarget = 96 * 1024;              // bands shrink until a CTA fits this (two CTAs per SM)
constexpr int kSmemMax = 227 * 1024;

struct Axis {
  int in;
  double scale, fs, ss;
  int ksize;
};

__device__ __forceinline__ Axis make_axis(int in, int out) {
  Axis a;
  a.in = in;
  a.scale = __ddiv_rn((double)(float)in, (double)out);   // PIL: (double)(in1 - in0) / outSize with float box coordinates
  a.fs = a.scale < 1.0 ? 1.0 : a.scale;                 // filterscale; the bilinear support is 1.0 * filterscale
  a.ss = __ddiv_rn(1.0, a.fs);
  a.ksize = 2 * (int)ceil(a.fs) + 1;
  return a;
}

__device__ __forceinline__ double bilinear_weight(const Axis& a, int x, double center) {
  double t = __dmul_rn(__dadd_rn(__dadd_rn((double)x, -center), 0.5), a.ss);
  t = fabs(t);
  return t < 1.0 ? __dadd_rn(1.0, -t) : 0.0;
}

// PIL precompute_coeffs + normalize_coeffs_8bpc for output index xx: writes k[0, n) and returns the first input index.
__device__ int axis_coeffs(const Axis& a, int xx, int* __restrict__ k, int* n_out) {
  const double center = __dmul_rn(__dadd_rn((double)xx, 0.5), a.scale);
  int xmin = __double2int_rz(__dadd_rn(__dadd_rn(center, -a.fs), 0.5));
  if (xmin < 0) xmin = 0;
  int xmax = __double2int_rz(__dadd_rn(__dadd_rn(center, a.fs), 0.5));
  if (xmax > a.in) xmax = a.in;
  const int n = xmax - xmin;
  double ww = 0.0;
  for (int x = 0; x < n; ++x) ww = __dadd_rn(ww, bilinear_weight(a, x + xmin, center));
  for (int x = 0; x < n; ++x) {
    double w = bilinear_weight(a, x + xmin, center);
    if (ww != 0.0) w = __ddiv_rn(w, ww);
    k[x] = __double2int_rz(__dadd_rn(0.5, __dmul_rn(w, (double)(1 << kPrecisionBits))));   // weights are >= 0
  }
  *n_out = n;
  return xmin;
}

__device__ __forceinline__ int clip8(int acc) {
  return acc >= (256 << kPrecisionBits) ? 255 : acc <= 0 ? 0 : acc >> kPrecisionBits;
}

// Largest filterscale any image of the batch can have on either axis: the resized side is >= S, and a long side L resizes to
// int(S * L / short) >= S * L / short - 1, so in / out < max_side / (S - 1).
double max_filterscale(int max_side, int S) {
  const double fs = (double)max_side / (S - 1);
  return fs < 1.0 ? 1.0 : fs;
}

struct Plan {
  int band, kmax, rows_cap;
  size_t smem;
};

Plan plan_for(int max_side, int S) {
  const double fs = max_filterscale(max_side, S);
  Plan p;
  p.kmax = 2 * (int)std::ceil(fs) + 1;
  for (p.band = 16;; p.band >>= 1) {
    // input rows of one band: (band - 1) * scale between the first and last centres, plus the support on both sides and the
    // rounding of the two bounds
    p.rows_cap = (int)std::ceil((p.band + 1) * fs) + 2;
    p.smem = sizeof(int) * ((size_t)(S + p.band) * p.kmax + 2 * (S + p.band)) + (size_t)p.rows_cap * S;
    if (p.smem <= kSmemTarget || p.band == 1) return p;
  }
}

__global__ void __launch_bounds__(kThreads) radiograph_prep_kernel(const uint8_t* __restrict__ px, long long total_bytes,
                                                                   const long long* __restrict__ geometry, int S, int max_side,
                                                                   int band, int kmax, int rows_cap, float inv255, float mean,
                                                                   float inv_std, float* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem[];
  int* hk = reinterpret_cast<int*>(smem);   // (S, kmax): horizontal coefficients of the cropped columns (odd kmax: no bank conflicts)
  int* hx = hk + (size_t)S * kmax;          // (S): first input column
  int* hn = hx + S;                         // (S): taps
  int* vk = hn + S;                         // (band, kmax): vertical coefficients of the band's rows
  int* vy = vk + band * kmax;               // (band): first input row
  int* vn = vy + band;                      // (band): taps
  uint8_t* rows = reinterpret_cast<uint8_t*>(vn + band);   // (rows_cap, S): horizontally resampled input rows

  const int b = blockIdx.y, y0 = blockIdx.x * band;
  const int nout = min(band, S - y0);
  const long long* g = geometry + (size_t)b * kGeomCols;
  const long long off = g[0];
  const int h = (int)g[1], w = (int)g[2], rh = (int)g[3], rw = (int)g[4], top = (int)g[5], left = (int)g[6];
  float* o = out + (size_t)b * 3 * S * S;

  // geometry the host did not validate: fill this band with NaN rather than read outside the pixel buffer or shared memory
  bool ok = g[1] >= 1 && g[2] >= 1 && g[1] <= max_side && g[2] <= max_side && off >= 0 && off <= total_bytes - g[1] * g[2] &&
            g[3] >= S && g[4] >= S && g[5] >= 0 && g[6] >= 0 && g[5] <= g[3] - S && g[6] <= g[4] - S;
  const bool hpass = rw != w, vpass = rh != h;
  Axis ah{}, av{};
  if (ok) {
    ah = make_axis(w, rw);
    av = make_axis(h, rh);
    ok = (!hpass || ah.ksize <= kmax) && (!vpass || av.ksize <= kmax);
  }
  if (ok) {
    if (hpass)
      for (int ox = threadIdx.x; ox < S; ox += kThreads) hx[ox] = axis_coeffs(ah, left + ox, hk + (size_t)ox * kmax, hn + ox);
    if (vpass)
      for (int j = threadIdx.x; j < nout; j += kThreads) vy[j] = axis_coeffs(av, top + y0 + j, vk + j * kmax, vn + j);
  }
  __syncthreads();
  // input rows [r0, r1) feed the band; first / last taps are monotone in the output index
  const int r0 = vpass ? vy[0] : top + y0;
  const int r1 = vpass ? vy[nout - 1] + vn[nout - 1] : top + y0 + nout;
  if (!ok || r0 < 0 || r1 > h || r1 - r0 > rows_cap) {
    const float nan = __int_as_float(0x7fc00000);
    for (int i = threadIdx.x; i < nout * S; i += kThreads) {
      const size_t p = (size_t)(y0 + i / S) * S + i % S;
      o[p] = nan;
      o[(size_t)S * S + p] = nan;
      o[(size_t)2 * S * S + p] = nan;
    }
    return;
  }

  const uint8_t* img = px + off;
  for (int i = threadIdx.x; i < (r1 - r0) * S; i += kThreads) {
    const int r = i / S, ox = i - r * S;
    const uint8_t* src = img + (size_t)(r0 + r) * w;
    int v;
    if (hpass) {
      const int* k = hk + (size_t)ox * kmax;
      const uint8_t* s = src + hx[ox];
      int acc = 1 << (kPrecisionBits - 1);
      for (int t = 0; t < hn[ox]; ++t) acc += (int)s[t] * k[t];
      v = clip8(acc);
    } else {
      v = src[left + ox];
    }
    rows[i] = (uint8_t)v;
  }
  __syncthreads();

  for (int i = threadIdx.x; i < nout * S; i += kThreads) {
    const int j = i / S, ox = i - j * S;
    int v;
    if (vpass) {
      const int* k = vk + j * kmax;
      const uint8_t* s = rows + (size_t)(vy[j] - r0) * S + ox;
      int acc = 1 << (kPrecisionBits - 1);
      for (int t = 0; t < vn[j]; ++t) acc += (int)s[(size_t)t * S] * k[t];
      v = clip8(acc);
    } else {
      v = rows[i];
    }
    // evaluate.normalise_u8 as torch computes it on the device: a division by a Python scalar is a multiply by the float
    // reciprocal; each step rounded on its own (no FMA)
    const float x = __fmul_rn(__fsub_rn(__fmul_rn((float)v, inv255), mean), inv_std);
    const size_t p = (size_t)(y0 + j) * S + ox;
    o[p] = x;
    o[(size_t)S * S + p] = x;
    o[(size_t)2 * S * S + p] = x;
  }
}

}  // namespace

extern "C" {

int aaconv_radiograph_prep(const uint8_t* pixels, int64_t total_bytes, const int64_t* geometry, int B, int max_side, int S,
                           float* out, void* stream) {
  if (!pixels || !geometry || !out || total_bytes <= 0 || B <= 0 || B > 65535)
    return fail(AACONV_E_ARG, "bad radiograph_prep arguments (null pointer, total_bytes <= 0 or B outside [1, 65535])");
  if (max_side < 1 || max_side > kMaxSide)
    return fail(AACONV_E_ARG, "radiograph_prep: max_side %d outside [1, %d]", max_side, kMaxSide);
  if (S < kMinSize || S > kMaxSize) return fail(AACONV_E_ARG, "radiograph_prep: S %d outside [%d, %d]", S, kMinSize, kMaxSize);
  const Plan p = plan_for(max_side, S);
  if (p.smem > (size_t)kSmemMax)
    return fail(AACONV_E_UNSUPPORTED, "radiograph_prep: max_side %d at S %d needs %zu bytes of shared memory", max_side, S, p.smem);
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  AACONV_CUDA_OK(cudaFuncSetAttribute(radiograph_prep_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p.smem));
  // the constants of normalise_u8 as torch's CUDA kernels see them: Python floats rounded to float, reciprocals in float
  const float inv255 = 1.0f / 255.0f, mean = (float)0.5330, inv_std = 1.0f / (float)0.0349;
  const dim3 grid((S + p.band - 1) / p.band, B);
  radiograph_prep_kernel<<<grid, kThreads, p.smem, AACONV_ST(st)>>>(pixels, total_bytes, reinterpret_cast<const long long*>(geometry),
                                                                     S, max_side, p.band, p.kmax, p.rows_cap, inv255, mean, inv_std,
                                                                     out);
  AACONV_LAUNCH_OK("radiograph_prep");
  return 0;
}

}  // extern "C"

}  // namespace aaconv
