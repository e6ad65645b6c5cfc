// Operand builders and relative-logit adjoints around the tcgen05 attention kernels (bf16 path).
//
//   aug_build_fwd   q,k,v (fp32, head-split) -> augmented bf16 operands Qa, Ka (layout in attn_tc_bwd.cu)
//   rel_bwd         dQa -> total dq (content + relative part) written as bf16 into the packed dqkv operand of the
//                   projection GEMMs, and the key_rel_w / key_rel_h gradients
//
// The relative logits are rel_to_abs as an index computation (attn_aug_conv.py:43-63):
//   Aq[row, x'] = sum_e q[row,e] key_rel_w[e, x' - x(row) + W-1],   Bq[row, y'] = sum_e q[row,e] key_rel_h[e, y' - y(row) + H-1]
// i.e. a rank-dkh product R = q . key_rel followed by a per-row shift.  The products are small (K = dkh) and the
// shift is per row, so they run on mma.sync m16n8k8 TF32 (fp32 operands, 10-bit mantissa, far inside the bf16
// budget of the operands they feed), with the shift applied when fragments are scattered / gathered in shared
// memory; the three contractions are
//   forward   R[rows x 2N-1]   = Q[rows x dkh] . T[dkh x 2N-1]            -> shift -> Aq / Bq columns of Qa
//   dq_rel    [rows x dkh]     = dR[rows x 2N-1] . T^T                      dR[row, r] = dAq[row, r + x - (N-1)]
//   dT^T      [2N-1 x dkh]    += dR^T[2N-1 x rows] . Q[rows x dkh]          (accumulated in registers, fixed order)
#include <algorithm>
#include <cuda_bf16.h>
#include "tc_common.cuh"
#include "bf16_path.cuh"

namespace aaconv {

typedef __nv_bfloat16 bf16;

// ------------------------------------------------------------------------------------------------
// layout of the augmented operands
// ------------------------------------------------------------------------------------------------
AugLayout aug_layout(const Dims& d) {
  AugLayout a;
  a.KD = d.dkh + (d.relative ? d.W + d.H : 0);
  a.C1 = cdiv(a.KD + 2, 16) * 16;
  a.KP = cdiv(a.C1 + 16, 64) * 64;
  a.NQ = cdiv(a.KD, 16) * 16;
  return a;
}

int aug_supported(const Dims& d) {
  const AugLayout a = aug_layout(d);
  if (d.dvh + 2 > 16) return fail(AACONV_E_UNSUPPORTED, "bf16 attention kernels support dv/nh <= 14 (got %d)", d.dvh);
  if (a.KP > 192 || d.dkh > 32)
    return fail(AACONV_E_UNSUPPORTED, "bf16 attention kernels support dk/nh <= 32 and dk/nh + H + W <= 158 (got %d, %d)",
                d.dkh, a.KD);
  return 0;
}

namespace {

constexpr float LOG2E = 1.4426950408889634f;
constexpr int TR = 64;             // rows per tile (4 row groups of 16)

// Round-to-nearest TF32 operand without the conversion unit: the MMA ignores the low 13 mantissa bits, so adding half an ulp
// in the integer domain rounds (half away from zero).  cvt.rna.tf32.f32 runs on the XU pipe (16 lanes/clk/SM, shared with
// MUFU); the ncu capture of rel_bwd showed that pipe 58 % busy with these conversions next to a 62 % busy HMMA pipe.
__device__ __forceinline__ uint32_t f2tf32_alu(float x) { return __float_as_uint(x) + 0x1000u; }
__device__ __forceinline__ uint32_t f2tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
// D += A(16x8, row) * B(8x8, col), TF32 inputs, fp32 accumulate.
// A: a0=(g,t) a1=(g+8,t) a2=(g,t+4) a3=(g+8,t+4);  B: b0=(k=t,n=g) b1=(k=t+4,n=g);  C: c0=(g,2t) c1=(g,2t+1) c2=(g+8,2t) c3=(g+8,2t+1)
__device__ __forceinline__ void mma_tf32(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3, uint32_t b0,
                                         uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}

__device__ __forceinline__ void cp_async4(void* smem_dst, const void* gsrc) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc) : "memory");
}
// 1-D bulk copy global -> shared (TMA unit, no tensor map): dst/src 16 B aligned, bytes a multiple of 16
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)), "l"(gsrc), "r"(bytes),
                 "r"((uint32_t)__cvta_generic_to_shared(bar))
               : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() {
  asm volatile("cp.async.commit_group;\ncp.async.wait_group 0;" ::: "memory");
}

__device__ __forceinline__ void split_bf16(float x, bf16& hi, bf16& lo) {
  hi = __float2bfloat16(x);
  lo = __float2bfloat16(x - __bfloat162float(hi));
}

inline int table_pitch(int R) {   // >= roundup8(R) and == 8 (mod 32): conflict-free B-fragment loads (k = t, n = g)
  const int r8 = cdiv(R, 8) * 8;
  int p = r8;
  while (p % 32 != 8) ++p;
  return p;
}

struct BuildP {
  const float *q, *k, *v, *krw, *krh;
  bf16 *qa, *ka;
  int L, H, W, dkh, dvh, KD, C1, KP, relative;
  int DK8, RW, RH, PBW, PBH;       // padded K, table extents and pitches
  int tiles_per_bn, ntiles;
};

// ------------------------------------------------------------------------------------------------
// forward builder
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) aug_build_fwd_kernel(const BuildP p) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  uint32_t* tabw = reinterpret_cast<uint32_t*>(smem_raw);                 // [DK8][PBW] tf32
  uint32_t* tabh = tabw + (p.relative ? p.DK8 * p.PBW : 0);               // [DK8][PBH]
  // q, k, v tiles are contiguous copies of the global rows (one bulk copy each).  The MMA K padding (columns
  // dkh..DK8 of a q row) therefore reads the head of the next row / of ks: finite values (the float region is zeroed
  // once) that meet zero table rows.
  float* qs = reinterpret_cast<float*>(tabh + (p.relative ? p.DK8 * p.PBH : 0));   // [TR][dkh]
  float* ks = qs + TR * p.dkh;                                            // [TR][dkh]
  float* vs = ks + TR * p.dkh;                                            // [TR][dvh] (+ pad)
  const int PT = p.KP + 8;
  const int PQ = p.dkh;
  bf16* tq = reinterpret_cast<bf16*>(vs + ((TR * p.dvh + 3) & ~3) + 4);   // [TR][PT]
  bf16* tk = tq + TR * PT;
  int* rx = reinterpret_cast<int*>(tk + TR * PT);                         // [TR] x and y of each tile row
  int* ry = rx + TR;
  uint64_t* bar = reinterpret_cast<uint64_t*>(ry + TR);
  if (threadIdx.x == 0) { tc::mbar_init(bar, 1); tc::fence_barrier_init(); }

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  if (p.relative) {
    for (int i = threadIdx.x; i < p.DK8 * p.PBW; i += blockDim.x) {
      const int e = i / p.PBW, r = i - e * p.PBW;
      tabw[i] = (e < p.dkh && r < p.RW) ? f2tf32(p.krw[e * p.RW + r]) : 0u;
    }
    for (int i = threadIdx.x; i < p.DK8 * p.PBH; i += blockDim.x) {
      const int e = i / p.PBH, r = i - e * p.PBH;
      tabh[i] = (e < p.dkh && r < p.RH) ? f2tf32(p.krh[e * p.RH + r]) : 0u;
    }
  }
  for (int i = threadIdx.x; i < 2 * TR * p.dkh + ((TR * p.dvh + 3) & ~3) + 4; i += blockDim.x) qs[i] = 0.f;
  uint32_t phase = 0;
  // The tiles keep their constant part across the tiles of this CTA: zeros everywhere, ones in the lse / delta slots of
  // Ka.  Per tile only the k, v, q columns, the relative columns (MMA phase) and the two one-hot positions per row change.
  for (int i = threadIdx.x; i < 2 * TR * PT; i += blockDim.x) tq[i] = __float2bfloat16(0.f);   // tq and tk are adjacent
  if (threadIdx.x < TR) { rx[threadIdx.x] = -1; ry[threadIdx.x] = -1; }
  __syncthreads();
  for (int i = threadIdx.x; i < TR * 4; i += blockDim.x) {
    const int r = i >> 2, w = i & 3;
    const int c = (w < 2 ? p.KD : p.C1 + p.dvh) + (w & 1);
    tk[r * PT + c] = __float2bfloat16(1.f);
  }
  for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x) {
    const int bn = tile / p.tiles_per_bn, l0 = (tile - bn * p.tiles_per_bn) * TR;
    const int nrows = min(TR, p.L - l0);
    const size_t row0 = (size_t)bn * p.L + l0;
    __syncthreads();                                   // previous tile fully copied out; tables visible
    if (threadIdx.x < TR) {
      const int r = threadIdx.x, l = l0 + r, y = l / p.W, x = l - y * p.W;
      if (p.relative) {
        if (rx[r] >= 0) { tk[r * PT + p.dkh + rx[r]] = __float2bfloat16(0.f); tk[r * PT + p.dkh + p.W + ry[r]] = __float2bfloat16(0.f); }
        if (y < p.H) { tk[r * PT + p.dkh + x] = __float2bfloat16(1.f); tk[r * PT + p.dkh + p.W + y] = __float2bfloat16(1.f); }
      }
      rx[r] = y < p.H ? x : -1;
      ry[r] = y;
    }
    // tile loads: three 1-D bulk copies (TMA unit) when the blocks are 16 B aligned, else per-element LDGSTS
    const bool bulk = (((row0 * p.dkh) | (size_t)(nrows * p.dkh) | (row0 * p.dvh) | (size_t)(nrows * p.dvh)) & 3) == 0;
    if (bulk) {
      if (threadIdx.x == 0) {
        const uint32_t bq = nrows * p.dkh * 4, bv = nrows * p.dvh * 4;
        tc::mbar_arrive_expect_tx(bar, 2 * bq + bv);
        bulk_g2s(qs, p.q + row0 * p.dkh, bq, bar);
        bulk_g2s(ks, p.k + row0 * p.dkh, bq, bar);
        bulk_g2s(vs, p.v + row0 * p.dvh, bv, bar);
      }
      tc::mbar_wait(bar, phase);
      phase ^= 1;
    } else {
      for (int r = warp; r < nrows; r += 8) {
        if (lane < p.dkh) {
          cp_async4(qs + r * PQ + lane, p.q + (row0 + r) * p.dkh + lane);
          cp_async4(ks + r * p.dkh + lane, p.k + (row0 + r) * p.dkh + lane);
        }
        if (lane < p.dvh) cp_async4(vs + r * p.dvh + lane, p.v + (row0 + r) * p.dvh + lane);
      }
      cp_async_wait_all();
    }
    __syncthreads();

    // ---- relative columns of Qa: warps 0-3 the W axis, warps 4-7 the H axis, 16 rows each ----
    if (p.relative) {
      const int axis = warp >> 2, rg = (warp & 3) * 16;
      const int N = axis ? p.H : p.W, R = axis ? p.RH : p.RW, PB = axis ? p.PBH : p.PBW;
      const uint32_t* tab = axis ? tabh : tabw;
      const int colbase = p.dkh + (axis ? p.W : 0);
      const int ra = rg + g, rb = rg + g + 8;
      const int pos_a = axis ? ry[ra] : rx[ra], pos_b = axis ? ry[rb] : rx[rb];
      uint32_t af[4][4];
      const int nks = p.DK8 >> 3;
#pragma unroll
      for (int s = 0; s < 4; ++s)
        if (s < nks) {
          af[s][0] = f2tf32_alu(qs[ra * PQ + 8 * s + t] * LOG2E);
          af[s][1] = f2tf32_alu(qs[rb * PQ + 8 * s + t] * LOG2E);
          af[s][2] = f2tf32_alu(qs[ra * PQ + 8 * s + t + 4] * LOG2E);
          af[s][3] = f2tf32_alu(qs[rb * PQ + 8 * s + t + 4] * LOG2E);
        }
      const int NT = (R + 7) >> 3;
      for (int nt = 0; nt < NT; ++nt) {
        float c[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
        for (int s = 0; s < 4; ++s)
          if (s < nks) mma_tf32(c, af[s][0], af[s][1], af[s][2], af[s][3], tab[(8 * s + t) * PB + 8 * nt + g],
                                tab[(8 * s + t + 4) * PB + 8 * nt + g]);
        const int r = 8 * nt + 2 * t;                  // R[row, r], R[row, r+1];  abs position = r + pos - (N-1)
        const int xa = r + pos_a - (N - 1), xb = r + pos_b - (N - 1);
        if ((unsigned)xa < (unsigned)N) tq[ra * PT + colbase + xa] = __float2bfloat16(c[0]);
        if ((unsigned)(xa + 1) < (unsigned)N) tq[ra * PT + colbase + xa + 1] = __float2bfloat16(c[1]);
        if ((unsigned)xb < (unsigned)N) tq[rb * PT + colbase + xb] = __float2bfloat16(c[2]);
        if ((unsigned)(xb + 1) < (unsigned)N) tq[rb * PT + colbase + xb + 1] = __float2bfloat16(c[3]);
      }
    }
    // ---- data columns: c*q into Qa, k and v into Ka (everything else in the tiles is constant or written above) ----
    // (row = warp-strided, column = lane: no integer division in the per-tile loops -- a runtime division is three XU-pipe
    //  instructions, and the XU pipe was 98 % busy in the ncu capture of this kernel)
    for (int r = warp; r < TR; r += 8) {
      if (lane < p.dkh) {
        tq[r * PT + lane] = __float2bfloat16(qs[r * p.dkh + lane] * LOG2E);
        tk[r * PT + lane] = __float2bfloat16(ks[r * p.dkh + lane]);
      }
      if (lane < p.dvh) tk[r * PT + p.C1 + lane] = __float2bfloat16(vs[r * p.dvh + lane]);
    }
    __syncthreads();
    // ---- coalesced copy-out: rows of KP bf16 are contiguous in global memory ----
    const int vec_per_row = p.KP >> 3;                 // uint4 = 8 bf16
    uint4* gq = reinterpret_cast<uint4*>(p.qa + row0 * p.KP);
    uint4* gk = reinterpret_cast<uint4*>(p.ka + row0 * p.KP);
    if ((vec_per_row & (vec_per_row - 1)) == 0) {       // 8 or 16 vectors per row: shifts instead of a division
      const int sh = 31 - __clz(vec_per_row);
      for (int i = threadIdx.x; i < nrows * vec_per_row; i += blockDim.x) {
        const int r = i >> sh, c = i & (vec_per_row - 1);
        gq[i] = *reinterpret_cast<const uint4*>(tq + r * PT + c * 8);
        gk[i] = *reinterpret_cast<const uint4*>(tk + r * PT + c * 8);
      }
    } else {
      for (int i = threadIdx.x; i < nrows * vec_per_row; i += blockDim.x) {
        const int r = i / vec_per_row, c = i - r * vec_per_row;
        gq[i] = *reinterpret_cast<const uint4*>(tq + r * PT + c * 8);
        gk[i] = *reinterpret_cast<const uint4*>(tk + r * PT + c * 8);
      }
    }
  }
}

constexpr int OBP_THREADS = 128;   // 25600 pixels at Transition 1 -> 200 CTAs (256 threads left 48 of 148 SMs idle)
// ------------------------------------------------------------------------------------------------
// out_proj adjoint + backward patch of Qa in ONE pass over the pixels (small value widths: dv = NH * DVH <= 16)
//   dO[b,n,l,e] = sum_c Wout[c, n*dvh+e] dy[b, Cc+c, l]        (attn_aug_conv.py:92 adjoint, data)
//   dWout[c,j] += dy[b, Cc+c, l] * o[b, n(j), l, e(j)]          (weight; per-block partials, summed in block order by
//                                                                out_w_reduce_kernel: deterministic)
//   delta[b,n,l] = dO . o;  the backward-only columns of Qa: -lse (hi/lo), dO, -delta (hi/lo)
// Replaces four launches (out_bwd_data, out_bwd_weight, splitk_reduce, aug_patch_bwd: 56 us at Transition 1) whose
// work is 25600 pixels x 8 channels.
// ------------------------------------------------------------------------------------------------
template <int NH, int DVH>
__global__ void __launch_bounds__(OBP_THREADS) out_bwd_patch_kernel(const float* __restrict__ dy, const float* __restrict__ o,
                                                            const float* __restrict__ lse, const float* __restrict__ wout,
                                                            float* __restrict__ d_o, float* __restrict__ delta_out,
                                                            bf16* __restrict__ qa, float* __restrict__ wpartial, int B, int L,
                                                            int Ctot, int coff, int KD, int C1, int KP) {
  constexpr int DV = NH * DVH;
  __shared__ float ws[DV * DV];
  __shared__ float red[OBP_THREADS / 32][DV * DV];
  for (int i = threadIdx.x; i < DV * DV; i += blockDim.x) ws[i] = wout[i];
  __syncthreads();
  const int m = blockIdx.x * blockDim.x + threadIdx.x;
  const bool live = m < B * L;
  const int b = live ? m / L : 0, l = live ? m - b * L : 0;
  float dyv[DV], oc[DV];
#pragma unroll
  for (int c = 0; c < DV; ++c) dyv[c] = live ? dy[((size_t)b * Ctot + coff + c) * L + l] : 0.f;
#pragma unroll
  for (int h = 0; h < NH; ++h)
#pragma unroll
    for (int e = 0; e < DVH; ++e) oc[h * DVH + e] = live ? o[((size_t)(b * NH + h) * L + l) * DVH + e] : 0.f;
  if (live) {
#pragma unroll
    for (int h = 0; h < NH; ++h) {
      const size_t row = (size_t)(b * NH + h) * L + l;
      bf16* dst = qa + row * KP;
      bf16 hi, lo;
      split_bf16(-lse[row] * LOG2E, hi, lo);
      dst[KD] = hi;
      dst[KD + 1] = lo;
      float delta = 0.f;
#pragma unroll
      for (int e = 0; e < DVH; ++e) {
        const int j = h * DVH + e;
        float g = 0.f;
#pragma unroll
        for (int c = 0; c < DV; ++c) g = fmaf(ws[c * DV + j], dyv[c], g);
        d_o[row * DVH + e] = g;
        delta = fmaf(g, oc[j], delta);
        dst[C1 + e] = __float2bfloat16(g);
      }
      split_bf16(-delta, hi, lo);
      dst[C1 + DVH] = hi;
      dst[C1 + DVH + 1] = lo;
      delta_out[row] = delta;
    }
  }
  if (wpartial) {                                   // block partial of dWout: warp shuffles, then the 8 warps in fixed order
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
    for (int c = 0; c < DV; ++c)
#pragma unroll
      for (int j = 0; j < DV; ++j) {
        float v = dyv[c] * oc[j];
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) v += __shfl_xor_sync(0xffffffffu, v, s);
        if (lane == 0) red[warp][c * DV + j] = v;
      }
    __syncthreads();
    for (int i = threadIdx.x; i < DV * DV; i += blockDim.x) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < OBP_THREADS / 32; ++w) t += red[w][i];
      wpartial[(size_t)blockIdx.x * DV * DV + i] = t;
    }
  }
}

// head combine + out_proj + concat write (attn_aug_conv.py:89-95): y[b, Cc + n, l] = sum_k Wout[n, k] o[b, k / dvh, l, k % dvh].
// One thread per (output channel, pixel), consecutive threads = consecutive pixels: coalesced o reads and y writes, the Wout row
// is a shared-memory broadcast.  (The generic 64 x 64-tiled FFMA GEMM spent 10.6 us on these 25600 x 8 x 8 MACs.)
__global__ void __launch_bounds__(256) out_proj_fwd_kernel(const float* __restrict__ o, const float* __restrict__ wout, void* __restrict__ y,
                                                           int BL, int L, int nh, int dvh, int coff, long long y_bs, int y_bf16) {
  extern __shared__ float ws[];
  const int dv = nh * dvh;
  for (int i = threadIdx.x; i < dv * dv; i += blockDim.x) ws[i] = wout[i];
  __syncthreads();
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (size_t)BL * dv) return;
  const int n = (int)(t / BL), pix = (int)(t - (size_t)n * BL);
  const int b = pix / L, l = pix - b * L;
  const float* wr = ws + n * dv;
  float acc = 0.f;
  for (int h = 0; h < nh; ++h) {
    const float* op = o + ((size_t)(b * nh + h) * L + l) * dvh;
    for (int e = 0; e < dvh; ++e) acc = fmaf(wr[h * dvh + e], __ldg(op + e), acc);
  }
  store_y(y, (size_t)b * y_bs + (size_t)(coff + n) * L + l, acc, y_bf16);
}

// Any value width (dv/nh <= 14; Transition 2 / 3: dvh = 3 / 6): out_proj adjoint (data part) + the Qa patch, one thread per
// (batch, head, pixel) row.  Replaces out_bwd_data_f32 (a 64 x 64-tiled FFMA GEMM whose M x N = pixels x dv output gave it
// 25-100 CTAs with strided gathers: 76 / 171 us at Transition 2 / 3) and aug_patch_bwd.  dWout stays a split-K GEMM.
__global__ void __launch_bounds__(256) out_bwd_data_patch_kernel(const float* __restrict__ dy, const float* __restrict__ o,
                                                                 const float* __restrict__ lse, const float* __restrict__ wout,
                                                                 float* __restrict__ d_o, float* __restrict__ delta_out,
                                                                 bf16* __restrict__ qa, int B, int L, int nh, int dvh, int Ctot, int coff,
                                                                 int KD, int C1, int KP) {
  // block = 32 consecutive pixels x nh heads (warp = one head: coalesced row writes); dy of the 32 pixels is staged in shared
  // memory once (coalesced along the pixels) instead of dv dependent global loads per thread
  extern __shared__ float ws[];                     // Wout (dv x dv), row c = output channel of out_proj; then dys[dv][33]
  const int dv = nh * dvh;
  float* dys = ws + dv * dv;
  const int pix0 = blockIdx.x * 32, npix = B * L;
  for (int i = threadIdx.x; i < dv * dv; i += blockDim.x) ws[i] = wout[i];
  for (int i = threadIdx.x; i < dv * 32; i += blockDim.x) {
    const int c = i >> 5, pp = i & 31, pix = pix0 + pp;
    float v = 0.f;
    if (pix < npix) { const int b = pix / L, l = pix - b * L; v = __ldg(dy + ((size_t)b * Ctot + coff + c) * L + l); }
    dys[c * 33 + pp] = v;
  }
  __syncthreads();
  const int pp = threadIdx.x & 31, h = threadIdx.x >> 5, pix = pix0 + pp;
  if (pix >= npix || h >= nh) return;
  const int b = pix / L, l = pix - b * L;
  const size_t row = (size_t)(b * nh + h) * L + l;
  float g[14];
#pragma unroll
  for (int e = 0; e < 14; ++e) g[e] = 0.f;
  for (int c = 0; c < dv; ++c) {
    const float v = dys[c * 33 + pp];
    const float* wr = ws + c * dv + h * dvh;
#pragma unroll
    for (int e = 0; e < 14; ++e)
      if (e < dvh) g[e] = fmaf(wr[e], v, g[e]);
  }
  bf16* dst = qa + row * KP;
  bf16 hi, lo;
  split_bf16(-lse[row] * LOG2E, hi, lo);
  dst[KD] = hi;
  dst[KD + 1] = lo;
  float delta = 0.f;
#pragma unroll
  for (int e = 0; e < 14; ++e)
    if (e < dvh) {
      d_o[row * dvh + e] = g[e];
      delta = fmaf(g[e], o[row * dvh + e], delta);
      dst[C1 + e] = __float2bfloat16(g[e]);
    }
  split_bf16(-delta, hi, lo);
  dst[C1 + dvh] = hi;
  dst[C1 + dvh + 1] = lo;
  delta_out[row] = delta;
}

// block = 32 outputs x 8 slices of the block partials; slices, then the 8 slice sums, are added in a fixed order
__global__ void __launch_bounds__(256) out_w_reduce_kernel(const float* __restrict__ wpartial, int nblocks, int n,
                                                           float* __restrict__ dw) {
  __shared__ float red[8][33];
  const int o = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + o;
  float t = 0.f;
  if (i < n) {
    int k = sl;
    for (; k + 24 < nblocks; k += 32) {
      const float a = wpartial[(size_t)k * n + i], b = wpartial[(size_t)(k + 8) * n + i], c = wpartial[(size_t)(k + 16) * n + i],
                  d = wpartial[(size_t)(k + 24) * n + i];
      t = (((t + a) + b) + c) + d;
    }
    for (; k < nblocks; k += 8) t += wpartial[(size_t)k * n + i];
  }
  red[sl][o] = t;
  __syncthreads();
  if (sl == 0 && i < n) {
    float tot = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) tot += red[k][o];
    dw[i] = tot;
  }
}
}  // namespace

size_t aug_build_smem(const Dims& d) {
  const AugLayout a = aug_layout(d);
  const int DK8 = cdiv(d.dkh, 8) * 8;
  size_t s = 0;
  if (d.relative) s += sizeof(uint32_t) * DK8 * (size_t)(table_pitch(d.RW) + table_pitch(d.RH));
  s += sizeof(float) * (2 * TR * d.dkh + ((TR * d.dvh + 3) & ~3) + 4);
  s += sizeof(bf16) * 2 * TR * (size_t)(a.KP + 8);
  s += sizeof(int) * 2 * TR + 16;
  return s;
}

int aug_build_fwd(const Dims& d, const float* q, const float* k, const float* v, const float* krw, const float* krh,
                  void* qa, void* ka, cudaStream_t st) {
  AACONV_TRY(aug_supported(d));
  if (aug_build_tc_supported(d) == 0) return aug_build_tc(d, q, k, v, krw, krh, qa, ka, st);
  const AugLayout a = aug_layout(d);
  BuildP p;
  p.q = q; p.k = k; p.v = v; p.krw = krw; p.krh = krh;
  p.qa = static_cast<bf16*>(qa); p.ka = static_cast<bf16*>(ka);
  p.L = d.L; p.H = d.H; p.W = d.W; p.dkh = d.dkh; p.dvh = d.dvh; p.KD = a.KD; p.C1 = a.C1; p.KP = a.KP;
  p.relative = d.relative;
  p.DK8 = cdiv(d.dkh, 8) * 8; p.RW = d.RW; p.RH = d.RH; p.PBW = table_pitch(d.RW); p.PBH = table_pitch(d.RH);
  p.tiles_per_bn = cdiv(d.L, TR); p.ntiles = p.tiles_per_bn * d.BN;
  const size_t smem = aug_build_smem(d);
  if (smem > 200 * 1024) return fail(AACONV_E_UNSUPPORTED, "aug_build: %zu B of shared memory needed", smem);
  AACONV_CUDA_OK(cudaFuncSetAttribute(aug_build_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int per_sm = std::max(1, std::min(4, (int)(220 * 1024 / (smem + 1024))));
  const int grid = std::min(p.ntiles, 148 * per_sm);
  aug_build_fwd_kernel<<<grid, 256, smem, AACONV_ST(st)>>>(p);
  AACONV_LAUNCH_OK("aug_build_fwd");
  return 0;
}


// ------------------------------------------------------------------------------------------------
// attention map of the visualise path (opt-in; attn_aug_conv.py:87) from the bf16 kernels' OWN operands and statistics:
//   P[q, k] = 2^( Qa[q, 0:KD] . Ka[k, 0:KD]  -  log2(e) * lse[q] )
// Qa / Ka are the bf16 augmented operands the tcgen05 score MMAs consumed (log2(e) is folded into Qa), lse is what the
// bf16 forward kernel's online softmax produced; the dot product is accumulated in fp32 like the tensor core does.  Not a
// hot path (the map is (B, nh, L, L) fp32 and only the visualise path asks for it): plain shared-memory tiles, FFMA.
// ------------------------------------------------------------------------------------------------
namespace {
constexpr int AW_T = 64, AW_KMAX = 160;
__global__ void __launch_bounds__(256) aug_weights_kernel(const bf16* __restrict__ qa, const bf16* __restrict__ ka,
                                                          const float* __restrict__ lse, float* __restrict__ w, int L, int KD, int KP) {
  __shared__ __align__(16) bf16 qs[AW_T][AW_KMAX + 8];
  __shared__ __align__(16) bf16 ks[AW_T][AW_KMAX + 8];
  const int bn = blockIdx.z, q0 = blockIdx.y * AW_T, k0 = blockIdx.x * AW_T;
  const int KD2 = (KD + 1) & ~1;
  const size_t base = (size_t)bn * L;
  for (int i = threadIdx.x; i < AW_T * (KD2 / 2); i += 256) {
    const int r = i / (KD2 / 2), c = (i - r * (KD2 / 2)) * 2;
    uint32_t vq = 0, vk = 0;
    if (q0 + r < L) vq = *reinterpret_cast<const uint32_t*>(qa + (base + q0 + r) * KP + c);
    if (k0 + r < L) vk = *reinterpret_cast<const uint32_t*>(ka + (base + k0 + r) * KP + c);
    if (c + 1 >= KD) { vq &= 0xffffu; vk &= 0xffffu; }      // odd KD: column KD belongs to the statistics block
    *reinterpret_cast<uint32_t*>(&qs[r][c]) = vq;
    *reinterpret_cast<uint32_t*>(&ks[r][c]) = vk;
  }
  __syncthreads();
  const int ty = threadIdx.x >> 4, tx = threadIdx.x & 15;     // 16 x 16 threads, 4 x 4 outputs each (rows ty + 16 i, cols tx + 16 j)
  float acc[4][4] = {};
  for (int c = 0; c < KD2; c += 2) {
    float2 a[4], b[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) a[i] = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&qs[ty + 16 * i][c]));
#pragma unroll
    for (int j = 0; j < 4; ++j) b[j] = __bfloat1622float2(*reinterpret_cast<const __nv_bfloat162*>(&ks[tx + 16 * j][c]));
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i].y, b[j].y, fmaf(a[i].x, b[j].x, acc[i][j]));
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int q = q0 + ty + 16 * i;
    if (q >= L) continue;
    const float l2 = lse[base + q] * 1.4426950408889634f;
    float* row = w + (base + q) * (size_t)L;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int k = k0 + tx + 16 * j;
      if (k < L) row[k] = exp2f(acc[i][j] - l2);
    }
  }
}
}  // namespace

int aug_weights(const Dims& d, const void* qa, const void* ka, const float* lse, float* weights, cudaStream_t st) {
  const AugLayout a = aug_layout(d);
  if (a.KD > AW_KMAX) return fail(AACONV_E_UNSUPPORTED, "aug_weights: %d logit columns > %d", a.KD, AW_KMAX);
  dim3 grid(cdiv(d.L, AW_T), cdiv(d.L, AW_T), d.BN);
  aug_weights_kernel<<<grid, 256, 0, AACONV_ST(st)>>>(static_cast<const bf16*>(qa), static_cast<const bf16*>(ka), lse, weights, d.L, a.KD,
                                                      a.KP);
  AACONV_LAUNCH_OK("aug_weights_bf16");
  return 0;
}

int out_bwd_data_patch(const Dims& d, const float* dy, const float* o, const float* lse, const float* wout, float* d_o, float* delta,
                       void* qa, cudaStream_t st) {
  if (d.dvh > 14 || d.nh > 8) return fail(AACONV_E_UNSUPPORTED, "out_bwd_data_patch: dv/nh <= 14, nh <= 8");
  const AugLayout a = aug_layout(d);
  const size_t smem = sizeof(float) * ((size_t)d.dv * d.dv + (size_t)d.dv * 33);
  if (smem > 48 * 1024) AACONV_CUDA_OK(cudaFuncSetAttribute(out_bwd_data_patch_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  out_bwd_data_patch_kernel<<<cdiv(d.B * d.L, 32), 32 * d.nh, smem, AACONV_ST(st)>>>(dy, o, lse, wout, d_o, delta, static_cast<bf16*>(qa), d.B, d.L,
                                                                            d.nh, d.dvh, d.Cout, d.Cc, a.KD, a.C1, a.KP);
  AACONV_LAUNCH_OK("out_bwd_data_patch");
  return 0;
}

int out_proj_fwd(const Dims& d, const float* o, const float* wout, void* y, cudaStream_t st) {
  const size_t n = (size_t)d.B * d.L * d.dv, smem = sizeof(float) * d.dv * d.dv;
  if (smem > 48 * 1024) AACONV_CUDA_OK(cudaFuncSetAttribute(out_proj_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  out_proj_fwd_kernel<<<(unsigned)((n + 255) / 256), 256, smem, AACONV_ST(st)>>>(o, wout, y, d.B * d.L, d.L, d.nh, d.dvh, d.Cc, d.y_bs, d.y_bf16);
  AACONV_LAUNCH_OK("out_proj_fwd");
  return 0;
}

int out_bwd_patch_supported(const Dims& d) { return (d.nh == 8 && (d.dvh == 1 || d.dvh == 2)) ? 0 : AACONV_E_UNSUPPORTED; }
size_t out_bwd_patch_partial_floats(const Dims& d) { return (size_t)cdiv(d.B * d.L, OBP_THREADS) * d.dv * d.dv; }

int out_bwd_patch(const Dims& d, const float* dy, const float* o, const float* lse, const float* wout, float* d_o, float* delta,
                  void* qa, float* dw, float* partial, cudaStream_t st) {
  if (out_bwd_patch_supported(d)) return fail(AACONV_E_UNSUPPORTED, "out_bwd_patch: nh = 8, dv/nh <= 2 only");
  const AugLayout a = aug_layout(d);
  const int grid = cdiv(d.B * d.L, OBP_THREADS);
  float* wp = dw ? partial : nullptr;
  if (d.dvh == 1)
    out_bwd_patch_kernel<8, 1><<<grid, OBP_THREADS, 0, AACONV_ST(st)>>>(dy, o, lse, wout, d_o, delta, static_cast<bf16*>(qa), wp, d.B, d.L, d.Cout, d.Cc,
                                                     a.KD, a.C1, a.KP);
  else
    out_bwd_patch_kernel<8, 2><<<grid, OBP_THREADS, 0, AACONV_ST(st)>>>(dy, o, lse, wout, d_o, delta, static_cast<bf16*>(qa), wp, d.B, d.L, d.Cout, d.Cc,
                                                     a.KD, a.C1, a.KP);
  AACONV_LAUNCH_OK("out_bwd_patch");
  if (dw) {
    out_w_reduce_kernel<<<cdiv(d.dv * d.dv, 32), 256, 0, AACONV_ST(st)>>>(partial, grid, d.dv * d.dv, dw);
    AACONV_LAUNCH_OK("out_w_reduce");
  }
  return 0;
}

}  // namespace aaconv

// ================================================================================================
// rel_bwd: dQa -> dq (content + relative) and the key_rel_w / key_rel_h gradients
// ================================================================================================
namespace aaconv {
namespace {

struct RelBwdP {
  const float *dqa, *q, *krw, *krh;
  float* dq;            // fp32 (B,nh,L,dkh) or NULL
  bf16* dqkvh;          // packed bf16 (B*L, KPq) or NULL: dq * qscale lands at column n*dkh + e
  float* partial;       // [grid][2][RP * DK8] key_rel gradient partials (transposed: [r][e])
  int L, H, W, nh, dkh, KD, KPq, relative;
  int DK8, RW, RH, PBW, PBH, PTW, PTH, PA, RP;
  int tiles_per_bn, ntiles, tile_floats;
  int pipelined;        // every tile can be fetched by bulk copies: tile i+1 is loaded while tile i is computed (two buffers)
  float qscale;
};


inline int pitch_mod32(int n, int want) {
  int p = n;
  while (p % 32 != want) ++p;
  return p;
}

// MT = 16-row tiles of the relative axis (2N-1 <= 16*MT), NTE = 8-column tiles of dkh (dkh <= 8*NTE)
template <int MT, int NTE>
__global__ void __launch_bounds__(256, (MT <= 5 ? 2 : 1)) rel_bwd_kernel(const RelBwdP p) {
  extern __shared__ __align__(16) uint8_t smem_raw[];
  uint32_t* tabw = reinterpret_cast<uint32_t*>(smem_raw);        // [DK8][PTW]  pitch == 4 (mod 32): B frags with n = e = g, k = r = t
  uint32_t* tabh = tabw + p.DK8 * p.PTW;                         // [DK8][PTH]
  // q and dQa tiles are contiguous copies of the global rows (one bulk copy each).  K/N padding of the q fragments
  // (columns dkh..8*NTE) reads the next row / the head of da: it only feeds output columns that are discarded.
  const int QF = (TR * p.dkh + 3) & ~3, BUF = QF + p.tile_floats;   // one buffer = q tile + dQa tile
  float* const buf0 = reinterpret_cast<float*>(tabh + p.DK8 * p.PTH);
  float* qs = buf0;                                              // [TR][dkh]   q
  float* da = qs + QF;                                           // [TR][PA]    dQa rows of the tile (PA == KD)
  const int PQ2 = p.dkh;
  const int nbuf = p.pipelined ? 2 : 1;
  uint64_t* bar = reinterpret_cast<uint64_t*>(buf0 + nbuf * BUF);   // one barrier per buffer
  if (threadIdx.x == 0) { tc::mbar_init(&bar[0], 1); tc::mbar_init(&bar[1], 1); tc::fence_barrier_init(); }
  uint32_t phase = 0;                                            // bit b = phase of buffer b
  auto fetch = [&](int tile, int b) {                            // thread 0: bulk copies of one tile into buffer b
    const int bn = tile / p.tiles_per_bn, l0 = (tile - bn * p.tiles_per_bn) * TR;
    const int nrows = min(TR, p.L - l0);
    const size_t row0 = (size_t)bn * p.L + l0;
    const uint32_t bq = nrows * p.dkh * 4, bd = nrows * p.KD * 4;
    tc::mbar_arrive_expect_tx(&bar[b], bq + bd);
    bulk_g2s(buf0 + b * BUF, p.q + row0 * p.dkh, bq, &bar[b]);
    bulk_g2s(buf0 + b * BUF + QF, p.dqa + row0 * p.KD, bd, &bar[b]);
  };
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;

  for (int i = threadIdx.x; i < p.DK8 * p.PTW; i += blockDim.x) {
    const int e = i / p.PTW, r = i - e * p.PTW;
    tabw[i] = (e < p.dkh && r < p.RW) ? f2tf32(p.krw[e * p.RW + r]) : 0u;
  }
  for (int i = threadIdx.x; i < p.DK8 * p.PTH; i += blockDim.x) {
    const int e = i / p.PTH, r = i - e * p.PTH;
    tabh[i] = (e < p.dkh && r < p.RH) ? f2tf32(p.krh[e * p.RH + r]) : 0u;
  }
  for (int i = threadIdx.x; i < nbuf * BUF; i += blockDim.x) buf0[i] = 0.f;
  float acc[MT][NTE][4];                                         // G role: dT^T[r][e] of this warp's axis / row half
#pragma unroll
  for (int a = 0; a < MT; ++a)
#pragma unroll
    for (int b = 0; b < NTE; ++b)
#pragma unroll
      for (int c = 0; c < 4; ++c) acc[a][b][c] = 0.f;

  __syncthreads();                                     // zero-fill and barrier init before the first copy
  if (p.pipelined && threadIdx.x == 0 && (int)blockIdx.x < p.ntiles) { tc::fence_proxy_async(); fetch(blockIdx.x, 0); }
  int cur = 0;
  for (int tile = blockIdx.x; tile < p.ntiles; tile += gridDim.x, cur ^= p.pipelined) {
    const int bn = tile / p.tiles_per_bn, l0 = (tile - bn * p.tiles_per_bn) * TR;
    const int nrows = min(TR, p.L - l0);
    const size_t row0 = (size_t)bn * p.L + l0;
    qs = buf0 + cur * BUF;
    da = qs + QF;
    __syncthreads();                                   // everyone is done with the other buffer (tile - gridDim.x)
    if (nrows < TR) {                                  // last tile of an image: rows past the end must contribute zero
      for (int i = threadIdx.x + nrows * p.dkh; i < TR * p.dkh; i += blockDim.x) qs[i] = 0.f;
      for (int i = threadIdx.x + nrows * p.PA; i < TR * p.PA; i += blockDim.x) da[i] = 0.f;
    }
    const bool bulk = p.PA == p.KD && (((row0 * p.dkh) | (size_t)(nrows * p.dkh) | (row0 * p.KD) | (size_t)(nrows * p.KD)) & 3) == 0;
    if (p.pipelined) {
      if (threadIdx.x == 0 && tile + (int)gridDim.x < p.ntiles) { tc::fence_proxy_async(); fetch(tile + gridDim.x, cur ^ 1); }
      tc::mbar_wait(&bar[cur], (phase >> cur) & 1);
      phase ^= 1u << cur;
    } else if (bulk) {
      if (threadIdx.x == 0) {
        const uint32_t bq = nrows * p.dkh * 4, bd = nrows * p.KD * 4;
        tc::mbar_arrive_expect_tx(&bar[0], bq + bd);
        bulk_g2s(qs, p.q + row0 * p.dkh, bq, &bar[0]);
        bulk_g2s(da, p.dqa + row0 * p.KD, bd, &bar[0]);
      }
      tc::mbar_wait(&bar[0], phase & 1);
      phase ^= 1;
    } else {
      for (int r = warp; r < nrows; r += 8) {
        for (int c = lane; c < p.KD; c += 32) cp_async4(da + r * p.PA + c, p.dqa + (row0 + r) * p.KD + c);
        if (lane < p.dkh) cp_async4(qs + r * PQ2 + lane, p.q + (row0 + r) * p.dkh + lane);
      }
      cp_async_wait_all();
    }
    __syncthreads();

    if (warp < 4) {
      // ---------------- dq role: 16 rows, both axes ----------------
      const int ra = warp * 16 + g, rb = ra + 8;
      const int la = l0 + ra, lb = l0 + rb;
      float c[NTE][4];
#pragma unroll
      for (int nt = 0; nt < NTE; ++nt) { c[nt][0] = c[nt][1] = c[nt][2] = c[nt][3] = 0.f; }
      for (int axis = 0; axis < 2; ++axis) {
        const int N = axis ? p.H : p.W, R = axis ? p.RH : p.RW, PT = axis ? p.PTH : p.PTW;
        const uint32_t* tab = axis ? tabh : tabw;
        const int colbase = p.dkh + (axis ? p.W : 0);
        const int pos_a = axis ? la / p.W : la % p.W, pos_b = axis ? lb / p.W : lb % p.W;
        const float* rowa = da + ra * p.PA + colbase + pos_a - (N - 1);
        const float* rowb = da + rb * p.PA + colbase + pos_b - (N - 1);
        const int lo_a = N - 1 - pos_a, lo_b = N - 1 - pos_b;   // valid r: lo <= r < lo + N
        const int KS = (R + 7) >> 3;
        for (int ks = 0; ks < KS; ++ks) {
          const int r0 = 8 * ks + t, r1 = r0 + 4;
          const uint32_t a0 = (unsigned)(r0 - lo_a) < (unsigned)N ? f2tf32_alu(rowa[r0]) : 0u;
          const uint32_t a1 = (unsigned)(r0 - lo_b) < (unsigned)N ? f2tf32_alu(rowb[r0]) : 0u;
          const uint32_t a2 = (unsigned)(r1 - lo_a) < (unsigned)N ? f2tf32_alu(rowa[r1]) : 0u;
          const uint32_t a3 = (unsigned)(r1 - lo_b) < (unsigned)N ? f2tf32_alu(rowb[r1]) : 0u;
#pragma unroll
          for (int nt = 0; nt < NTE; ++nt)
            mma_tf32(c[nt], a0, a1, a2, a3, tab[(8 * nt + g) * PT + r0], tab[(8 * nt + g) * PT + r1]);
        }
      }
      const int b = bn / p.nh, n = bn - b * p.nh;
#pragma unroll
      for (int nt = 0; nt < NTE; ++nt)
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const int r = h ? rb : ra, e = 8 * nt + 2 * t;
          if (r < nrows && e < p.dkh) {
            const float v0 = c[nt][2 * h] + da[r * p.PA + e];
            const float v1 = (e + 1 < p.dkh) ? c[nt][2 * h + 1] + da[r * p.PA + e + 1] : 0.f;
            if (p.dq) {
              p.dq[(row0 + r) * p.dkh + e] = v0;
              if (e + 1 < p.dkh) p.dq[(row0 + r) * p.dkh + e + 1] = v1;
            }
            if (p.dqkvh) {
              bf16* dst = p.dqkvh + ((size_t)b * p.L + l0 + r) * p.KPq + n * p.dkh + e;
              if (((p.dkh | p.KPq) & 1) == 0) {              // e is even: 4-byte aligned pair
                *reinterpret_cast<__nv_bfloat162*>(dst) = __floats2bfloat162_rn(v0 * p.qscale, v1 * p.qscale);
              } else {
                dst[0] = __float2bfloat16(v0 * p.qscale);
                if (e + 1 < p.dkh) dst[1] = __float2bfloat16(v1 * p.qscale);
              }
            }
          }
        }
    } else {
      // ---------------- G role: one axis, 32 rows ----------------
      const int axis = (warp - 4) >> 1, rh = ((warp - 4) & 1) * 32;
      const int N = axis ? p.H : p.W, R = axis ? p.RH : p.RW;
      const int colbase = p.dkh + (axis ? p.W : 0);
#pragma unroll
      for (int ks = 0; ks < 4; ++ks) {
        const int k0 = rh + 8 * ks + t, k1 = k0 + 4;
        const int l_0 = l0 + k0, l_1 = l0 + k1;
        const int pos0 = axis ? l_0 / p.W : l_0 % p.W, pos1 = axis ? l_1 / p.W : l_1 % p.W;
        const float* row0p = da + k0 * p.PA + colbase + pos0 - (N - 1);
        const float* row1p = da + k1 * p.PA + colbase + pos1 - (N - 1);
        const int lo0 = N - 1 - pos0, lo1 = N - 1 - pos1;
        uint32_t b0[NTE], b1[NTE];
#pragma unroll
        for (int nt = 0; nt < NTE; ++nt) {
          b0[nt] = f2tf32_alu(qs[k0 * PQ2 + 8 * nt + g]);
          b1[nt] = f2tf32_alu(qs[k1 * PQ2 + 8 * nt + g]);
        }
#pragma unroll
        for (int mt = 0; mt < MT; ++mt) {
          const int r_a = 16 * mt + g, r_b = r_a + 8;
          if (16 * mt < R) {
            const uint32_t a0 = (unsigned)(r_a - lo0) < (unsigned)N ? f2tf32_alu(row0p[r_a]) : 0u;
            const uint32_t a1 = (unsigned)(r_b - lo0) < (unsigned)N ? f2tf32_alu(row0p[r_b]) : 0u;
            const uint32_t a2 = (unsigned)(r_a - lo1) < (unsigned)N ? f2tf32_alu(row1p[r_a]) : 0u;
            const uint32_t a3 = (unsigned)(r_b - lo1) < (unsigned)N ? f2tf32_alu(row1p[r_b]) : 0u;
#pragma unroll
            for (int nt = 0; nt < NTE; ++nt) mma_tf32(acc[mt][nt], a0, a1, a2, a3, b0[nt], b1[nt]);
          }
        }
      }
    }
  }
  // ---- CTA partial of the key_rel gradients: sum the two row-half warps of each axis in a fixed order ----
  __syncthreads();
  float* red = buf0 + QF;                            // [4 warps][RP * DK8]: aliases buffer 0's dQa tile (sized for it on the host)
  if (warp >= 4) {
    float* mine = red + (warp - 4) * p.RP * p.DK8;
#pragma unroll
    for (int mt = 0; mt < MT; ++mt)
#pragma unroll
      for (int nt = 0; nt < NTE; ++nt) {
        const int r = 16 * mt + g, e = 8 * nt + 2 * t;
        if (r < p.RP && e < p.DK8) {
          mine[r * p.DK8 + e] = acc[mt][nt][0];
          mine[r * p.DK8 + e + 1] = acc[mt][nt][1];
        }
        if (r + 8 < p.RP && e < p.DK8) {
          mine[(r + 8) * p.DK8 + e] = acc[mt][nt][2];
          mine[(r + 8) * p.DK8 + e + 1] = acc[mt][nt][3];
        }
      }
  }
  __syncthreads();
  const int per_axis = p.RP * p.DK8;
  float* out = p.partial + (size_t)blockIdx.x * 2 * per_axis;
  for (int i = threadIdx.x; i < 2 * per_axis; i += blockDim.x) {
    const int axis = i / per_axis, j = i - axis * per_axis;
    out[i] = red[(2 * axis) * per_axis + j] + red[(2 * axis + 1) * per_axis + j];
  }
}

// dkr[e, r] = sum over CTAs of partial[cta][axis][r][e]   (fixed order: deterministic).  Block = 32 outputs x 8 slices of parts.
__global__ void __launch_bounds__(256) rel_bwd_reduce_kernel(const float* __restrict__ partial, int nparts, int RP, int DK8,
                                                             int dkh, int RW, int RH, float* __restrict__ dkrw,
                                                             float* __restrict__ dkrh) {
  __shared__ float red[8][33];
  const int o = threadIdx.x & 31, sl = threadIdx.x >> 5;
  const int i = blockIdx.x * 32 + o;
  const int per_axis = RP * DK8;
  float s = 0.f;
  if (i < 2 * per_axis) {
    const float* src = partial + i;
    const size_t step = (size_t)2 * per_axis;
    int c = sl;
    for (; c + 24 < nparts; c += 32) {               // four loads in flight per add chain; order fixed
      const float a = src[(size_t)c * step], b = src[(size_t)(c + 8) * step], d = src[(size_t)(c + 16) * step],
                  e = src[(size_t)(c + 24) * step];
      s = (((s + a) + b) + d) + e;
    }
    for (; c < nparts; c += 8) s += src[(size_t)c * step];
  }
  red[sl][o] = s;
  __syncthreads();
  if (sl == 0 && i < 2 * per_axis) {
    float tot = 0.f;
#pragma unroll
    for (int k = 0; k < 8; ++k) tot += red[k][o];
    const int axis = i / per_axis, j = i - axis * per_axis, r = j / DK8, e = j - r * DK8;
    float* dst = axis ? dkrh : dkrw;
    const int R = axis ? RH : RW;
    if (dst && r < R && e < dkh) dst[e * R + r] = tot;
  }
}

template <int MT, int NTE>
int launch_rel_bwd(const RelBwdP& p, int grid, size_t smem, cudaStream_t st) {
  auto kern = rel_bwd_kernel<MT, NTE>;
  AACONV_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, 256, smem, AACONV_ST(st)>>>(p);
  AACONV_LAUNCH_OK("rel_bwd");
  return 0;
}

template <int NTE>
int dispatch_rel_bwd(int mt, const RelBwdP& p, int grid, size_t smem, cudaStream_t st) {
  if (mt <= 1) return launch_rel_bwd<1, NTE>(p, grid, smem, st);
  if (mt <= 2) return launch_rel_bwd<2, NTE>(p, grid, smem, st);
  if (mt <= 3) return launch_rel_bwd<3, NTE>(p, grid, smem, st);
  if (mt <= 5) return launch_rel_bwd<5, NTE>(p, grid, smem, st);
  return launch_rel_bwd<8, NTE>(p, grid, smem, st);
}

constexpr int REL_BWD_GRID = 148 * 2;

}  // namespace

int rel_bwd_reduce(const Dims& d, const float* partial, int nparts, int RP, int DK8, float* dkrw, float* dkrh, cudaStream_t st) {
  const int n = 2 * RP * DK8;
  rel_bwd_reduce_kernel<<<cdiv(n, 32), 256, 0, AACONV_ST(st)>>>(partial, nparts, RP, DK8, d.dkh, d.RW, d.RH, dkrw, dkrh);
  AACONV_LAUNCH_OK("rel_bwd_reduce");
  return 0;
}

int rel_bwd_supported(const Dims& d) {
  if (!d.relative) return AACONV_E_UNSUPPORTED;
  if (std::max(d.RW, d.RH) > 128 || d.dkh > 32) return AACONV_E_UNSUPPORTED;
  return 0;
}

size_t rel_bwd_partial_floats(const Dims& d) {
  if (rel_bwd_supported(d)) return 0;
  const int RP = cdiv(std::max(d.RW, d.RH), 16) * 16, DK8 = cdiv(d.dkh, 8) * 8;
  return (size_t)REL_BWD_GRID * 2 * RP * DK8;
}

// dqa (B,nh,L,KD) fp32, q (B,nh,L,dkh) fp32 (scaled q).  Writes dq (fp32, optional), dqkvh (bf16 packed, optional),
// and the key_rel gradients (optional).
int rel_bwd(const Dims& d, const float* dqa, const float* q, const float* krw, const float* krh, float* dq, void* dqkvh,
            int KPq, float* dkrw, float* dkrh, float* partial, cudaStream_t st) {
  AACONV_TRY(rel_bwd_supported(d));
  if (!dq && dqkvh && rel_bwd_tc_supported(d, KPq) == 0) {
    const int RP = cdiv(std::max(d.RW, d.RH), 16) * 16, DK8 = cdiv(d.dkh, 8) * 8;
    int nparts = 0;
    AACONV_TRY(rel_bwd_tc(d, dqa, q, krw, krh, dqkvh, KPq, partial, RP, DK8, &nparts, st));
    if (dkrw || dkrh) AACONV_TRY(rel_bwd_reduce(d, partial, nparts, RP, DK8, dkrw, dkrh, st));
    return 0;
  }
  const AugLayout a = aug_layout(d);
  RelBwdP p;
  p.dqa = dqa; p.q = q; p.krw = krw; p.krh = krh; p.dq = dq; p.dqkvh = static_cast<bf16*>(dqkvh); p.partial = partial;
  p.L = d.L; p.H = d.H; p.W = d.W; p.nh = d.nh; p.dkh = d.dkh; p.KD = a.KD; p.KPq = KPq; p.relative = d.relative;
  p.DK8 = cdiv(d.dkh, 8) * 8; p.RW = d.RW; p.RH = d.RH;
  p.PBW = p.PBH = 0;
  p.PTW = pitch_mod32(cdiv(d.RW, 8) * 8, 4); p.PTH = pitch_mod32(cdiv(d.RH, 8) * 8, 4);
  p.PA = a.KD;                                                       // contiguous rows: one bulk copy per tile
  p.RP = cdiv(std::max(d.RW, d.RH), 16) * 16;
  p.tiles_per_bn = cdiv(d.L, TR); p.ntiles = p.tiles_per_bn * d.BN;
  p.qscale = d.qscale;
  const int mt = p.RP / 16, nte = p.DK8 / 8;
  size_t tile_floats = (size_t)TR * p.PA;
  tile_floats = (std::max(tile_floats, (size_t)4 * p.RP * p.DK8) + 3) & ~size_t(3);       // the reduction buffer aliases the dQa tile
  p.tile_floats = (int)tile_floats;
  // bulk copies need 16-byte aligned, 16-byte multiple row blocks for EVERY tile: then the next tile is prefetched
  p.pipelined = (p.PA == p.KD && ((d.L * d.dkh) % 4) == 0 && ((d.L * a.KD) % 4) == 0 && ((TR * d.dkh) % 4) == 0 && ((TR * a.KD) % 4) == 0 &&
                 ((std::min(TR, d.L - (p.tiles_per_bn - 1) * TR) * d.dkh) % 4) == 0 &&
                 ((std::min(TR, d.L - (p.tiles_per_bn - 1) * TR) * a.KD) % 4) == 0) ? 1 : 0;
  const size_t one_buf = sizeof(float) * (((TR * d.dkh + 3) & ~3) + tile_floats);
  size_t smem = sizeof(uint32_t) * p.DK8 * (size_t)(p.PTW + p.PTH) + (p.pipelined ? 2 : 1) * one_buf + 32;
  if (p.pipelined && smem > 100 * 1024) {              // keep two CTAs per SM
    p.pipelined = 0;
    smem -= one_buf;
  }
  if (smem > 200 * 1024) return fail(AACONV_E_UNSUPPORTED, "rel_bwd: %zu B of shared memory needed", smem);
  const int grid = std::min(p.ntiles, REL_BWD_GRID);
  if (nte <= 3) AACONV_TRY(dispatch_rel_bwd<3>(mt, p, grid, smem, st));
  else AACONV_TRY(dispatch_rel_bwd<4>(mt, p, grid, smem, st));
  if (dkrw || dkrh) {
    const int n = 2 * p.RP * p.DK8;
    rel_bwd_reduce_kernel<<<cdiv(n, 32), 256, 0, AACONV_ST(st)>>>(partial, grid, p.RP, p.DK8, d.dkh, d.RW, d.RH, dkrw, dkrh);
    AACONV_LAUNCH_OK("rel_bwd_reduce");
  }
  return 0;
}

}  // namespace aaconv
