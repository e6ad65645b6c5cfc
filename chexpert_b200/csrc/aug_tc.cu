// tcgen05 builder of the augmented attention operands Qa / Ka (layout: attn_tc_bwd.cu header) -- round-2 replacement of
// aug_build_fwd_kernel (mma.sync TF32 + predicated fragment scatter, instruction bound at ~150 thread instructions per 16 B).
//
//   R_w[row, r] = c * sum_e q[row,e] key_rel_w[e, r]      (128 x NW tile, kind::tf32, A = q tile via TMA, B = table in smem)
//   Aq[row, x'] = R_w[row, x' + (W-1 - x(row))]            rel_to_abs as an index computation (attn_aug_conv.py:43-63)
//
// One thread owns one row (= one TMEM lane): it pulls its R row out of TMEM, parks it in a private shared-memory row and
// reads the W-wide window back at its own offset (the "skew" of rel_to_abs is a per-row constant), packs the bf16 row in
// registers with a compile-time column map and writes 16-byte chunks into a 128B-swizzled staging tile that leaves through
// TMA tensor stores.  Persistent CTAs: TMA warp (q tiles), MMA warp (two TMEM accumulator buffers), one or two epilogue warpgroups.
// Reference rows a4-a6 (attn_aug_conv.py:55-63,77-86).
#include <algorithm>
#include "tc_common.cuh"
#include "bf16_path.cuh"

namespace aaconv {

using tc::smem_u32;
typedef __nv_bfloat16 bf16;

int make_tmap_f32(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                  const uint32_t* box);

namespace {

constexpr float LOG2E = 1.4426950408889634f;
constexpr int AB_BM = 128;

__host__ __device__ constexpr int ru16(int n) { return (n + 15) / 16 * 16; }
__host__ __device__ constexpr uint32_t idesc_tf32_f32(int M, int N) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ void mma_ss_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}\n"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* m, const void* src, int c0, int c1, int c2) {
  asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];"
               ::"l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait0() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void sts128(uint32_t saddr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(saddr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ float4 lds128f(uint32_t saddr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t lds32u(uint32_t saddr) {
  uint32_t v;
  asm volatile("ld.shared.b32 %0, [%1];" : "=r"(v) : "r"(saddr) : "memory");
  return v;
}
__device__ __forceinline__ uint32_t pk(uint32_t lo, uint32_t hi) { return tc::pack_bf16x2(__uint_as_float(lo), __uint_as_float(hi)); }
__device__ __forceinline__ float lds32f(uint32_t saddr) {
  float v;
  asm volatile("ld.shared.f32 %0, [%1];" : "=f"(v) : "r"(saddr) : "memory");
  return v;
}

template <int W, int H, int DKH>
struct AbCfg {
  static constexpr int NW = ru16(2 * W - 1), NH = ru16(2 * H - 1);
  static constexpr int NMAX = NW > NH ? NW : NH;
  static constexpr int PITCH = 2 * NMAX + 16;             // bytes of a private bf16 row; PITCH / 16 odd: conflict-free 16 B row-strided stores
  static constexpr int KD = DKH + W + H, C1 = ru16(KD + 2), KP = (C1 + 16 + 63) / 64 * 64, KATOMS = KP / 64;
  static constexpr int TCOLS = NW + NH;                   // accumulator columns per buffer
  static constexpr int TALLOC = 2 * TCOLS <= 32 ? 32 : 2 * TCOLS <= 64 ? 64 : 2 * TCOLS <= 128 ? 128 : 2 * TCOLS <= 256 ? 256 : 512;
  static constexpr int KSTEPS = (DKH + 7) / 8;            // tf32: K = 8 per MMA
  // Epilogue warpgroups: two (tile i -> warpgroup i % 2, each with its own TMEM buffer, skew rows and staging tile) when the
  // shared memory allows it.  Measured (B200, T1, B = 16): one warpgroup = one warp per scheduler ran the per-tile chain
  // TMEM -> skew rows -> window -> pack -> staging -> TMA store with every latency exposed (39.6 us; 2 or 6 q stages alike).
  static constexpr int per_wg = AB_BM * PITCH + KATOMS * AB_BM * 128;       // skew rows + one staging tile (Qa, then Ka)
  static constexpr int tables = (NW + NH) * 128;
  static constexpr int NWG = tables + 2 * per_wg + 2 * AB_BM * 128 + 2048 <= 225 * 1024 ? 2 : 1;
  static constexpr int fit = (225 * 1024 - tables - NWG * per_wg - 2048) / (AB_BM * 128);
  static constexpr int STAGES = fit > 4 ? 4 : fit;        // q stages (16 KB each)
  static constexpr int THREADS = 32 * (4 * NWG + 2);      // epilogue warps, TMA producer, MMA issuer (+ TMEM alloc)
  static_assert(DKH <= 32 && DKH % 4 == 0, "q rows must be 16-byte multiples and fit one 128-byte atom");
  static_assert((W % 2 == 0) && (H % 2 == 0) && (DKH % 2 == 0), "bf16 pairs must not straddle column blocks");
  static_assert(2 * TCOLS <= 512 && STAGES >= 2, "does not fit");
};

template <class C>
struct __align__(1024) AbSmem {
  float q[C::STAGES][AB_BM * 32];                 // q tile, 128 B rows (32 fp32, dkh valid), 128B swizzle (TMA)
  float tw[C::NW * 32];                           // c * key_rel_w^T as a K-major B operand: row r = 32 fp32 (e), swizzled
  float th[C::NH * 32];
  bf16 stg[C::NWG][C::KATOMS][AB_BM * 64];        // staging tile of a warpgroup: Qa, then Ka (TMA store source)
  uint8_t skew[C::NWG][AB_BM * C::PITCH];         // private bf16 row of every epilogue thread
  uint64_t bar_full[C::STAGES], bar_empty[C::STAGES], bar_tfull[2], bar_tempty[2];
  uint32_t tmem_base;
};

template <int W, int H, int DKH>
__global__ void __launch_bounds__(AbCfg<W, H, DKH>::THREADS, 1) aug_build_tc_kernel(
    const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_qa, const __grid_constant__ CUtensorMap tm_ka,
    const float* __restrict__ kg, const float* __restrict__ vg, const float* __restrict__ krw, const float* __restrict__ krh,
    int L, int dvh, int tiles_per_bn, int ntiles, uint32_t dep_zero /* always 0: see tc::mbar_arrive_after */) {
  typedef AbCfg<W, H, DKH> C;
  typedef AbSmem<C> Smem;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int ST = C::STAGES, NWG = C::NWG, W_TMA = 4 * NWG, W_MMA = W_TMA + 1;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int my_tiles = (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (warp == W_TMA && lane == 0) {     // barrier set-up + the first q tiles before the CTA-wide sync (their latency runs under the table build)
    for (int s = 0; s < ST; ++s) { tc::mbar_init(&sm.bar_full[s], 1); tc::mbar_init(&sm.bar_empty[s], 128); }
    for (int s = 0; s < 2; ++s) { tc::mbar_init(&sm.bar_tfull[s], 1); tc::mbar_init(&sm.bar_tempty[s], 128); }
    tc::fence_barrier_init();
    for (int i = 0; i < ST && i < my_tiles; ++i) {
      const int tile = blockIdx.x + i * gridDim.x, bn = tile / tiles_per_bn, l0 = (tile - bn * tiles_per_bn) * AB_BM;
      tc::mbar_arrive_expect_tx(&sm.bar_full[i], AB_BM * 128);
      tc::tma_load_3d(sm.q[i], &tm_q, &sm.bar_full[i], 0, l0, bn);
    }
    tc::tma_prefetch_desc(&tm_qa);
    tc::tma_prefetch_desc(&tm_ka);
  }
  if (warp == W_MMA) tc::tmem_alloc<C::TALLOC>(&sm.tmem_base);
  // B operands: tables transposed, scaled by log2(e), rounded to TF32, in the 128B-swizzled K-major layout of a TMA tile.
  // Warps 0-3: zero fill first (most of the tile is K / N padding), then the dkh x (2N-1) values -- coalesced reads, all of a
  // thread's loads in flight at once (the prologue is one DRAM round trip, not one per loop iteration).
  if (warp < 4) {
    float4* z = reinterpret_cast<float4*>(sm.tw);                     // tw and th are adjacent
    for (int i = threadIdx.x; i < (C::NW + C::NH) * 8; i += 128) z[i] = make_float4(0.f, 0.f, 0.f, 0.f);
    constexpr int RW_ = 2 * W - 1, RH_ = 2 * H - 1, NTAB = DKH * (RW_ + RH_), PER = (NTAB + 127) / 128;
    float tv[PER];
#pragma unroll
    for (int u = 0; u < PER; ++u) {
      const int i = threadIdx.x + u * 128;
      tv[u] = i < NTAB ? __ldg((i >= DKH * RW_ ? krh - DKH * RW_ : krw) + i) : 0.f;
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");
#pragma unroll
    for (int u = 0; u < PER; ++u) {
      const int i = threadIdx.x + u * 128;
      if (i < NTAB) {
        const bool hax = i >= DKH * RW_;
        const int j = hax ? i - DKH * RW_ : i, R = hax ? RH_ : RW_;
        const int e = j / R, r = j - e * R;
        uint32_t t;
        asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(t) : "f"(LOG2E * tv[u]));
        (hax ? sm.th : sm.tw)[r * 32 + ((((e >> 2) ^ (r & 7)) << 2) | (e & 3))] = __uint_as_float(t);
      }
    }
  }
  tc::fence_proxy_async();           // generic-proxy writes of the tables -> visible to the tensor core's async-proxy reads
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = sm.tmem_base;

  if (warp == W_TMA) {
    // ===================== TMA producer: q tiles (the first ST were issued during set-up) =====================
    if (lane == 0) {
      for (int i = ST; i < my_tiles; ++i) {
        const int tile = blockIdx.x + i * gridDim.x, bn = tile / tiles_per_bn, l0 = (tile - bn * tiles_per_bn) * AB_BM;
        const int s = i % ST;
        tc::mbar_wait(&sm.bar_empty[s], ((i / ST) & 1) ^ 1);
        tc::mbar_arrive_expect_tx(&sm.bar_full[s], AB_BM * 128);
        tc::tma_load_3d(sm.q[s], &tm_q, &sm.bar_full[s], 0, l0, bn);
      }
    }
  } else if (warp == W_MMA) {
    // ===================== MMA issuer: R_w | R_h of tile i -> TMEM buffer i % 2 =====================
    constexpr uint32_t idw = idesc_tf32_f32(AB_BM, C::NW), idh = idesc_tf32_f32(AB_BM, C::NH);
    const uint32_t bw = tc::desc_lo_k(smem_u32(sm.tw)), bh = tc::desc_lo_k(smem_u32(sm.th));
    for (int i = 0; i < my_tiles; ++i) {
      const int buf = i & 1, s = i % ST;
      tc::mbar_wait(&sm.bar_full[s], (i / ST) & 1);
      if (i >= 2) tc::mbar_wait(&sm.bar_tempty[buf], ((i >> 1) & 1) ^ 1);
      tc::tc_fence_after();
      if (tc::elect_one()) {
        const uint32_t a = tc::desc_lo_k(smem_u32(sm.q[s]));
        const uint32_t d0 = tmem + buf * C::TCOLS;
#pragma unroll
        for (int ks = 0; ks < C::KSTEPS; ++ks) mma_ss_tf32(d0, tc::desc64(a + ks * 2), tc::desc64(bw + ks * 2), idw, ks > 0);
#pragma unroll
        for (int ks = 0; ks < C::KSTEPS; ++ks) mma_ss_tf32(d0 + C::NW, tc::desc64(a + ks * 2), tc::desc64(bh + ks * 2), idh, ks > 0);
        tc::mma_commit(&sm.bar_tfull[buf]);
      }
      __syncwarp();
    }
  } else {
    // ===================== epilogue warpgroups: thread == row == TMEM lane; tile i -> warpgroup i % NWG =====================
    const int wg = warp >> 2;
    const int r = threadIdx.x & 127;
    const bool leader = r == 0;
    const uint32_t tlane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const uint32_t skew = smem_u32(sm.skew[wg]) + r * C::PITCH;
    const uint32_t stg0 = smem_u32(sm.stg[wg][0]) + r * 128;
    const uint32_t swz = (uint32_t)(r & 7);
    auto wg_sync = [&]() { asm volatile("bar.sync %0, 128;" ::"r"(1 + wg) : "memory"); };
    for (int i = wg; i < my_tiles; i += NWG) {
      const int tile = blockIdx.x + i * gridDim.x, bn = tile / tiles_per_bn, l0 = (tile - bn * tiles_per_bn) * AB_BM;
      const int buf = i & 1, s = i % ST;
      const int l = min(l0 + r, L - 1);             // rows past L: clipped by the TMA store, indices kept in range
      const int y = l / W, x = l - y * W;
      const size_t grow = (size_t)bn * L + l;
      // this row's k and v (fp32, global): issued first, consumed last
      float kf[DKH];
#pragma unroll
      for (int e = 0; e < DKH; e += 4) {
        const float4 t4 = __ldg(reinterpret_cast<const float4*>(kg + grow * DKH + e));
        kf[e] = t4.x; kf[e + 1] = t4.y; kf[e + 2] = t4.z; kf[e + 3] = t4.w;
      }
      float vf[14];
#pragma unroll
      for (int e = 0; e < 14; ++e) vf[e] = e < dvh ? __ldg(vg + grow * dvh + e) : 0.f;

      tc::mbar_wait(&sm.bar_tfull[buf], (i >> 1) & 1);
      tc::tc_fence_after();
      uint32_t aq[W / 2], bq[H / 2];
      // ---- W axis: R_w row -> private shared row (bf16) -> window [W-1-x, 2W-1-x) ----
      {
        const uint32_t tcol = tlane + buf * C::TCOLS;
#pragma unroll
        for (int b0 = 0; b0 < C::NW; b0 += 64) {            // at most 64 columns in flight (registers)
          uint32_t v[64];
#pragma unroll
          for (int c0 = 0; c0 < 64; c0 += 16)
            if (b0 + c0 < C::NW) tc::tmem_ld_x16(tcol + b0 + c0, reinterpret_cast<uint32_t(&)[16]>(v[c0]));
          tc::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 64; j += 8)                  // rounded to bf16 here: the window read moves bits only
            if (b0 + j < C::NW)
              sts128(skew + (b0 + j) * 2, pk(v[j], v[j + 1]), pk(v[j + 2], v[j + 3]), pk(v[j + 4], v[j + 5]), pk(v[j + 6], v[j + 7]));
        }
        const int sh = W - 1 - x;                           // window = elements [sh, sh + W) of the row
        const uint32_t win = skew + (sh >> 1) * 4, fs = (uint32_t)(sh & 1) << 4;
        uint32_t wd[W / 2 + 1];
#pragma unroll
        for (int j = 0; j <= W / 2; ++j) wd[j] = lds32u(win + 4 * j);
#pragma unroll
        for (int j = 0; j < W / 2; ++j) aq[j] = __funnelshift_r(wd[j], wd[j + 1], fs);
      }
      // ---- H axis ----
      {
        const uint32_t tcol = tlane + buf * C::TCOLS + C::NW;
#pragma unroll
        for (int b0 = 0; b0 < C::NH; b0 += 64) {
          uint32_t v[64];
#pragma unroll
          for (int c0 = 0; c0 < 64; c0 += 16)
            if (b0 + c0 < C::NH) tc::tmem_ld_x16(tcol + b0 + c0, reinterpret_cast<uint32_t(&)[16]>(v[c0]));
          tc::tmem_ld_wait();
#pragma unroll
          for (int j = 0; j < 64; j += 8)
            if (b0 + j < C::NH)
              sts128(skew + (b0 + j) * 2, pk(v[j], v[j + 1]), pk(v[j + 2], v[j + 3]), pk(v[j + 4], v[j + 5]), pk(v[j + 6], v[j + 7]));
        }
        const int sh = H - 1 - y;
        const uint32_t win = skew + (sh >> 1) * 4, fs = (uint32_t)(sh & 1) << 4;
        uint32_t wd[H / 2 + 1];
#pragma unroll
        for (int j = 0; j <= H / 2; ++j) wd[j] = lds32u(win + 4 * j);
#pragma unroll
        for (int j = 0; j < H / 2; ++j) bq[j] = __funnelshift_r(wd[j], wd[j + 1], fs);
      }
      tc::tc_fence_before();
      tc::mbar_arrive(&sm.bar_tempty[buf]);         // accumulator buffer read: the MMA warp may overwrite it
      // ---- c * q from the TMA tile (bar_full completed before the MMA that filled the buffer; waited here for visibility) ----
      tc::mbar_wait(&sm.bar_full[s], (i / ST) & 1);
      uint32_t qp[DKH / 2];
      {
        const uint32_t qrow = smem_u32(sm.q[s]) + r * 128;
#pragma unroll
        for (int c = 0; c < DKH / 4; ++c) {
          const float4 t4 = lds128f(qrow + ((c ^ swz) << 4));
          qp[2 * c] = tc::pack_bf16x2(t4.x * LOG2E, t4.y * LOG2E);
          qp[2 * c + 1] = tc::pack_bf16x2(t4.z * LOG2E, t4.w * LOG2E);
        }
      }
      {   // release the q stage only once the loads above have delivered (see mbar_arrive_after)
        uint32_t fold = 0u;
#pragma unroll
        for (int c = 0; c < DKH / 2; ++c) fold ^= qp[c];
        tc::mbar_arrive_after(&sm.bar_empty[s], fold & dep_zero);
      }
      // ---- Qa row: [ c q | c Aq | c Bq | 0 (lse slots, backward) | 0 .. ] -> staging tile -> TMA store ----
      if (leader) bulk_wait_read0();                 // the previous tile's Ka store has finished READING the staging tile
      wg_sync();
      auto qa_word = [&](int wi) -> uint32_t {      // packed columns 2 wi, 2 wi + 1 (compile-time wi after unrolling)
        const int c = 2 * wi;
        if (c < DKH) return qp[wi];
        if (c < DKH + W) return aq[(c - DKH) / 2];
        if (c < DKH + W + H) return bq[(c - DKH - W) / 2];
        return 0u;
      };
#pragma unroll
      for (int ch = 0; ch < C::KP / 8; ++ch) {
        const uint32_t dst = stg0 + (ch >> 3) * (AB_BM * 128) + ((((uint32_t)ch & 7) ^ swz) << 4);
        sts128(dst, qa_word(4 * ch), qa_word(4 * ch + 1), qa_word(4 * ch + 2), qa_word(4 * ch + 3));
      }
      tc::fence_proxy_async();
      wg_sync();
      if (leader) {
#pragma unroll
        for (int a = 0; a < C::KATOMS; ++a) tma_store_3d(&tm_qa, sm.stg[wg][a], a * 64, l0, bn);
        bulk_commit();
      }
      // ---- Ka row: [ k | 1hot(x) | 1hot(y) | 1 1 | 0 .. | v | 1 1 | 0 .. ]: words built while the Qa store reads the tile ----
      const uint32_t hx = 0x3F80u << ((x & 1) << 4), hy = 0x3F80u << ((y & 1) << 4);
      const int ix = x >> 1, iy = y >> 1;
      auto ka_word = [&](int wi) -> uint32_t {
        const int c = 2 * wi;
        if (c < DKH) return tc::pack_bf16x2(kf[c], kf[c + 1]);
        if (c < DKH + W) return ((c - DKH) / 2 == ix) ? hx : 0u;
        if (c < DKH + W + H) return ((c - DKH - W) / 2 == iy) ? hy : 0u;
        if (c == C::KD) return 0x3F803F80u;         // the two lse slots
        if (c >= C::C1 && c < C::C1 + 16) {         // value block: v[0..dvh), 1, 1 (dvh is a run-time value)
          const int e = c - C::C1;
          const float lo = e < dvh ? vf[e < 14 ? e : 13] : (e < dvh + 2 ? 1.f : 0.f);
          const float hi = e + 1 < dvh ? vf[e + 1 < 14 ? e + 1 : 13] : (e + 1 < dvh + 2 ? 1.f : 0.f);
          return tc::pack_bf16x2(lo, hi);
        }
        return 0u;
      };
      uint32_t kw[C::KP / 2];
#pragma unroll
      for (int wi = 0; wi < C::KP / 2; ++wi) kw[wi] = ka_word(wi);
      if (leader) bulk_wait_read0();
      wg_sync();
#pragma unroll
      for (int ch = 0; ch < C::KP / 8; ++ch) {
        const uint32_t dst = stg0 + (ch >> 3) * (AB_BM * 128) + ((((uint32_t)ch & 7) ^ swz) << 4);
        sts128(dst, kw[4 * ch], kw[4 * ch + 1], kw[4 * ch + 2], kw[4 * ch + 3]);
      }
      tc::fence_proxy_async();
      wg_sync();
      if (leader) {
#pragma unroll
        for (int a = 0; a < C::KATOMS; ++a) tma_store_3d(&tm_ka, sm.stg[wg][a], a * 64, l0, bn);
        bulk_commit();
      }
    }
    if (leader) bulk_wait0();
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == W_MMA) tc::tmem_dealloc<C::TALLOC>(tmem);
}

int sm_count_ab() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
  }
  return n;
}

template <int W, int H, int DKH>
int launch_aug_build_tc(const Dims& d, const float* q, const float* k, const float* v, const float* krw, const float* krh, void* qa,
                        void* ka, cudaStream_t st) {
  typedef AbCfg<W, H, DKH> C;
  CUtensorMap tq, tqa, tka;
  {
    const uint64_t dims[3] = {(uint64_t)DKH, (uint64_t)d.L, (uint64_t)d.BN};
    const uint64_t strides[2] = {(uint64_t)DKH * 4, (uint64_t)d.L * DKH * 4};
    const uint32_t box[3] = {32, AB_BM, 1};
    AACONV_TRY(make_tmap_f32(&tq, q, 3, dims, strides, box));
  }
  for (int i = 0; i < 2; ++i) {
    const uint64_t dims[3] = {(uint64_t)C::KP, (uint64_t)d.L, (uint64_t)d.BN};
    const uint64_t strides[2] = {(uint64_t)C::KP * 2, (uint64_t)d.L * C::KP * 2};
    const uint32_t box[3] = {64, AB_BM, 1};
    AACONV_TRY(make_tmap_bf16(i ? &tka : &tqa, i ? ka : qa, 3, dims, strides, box, nullptr));
  }
  const size_t smem = sizeof(AbSmem<C>) + 1024;
  auto kern = aug_build_tc_kernel<W, H, DKH>;
  AACONV_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int tiles_per_bn = cdiv(d.L, AB_BM), ntiles = tiles_per_bn * d.BN;
  kern<<<std::min(ntiles, sm_count_ab()), C::THREADS, smem, AACONV_ST(st)>>>(tq, tqa, tka, k, v, krw, krh, d.L, d.dvh, tiles_per_bn, ntiles, 0u);
  AACONV_LAUNCH_OK("aug_build_tc");
  return 0;
}

}  // namespace

// 0 when the tcgen05 builder covers the shape (relative attention on the square DenseNet maps, dk/nh = 20)
int aug_build_tc_supported(const Dims& d) {
  if (!d.relative || d.dkh != 20 || d.H != d.W || d.dvh < 1 || d.dvh > 14) return AACONV_E_UNSUPPORTED;
  if (d.W != 10 && d.W != 20 && d.W != 40 && d.W != 64) return AACONV_E_UNSUPPORTED;
  const AugLayout a = aug_layout(d);
  if (a.KD != d.dkh + d.W + d.H) return AACONV_E_UNSUPPORTED;
  return 0;
}

int aug_build_tc(const Dims& d, const float* q, const float* k, const float* v, const float* krw, const float* krh, void* qa,
                 void* ka, cudaStream_t st) {
  if (aug_build_tc_supported(d)) return fail(AACONV_E_UNSUPPORTED, "aug_build_tc: shape not covered");
  switch (d.W) {
    case 10: return launch_aug_build_tc<10, 10, 20>(d, q, k, v, krw, krh, qa, ka, st);
    case 20: return launch_aug_build_tc<20, 20, 20>(d, q, k, v, krw, krh, qa, ka, st);
    case 40: return launch_aug_build_tc<40, 40, 20>(d, q, k, v, krw, krh, qa, ka, st);
    default: return launch_aug_build_tc<64, 64, 20>(d, q, k, v, krw, krh, qa, ka, st);
  }
}

namespace {

// ================================================================================================
// rel_bwd_tc: dQa -> total dq (content + relative part, bf16 into the packed dqkv operand of the projection GEMMs) and the
// key_rel_w / key_rel_h gradient partials, on tcgen05 -- round-2 replacement of rel_bwd_kernel (mma.sync TF32).
//
//   dR[row, r]  = dAq[row, r - (W-1-x(row))] inside the window, 0 elsewhere  (adjoint of the rel_to_abs index law)
//   dq_rel      = dR . T^T          MMA1: D1[128 rows x 32] = A[rows x K] . B[e x K]^T, A = dR tile (K-major), B = tables
//   dT^T[r, e] += dR^T . q          MMA2: D2[128 r x 32]   += A^T (the same tile viewed MN-major) . q tile (MN-major)
//
// One thread owns one row: it reads its dQa row from the staged tile, writes the window of packed bf16 pairs at its own
// offset into the 128B-swizzled A tile (zero elsewhere) and its q row into the q tile; the MMA warp issues both products; the
// thread then adds D1 to the content part and stores 20 bf16.  D2 accumulates over all tiles of the CTA and is written once
// as a partial for rel_bwd_reduce_kernel.  Reference: adjoint of attn_aug_conv.py:55-63,77-86.
// ================================================================================================
template <int W, int H, int DKH>
struct RbCfg {
  static constexpr int NW = ru16(2 * W - 1), NH = ru16(2 * H - 1), KCOLS = NW + NH;
  static constexpr int KA = (KCOLS + 63) / 64 < 2 ? 2 : (KCOLS + 63) / 64;     // 64-column atoms of the A tile (>= 2: M = 128 blocks)
  static constexpr int NBLK = KA >= 3 ? 2 : 1;            // D2 blocks of 128 A-columns: atoms {0,1} and {KA-2, KA-1}
  static constexpr int KD = DKH + W + H;
  static constexpr int NKS1 = (KCOLS + 15) / 16;
  static constexpr int IN_BYTES = AB_BM * KD * 4;
  static constexpr int fixed = KA * AB_BM * 128 + AB_BM * 128 + KA * 32 * 128 + 2048;
  static constexpr int fit = (225 * 1024 - fixed) / IN_BYTES;
  static constexpr int STAGES = fit > 3 ? 3 : fit;
  static_assert(STAGES >= 1 && KD % 4 == 0 && DKH % 4 == 0 && DKH <= 32, "rel_bwd_tc configuration");
};

template <class C>
struct __align__(1024) RbSmem {
  bf16 a[C::KA][AB_BM * 64];                      // dR tile: 128 rows x (NW | NH) columns, 128B-swizzled atoms
  bf16 qt[AB_BM * 64];                            // q tile (first 32 columns used)
  bf16 t[C::KA][32 * 64];                         // tables as the B operand of MMA1: row e, K = A column
  float in[C::STAGES][AB_BM * C::KD];             // dQa tiles (1-D bulk copies)
  uint64_t bar_full[C::STAGES], bar_empty[C::STAGES], bar_a_ready, bar_done;
  uint32_t tmem_base;
};

__device__ __forceinline__ void bulk_g2s_1d(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
__device__ __forceinline__ void sts32(uint32_t saddr, uint32_t v) { asm volatile("st.shared.b32 [%0], %1;" ::"r"(saddr), "r"(v) : "memory"); }

// N fp32 values at byte offset OFF of a staged row -> packed bf16 pairs dst[1 .. N/2] (16-byte loads when OFF allows, else 8-byte)
template <int N, int OFF>
__device__ __forceinline__ void load_pairs(uint32_t row, bool live, uint32_t* dst) {
  if (OFF % 16 == 0) {
#pragma unroll
    for (int c = 0; c < N / 4; ++c) {
      const float4 t4 = live ? lds128f(row + OFF + 16 * c) : make_float4(0.f, 0.f, 0.f, 0.f);
      dst[1 + 2 * c] = tc::pack_bf16x2(t4.x, t4.y);
      dst[2 + 2 * c] = tc::pack_bf16x2(t4.z, t4.w);
    }
    if (N % 4) {
      const float a0 = live ? lds32f(row + OFF + (N - 2) * 4) : 0.f, a1 = live ? lds32f(row + OFF + (N - 1) * 4) : 0.f;
      dst[N / 2] = tc::pack_bf16x2(a0, a1);
    }
  } else {
#pragma unroll
    for (int c = 0; c < N / 2; ++c) {
      float a0 = 0.f, a1 = 0.f;
      if (live) asm volatile("ld.shared.v2.f32 {%0,%1}, [%2];" : "=f"(a0), "=f"(a1) : "r"(row + OFF + 8 * c) : "memory");
      dst[1 + c] = tc::pack_bf16x2(a0, a1);
    }
  }
}

template <int W, int H, int DKH>
__global__ void __launch_bounds__(192, 1) rel_bwd_tc_kernel(const float* __restrict__ dqa, const float* __restrict__ qg,
                                                            const float* __restrict__ krw, const float* __restrict__ krh,
                                                            bf16* __restrict__ dqkvh, float* __restrict__ partial, int L, int nh,
                                                            int KPq, int RP, int DK8, float qscale, int tiles_per_bn, int ntiles,
                                                            uint32_t dep_zero /* always 0: see tc::mbar_arrive_after */) {
  typedef RbCfg<W, H, DKH> C;
  typedef RbSmem<C> Smem;
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  Smem& sm = *reinterpret_cast<Smem*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int ST = C::STAGES, KA = C::KA;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int my_tiles = (ntiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  auto tile_rows = [&](int i, int& bn, int& l0) {
    const int tile = blockIdx.x + i * gridDim.x;
    bn = tile / tiles_per_bn;
    l0 = (tile - bn * tiles_per_bn) * AB_BM;
    return min(AB_BM, L - l0);
  };

  if (warp == 4 && lane == 0) {
    for (int s = 0; s < ST; ++s) { tc::mbar_init(&sm.bar_full[s], 1); tc::mbar_init(&sm.bar_empty[s], 128); }
    tc::mbar_init(&sm.bar_a_ready, 128);
    tc::mbar_init(&sm.bar_done, 1);
    tc::fence_barrier_init();
    for (int i = 0; i < ST && i < my_tiles; ++i) {
      int bn, l0;
      const int nrows = tile_rows(i, bn, l0);
      tc::mbar_arrive_expect_tx(&sm.bar_full[i], nrows * C::KD * 4);
      bulk_g2s_1d(sm.in[i], dqa + ((size_t)bn * L + l0) * C::KD, nrows * C::KD * 4, &sm.bar_full[i]);
    }
  }
  if (warp == 5) tc::tmem_alloc<128>(&sm.tmem_base);
  if (warp < 4) {
    // tables as MMA1's B operand (row e, K = A column: W axis at [0, NW), H axis at [NW, NW + NH)), zero padded; and the
    // constant parts of the A / q tiles (everything a row owner does not rewrite per tile)
    uint4* z = reinterpret_cast<uint4*>(sm.a);                        // a, qt, t are adjacent
    constexpr int NZ = (KA * AB_BM * 128 + AB_BM * 128 + KA * 32 * 128) / 16;
    for (int i = threadIdx.x; i < NZ; i += 128) z[i] = make_uint4(0u, 0u, 0u, 0u);
    constexpr int RW_ = 2 * W - 1, RH_ = 2 * H - 1, NTAB = DKH * (RW_ + RH_), PER = (NTAB + 127) / 128;
    float tv[PER];
#pragma unroll
    for (int u = 0; u < PER; ++u) {
      const int i = threadIdx.x + u * 128;
      tv[u] = i < NTAB ? __ldg((i >= DKH * RW_ ? krh - DKH * RW_ : krw) + i) : 0.f;
    }
    asm volatile("bar.sync 1, 128;" ::: "memory");
#pragma unroll
    for (int u = 0; u < PER; ++u) {
      const int i = threadIdx.x + u * 128;
      if (i < NTAB) {
        const bool hax = i >= DKH * RW_;
        const int j = hax ? i - DKH * RW_ : i, R = hax ? RH_ : RW_;
        const int e = j / R, k = j - e * R + (hax ? C::NW : 0);
        const int at = k >> 6, kc = k & 63;
        sm.t[at][e * 64 + ((((kc >> 3) ^ (e & 7)) << 3) | (kc & 7))] = __float2bfloat16(tv[u]);
      }
    }
  }
  tc::fence_proxy_async();
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = sm.tmem_base;
  constexpr uint32_t COL_D1 = 0, COL_D2 = 32;

  if (warp == 4) {
    if (lane == 0) {
      for (int i = ST; i < my_tiles; ++i) {
        int bn, l0;
        const int nrows = tile_rows(i, bn, l0), s = i % ST;
        tc::mbar_wait(&sm.bar_empty[s], ((i / ST) & 1) ^ 1);
        tc::mbar_arrive_expect_tx(&sm.bar_full[s], nrows * C::KD * 4);
        bulk_g2s_1d(sm.in[s], dqa + ((size_t)bn * L + l0) * C::KD, nrows * C::KD * 4, &sm.bar_full[s]);
      }
    }
  } else if (warp == 5) {
    // ===================== MMA issuer =====================
    constexpr uint32_t id1 = tc::idesc_bf16_f32(AB_BM, 32);
    constexpr uint32_t id2 = tc::idesc_bf16_f32(AB_BM, 32) | (1u << 15) | (1u << 16);     // A and B MN-major
    const uint32_t a_k = tc::desc_lo_k(smem_u32(sm.a[0])), t_k = tc::desc_lo_k(smem_u32(sm.t[0]));
    const uint32_t q_mn = tc::desc_lo_mn(smem_u32(sm.qt), AB_BM * 128);
    for (int i = 0; i < my_tiles; ++i) {
      tc::mbar_wait(&sm.bar_a_ready, i & 1);
      tc::tc_fence_after();
      if (tc::elect_one()) {
#pragma unroll
        for (int ks = 0; ks < C::NKS1; ++ks)
          tc::mma_ss(tmem + COL_D1, tc::desc64(a_k + (ks >> 2) * ((AB_BM * 128) >> 4) + (ks & 3) * 2),
                     tc::desc64(t_k + (ks >> 2) * ((32 * 128) >> 4) + (ks & 3) * 2), id1, ks > 0);
#pragma unroll
        for (int b = 0; b < C::NBLK; ++b) {
          const uint32_t a_mn = tc::desc_lo_mn(smem_u32(sm.a[b == 0 ? 0 : KA - 2]), AB_BM * 128);
#pragma unroll
          for (int ks = 0; ks < AB_BM / 16; ++ks)
            tc::mma_ss(tmem + COL_D2 + 32 * b, tc::desc64(a_mn + ks * 128), tc::desc64(q_mn + ks * 128), id2, (i > 0 || ks > 0) ? 1u : 0u);
        }
        tc::mma_commit(&sm.bar_done);
      }
      __syncwarp();
    }
  } else {
    // ===================== row owners =====================
    const int r = threadIdx.x;
    const uint32_t tlane = tmem + ((uint32_t)(warp * 32) << 16);
    const uint32_t swz = (uint32_t)(r & 7);
    const uint32_t arow = smem_u32(sm.a[0]) + r * 128, qrow = smem_u32(sm.qt) + r * 128;
    float dqc[DKH];                                  // content part of the PREVIOUS tile's row, waiting for its D1
    bf16* dst_prev = nullptr;
    auto finish_prev = [&](int iprev) {              // D1 of tile iprev -> dq_total -> bf16 store
      tc::mbar_wait(&sm.bar_done, iprev & 1);
      tc::tc_fence_after();
      uint32_t d1[32];
      tc::tmem_ld_x32(tlane + COL_D1, d1);
      tc::tmem_ld_wait();
      tc::tc_fence_before();
      if (dst_prev) {
#pragma unroll
        for (int e = 0; e < DKH; e += 4) {
          uint2 w2;
          w2.x = tc::pack_bf16x2((dqc[e] + __uint_as_float(d1[e])) * qscale, (dqc[e + 1] + __uint_as_float(d1[e + 1])) * qscale);
          w2.y = tc::pack_bf16x2((dqc[e + 2] + __uint_as_float(d1[e + 2])) * qscale, (dqc[e + 3] + __uint_as_float(d1[e + 3])) * qscale);
          *reinterpret_cast<uint2*>(dst_prev + e) = w2;
        }
      }
    };
    for (int i = 0; i < my_tiles; ++i) {
      int bn, l0;
      const int nrows = tile_rows(i, bn, l0), s = i % ST;
      const bool live = r < nrows;
      const int l = min(l0 + r, L - 1);
      const int y = l / W, x = l - y * W;
      const size_t grow = (size_t)bn * L + l;
      float qf[DKH];
#pragma unroll
      for (int e = 0; e < DKH; e += 4) {
        const float4 t4 = live ? __ldg(reinterpret_cast<const float4*>(qg + grow * DKH + e)) : make_float4(0.f, 0.f, 0.f, 0.f);
        qf[e] = t4.x; qf[e + 1] = t4.y; qf[e + 2] = t4.z; qf[e + 3] = t4.w;
      }
      // ---- this row of the staged dQa tile: [ dq | dAq | dBq ] ----
      tc::mbar_wait(&sm.bar_full[s], (i / ST) & 1);
      const uint32_t irow = smem_u32(sm.in[s]) + r * (C::KD * 4);
      float cur[DKH];
      uint32_t pa[W / 2 + 2], pb[H / 2 + 2];        // packed pairs with a zero word on either side
      pa[0] = pa[W / 2 + 1] = pb[0] = pb[H / 2 + 1] = 0u;
#pragma unroll
      for (int c = 0; c < DKH / 4; ++c) {
        const float4 t4 = live ? lds128f(irow + 16 * c) : make_float4(0.f, 0.f, 0.f, 0.f);
        cur[4 * c] = t4.x; cur[4 * c + 1] = t4.y; cur[4 * c + 2] = t4.z; cur[4 * c + 3] = t4.w;
      }
      load_pairs<W, DKH * 4>(irow, live, pa);
      load_pairs<H, (DKH + W) * 4>(irow, live, pb);
      {   // release the stage only once every load above has delivered (see mbar_arrive_after)
        uint32_t fold = 0u;
#pragma unroll
        for (int e = 0; e < DKH; ++e) fold ^= __float_as_uint(cur[e]);
#pragma unroll
        for (int j = 1; j <= W / 2; ++j) fold ^= pa[j];
#pragma unroll
        for (int j = 1; j <= H / 2; ++j) fold ^= pb[j];
        tc::mbar_arrive_after(&sm.bar_empty[s], fold & dep_zero);
      }
      // ---- the previous tile's products are done: its D1 leaves, and the A / q tiles may be rewritten ----
      if (i > 0) finish_prev(i - 1);
#pragma unroll
      for (int e = 0; e < DKH; ++e) dqc[e] = cur[e];
      {
        const int b = bn / nh, n = bn - b * nh;
        dst_prev = live ? dqkvh + ((size_t)b * L + l) * KPq + n * DKH : nullptr;
      }
      // zero row, then the two windows: word j of a window = pairs shifted by the parity of its start column
#pragma unroll
      for (int at = 0; at < KA; ++at)
#pragma unroll
        for (int ch = 0; ch < 8; ++ch) sts128(arow + at * (AB_BM * 128) + (ch << 4), 0u, 0u, 0u, 0u);
      auto put_word = [&](int wi, uint32_t v) {      // packed A columns 2 wi, 2 wi + 1
        const uint32_t at = (uint32_t)wi >> 5, w5 = (uint32_t)wi & 31;
        sts32(arow + at * (AB_BM * 128) + ((((w5 >> 2) ^ swz) << 4) | ((w5 & 3) << 2)), v);
      };
      {
        const int sh = W - 1 - x, w0 = sh >> 1;
        const uint32_t fs = (uint32_t)(sh & 1) << 4;
#pragma unroll
        for (int j = 0; j <= W / 2; ++j) put_word(w0 + j, __funnelshift_l(pa[j], pa[j + 1], fs));
      }
      {
        const int sh = C::NW + H - 1 - y, w0 = sh >> 1;
        const uint32_t fs = (uint32_t)(sh & 1) << 4;
#pragma unroll
        for (int j = 0; j <= H / 2; ++j) put_word(w0 + j, __funnelshift_l(pb[j], pb[j + 1], fs));
      }
      // q row (bf16) into the q tile: columns [0, 32)
#pragma unroll
      for (int ch = 0; ch < 4; ++ch) {
        uint32_t w4[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int e = 8 * ch + 2 * u;
          w4[u] = e < DKH ? tc::pack_bf16x2(qf[e < DKH ? e : 0], qf[e + 1 < DKH ? e + 1 : 0]) : 0u;
        }
        sts128(qrow + (((uint32_t)ch ^ swz) << 4), w4[0], w4[1], w4[2], w4[3]);
      }
      tc::fence_proxy_async();
      tc::mbar_arrive(&sm.bar_a_ready);
    }
    if (my_tiles > 0) {
      finish_prev(my_tiles - 1);                     // also: every MMA of this CTA has completed
      // ---- key_rel gradient partial: D2 block b, lane = A column (colbase + r), 32 columns = e ----
      tc::tc_fence_after();
      float* out = partial + (size_t)blockIdx.x * 2 * RP * DK8;
#pragma unroll
      for (int b = 0; b < C::NBLK; ++b) {
        uint32_t d2[32];
        tc::tmem_ld_x32(tlane + COL_D2 + 32 * b, d2);
        tc::tmem_ld_wait();
        const int k = (b == 0 ? 0 : (KA - 2) * 64) + r;
        if (b == 1 && k < 128) continue;             // columns already covered by block 0
        const int axis = k >= C::NW ? 1 : 0, rr = k - (axis ? C::NW : 0);
        if (rr < (axis ? 2 * H - 1 : 2 * W - 1) && rr < RP) {
          float* o = out + ((size_t)axis * RP + rr) * DK8;
#pragma unroll
          for (int e = 0; e < DKH; ++e) o[e] = __uint_as_float(d2[e]);
        }
      }
      tc::tc_fence_before();
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == 5) tc::tmem_dealloc<128>(tmem);
}

template <int W, int H, int DKH>
int launch_rel_bwd_tc(const Dims& d, const float* dqa, const float* q, const float* krw, const float* krh, void* dqkvh, int KPq,
                      float* partial, int RP, int DK8, int* grid_out, cudaStream_t st) {
  typedef RbCfg<W, H, DKH> C;
  const size_t smem = sizeof(RbSmem<C>) + 1024;
  auto kern = rel_bwd_tc_kernel<W, H, DKH>;
  AACONV_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int tiles_per_bn = cdiv(d.L, AB_BM), ntiles = tiles_per_bn * d.BN;
  const int grid = std::min(ntiles, sm_count_ab());
  kern<<<grid, 192, smem, AACONV_ST(st)>>>(dqa, q, krw, krh, static_cast<bf16*>(dqkvh), partial, d.L, d.nh, KPq, RP, DK8, d.qscale,
                                           tiles_per_bn, ntiles, 0u);
  AACONV_LAUNCH_OK("rel_bwd_tc");
  *grid_out = grid;
  return 0;
}

}  // namespace

// same shapes as the builder, bf16 packed output only (KPq a multiple of 4: 8-byte stores)
int rel_bwd_tc_supported(const Dims& d, int KPq) {
  if (aug_build_tc_supported(d)) return AACONV_E_UNSUPPORTED;
  if (KPq & 3) return AACONV_E_UNSUPPORTED;
  return 0;
}

// -> number of partials written (one per CTA), layout [part][axis][RP][DK8] as rel_bwd_kernel's
int rel_bwd_tc(const Dims& d, const float* dqa, const float* q, const float* krw, const float* krh, void* dqkvh, int KPq,
               float* partial, int RP, int DK8, int* nparts, cudaStream_t st) {
  if (rel_bwd_tc_supported(d, KPq)) return fail(AACONV_E_UNSUPPORTED, "rel_bwd_tc: shape not covered");
  switch (d.W) {
    case 10: return launch_rel_bwd_tc<10, 10, 20>(d, dqa, q, krw, krh, dqkvh, KPq, partial, RP, DK8, nparts, st);
    case 20: return launch_rel_bwd_tc<20, 20, 20>(d, dqa, q, krw, krh, dqkvh, KPq, partial, RP, DK8, nparts, st);
    case 40: return launch_rel_bwd_tc<40, 40, 20>(d, dqa, q, krw, krh, dqkvh, KPq, partial, RP, DK8, nparts, st);
    default: return launch_rel_bwd_tc<64, 64, 20>(d, dqa, q, krw, krh, dqkvh, KPq, partial, RP, DK8, nparts, st);
  }
}

}  // namespace aaconv
