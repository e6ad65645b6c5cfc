// bf16 tcgen05 attention core of AAConv2d for small value widths (dv/nh <= 2, the Transition-1 case): forward, dK/dV and dQa
// kernels in which only the dense contractions stay on the tensor cores and the rank-dvh value terms run on the CUDA cores:
//
//   forward   S' = Qa.Ka^T (tcgen05, TS)           p = 2^(S'-m),  l += p,  o += p v[k]           (no P write-back, no P.V MMA)
//   backward  S' = Qa.Ka^T - lse2 (tcgen05, TS)    p = 2^S',  dP = dO.v[k] - delta,  dS = p dP    (no dP' MMA, no dP' TMEM read)
//             dQa += dS.Ka,  dK += dS^T.Qa,  dV += P^T.dO  (tcgen05, TS, MN-major B)
//
// Why (measured, DESIGN.md section 4): the value width is 1..2, so P.V / dO.v are 1-2 FMAs per score next to one MUFU.EX2;
// doing them in registers halves the TMEM reads, removes two of the four barrier round trips per tile and shrinks a score
// slot to the S' columns alone, so that five slots fit in TMEM and the issuing warps run far enough ahead of the math
// warpgroups to keep both busy.  v / dO / delta tiles come as fp32 through 1-D bulk copies on the K/Q tile's barrier.
// All three kernels are PERSISTENT (one CTA per SM walks a list of (batch*head, stationary tile) items with its barrier
// rings running on a global tile counter); the rules that keeps their mbarrier parity waits exact are next to cb_plan.
// Reference rows a3-a8 (attn_aug_conv.py:75-91) and their adjoint; layouts as in attn_tc_bwd.cu.
#include <algorithm>
#include <cstdlib>
#include "tc_common.cuh"
#include "bf16_path.cuh"

namespace aaconv {

using tc::smem_u32;
typedef __nv_bfloat16 bf16;

// ablation switches for tools/attn_ablate.py (0 in production): 1 no MUFU, 2 no global traffic after the first tiles,
// 4 no gradient MMAs, 8 no math at all, 32 dQa drain by per-row stores; 16 = soft mbarrier timeouts (tools/dbg_shape.py)
int g_attn_dbg_mode = 0;
static unsigned long long* g_mbar_host_log = nullptr;
extern long long* g_attn_dbg;      // attn_tc_bwd.cu: timeline buffer of TL_EVENTS x TL_COLS stamps (tools/attn_timeline.py)
constexpr int TL_COLS = 96, TL_CTA = 40;
#define TL_STAMP(tl, ev, col) do { if ((tl) && (col) < TL_COLS) (tl)[(ev) * TL_COLS + (col)] = clock64(); } while (0)
extern "C" void aaconv_debug_set_mode(int m) {
  g_attn_dbg_mode = m & 47;            // bit 32: dQa drain by per-row stores instead of the bulk store
  const unsigned soft = (m >> 4) & 1;                    // bit 16: soft mbarrier timeouts in this file's kernels (see tc_common.cuh)
  static unsigned long long* host_log = nullptr;
  if (soft && !host_log) cudaHostAlloc(reinterpret_cast<void**>(&host_log), 65 * sizeof(unsigned long long), cudaHostAllocMapped);
  if (host_log) {
    for (int i = 0; i < 65; ++i) host_log[i] = 0;
    unsigned long long* dev = nullptr;
    cudaHostGetDevicePointer(reinterpret_cast<void**>(&dev), host_log, 0);
    cudaMemcpyToSymbol(tc::g_mbar_log, &dev, sizeof dev);
  }
  cudaMemcpyToSymbol(tc::g_mbar_soft, &soft, sizeof soft);
  g_mbar_host_log = host_log;
}
// -> number of timed-out waits logged since the mode was set (readable even after the kernel faulted: the log lives in mapped
// host memory); out[i] = smem barrier address << 32 | parity << 31 | block << 12 | thread
extern "C" int aaconv_debug_read_mbar_log(unsigned long long* out, int max_entries) {
  if (!g_mbar_host_log) return 0;
  const int n = (int)g_mbar_host_log[0];
  for (int i = 0; i < n && i < 64 && i < max_entries; ++i) out[i] = g_mbar_host_log[1 + i];
  return n;
}

namespace {

__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gsrc, uint32_t bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}

// index + phase of a ring of n entries, advanced without integer division (a runtime modulo costs a MUFU.RCP, and the MUFU
// pipe is what the math warps saturate)
__device__ __forceinline__ int lane_id() { return threadIdx.x & 31; }

struct Ring {
  int i = 0;
  uint32_t ph = 0;
  __device__ __forceinline__ void next(int n) { if (++i == n) { i = 0; ph ^= 1; } }
  __device__ __forceinline__ void advance(int k, int n) { i += k; if (i >= n) { i -= n; ph ^= 1; } }   // k <= n
};

__device__ __forceinline__ float4 lds128(uint32_t saddr) {
  float4 v;
  asm volatile("ld.shared.v4.f32 {%0,%1,%2,%3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(saddr));
  return v;
}

// stationary tile (shared memory, 128B-swizzled K-major atoms) -> TMEM: row r -> lane r, column c <- elements 2c, 2c+1
template <int KATOMS>
__device__ __forceinline__ void stationary_to_tmem(const bf16 (*stat)[128 * 64], uint32_t tlane_a, int r) {
#pragma unroll
  for (int a = 0; a < KATOMS; ++a) {
    uint32_t w[32];
    const uint8_t* rowp = reinterpret_cast<const uint8_t*>(stat[a]) + r * 128;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
      const uint4 v = *reinterpret_cast<const uint4*>(rowp + ((c ^ (r & 7)) << 4));
      w[4 * c] = v.x; w[4 * c + 1] = v.y; w[4 * c + 2] = v.z; w[4 * c + 3] = v.w;
    }
    tc::tmem_st_x32(tlane_a + a * 32, w);
  }
  tc::tmem_st_wait();
  tc::tc_fence_before();
}

// 64 keys of the forward softmax: scores of this thread's query row in r (log2 units), fp32 values in shared memory.
// Online softmax with lazy rescale: the reference maximum m only moves when the tile maximum exceeds it by 2^8.
template <int DVH, bool TAIL>
__device__ __forceinline__ void fwd_cc_half(uint32_t (&r)[2][32], uint32_t vt, int nvalid, float& m, float& l, float (&acc)[DVH]) {
  if (TAIL) {
#pragma unroll
    for (int c = 0; c < 2; ++c)
#pragma unroll
      for (int i = 0; i < 32; ++i)
        if (c * 32 + i >= nvalid) r[c][i] = 0xff800000u;   // zero-filled keys past L: logit -> -inf
  }
  float mx[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};   // four independent chains
#pragma unroll
  for (int c = 0; c < 2; ++c)
#pragma unroll
    for (int i = 0; i < 32; i += 8) {
#pragma unroll
      for (int u = 0; u < 4; ++u) mx[u] = fmaxf(mx[u], fmaxf(__uint_as_float(r[c][i + 2 * u]), __uint_as_float(r[c][i + 2 * u + 1])));
    }
  const float mt = fmaxf(fmaxf(mx[0], mx[1]), fmaxf(mx[2], mx[3]));
  if (mt > m + 8.f) {                          // lazy rescale: exponentials stay below 2^8
    const float m_new = fmaxf(m, mt);
    const float alpha = tc::ex2f(m - m_new);   // 0 on the first tile (m = -inf)
    l *= alpha;
#pragma unroll
    for (int e = 0; e < DVH; ++e) acc[e] *= alpha;
    m = m_new;
  }
  const float mneg = -m;
  float l2 = 0.f;
#pragma unroll
  for (int c = 0; c < 2; ++c)
#pragma unroll
    for (int i = 0; i < 32; i += 4) {
      float vv[4 * DVH];
#pragma unroll
      for (int u = 0; u < DVH; ++u) {
        const float4 t4 = lds128(vt + ((c * 32 + i) * DVH + 4 * u) * 4);
        vv[4 * u] = t4.x; vv[4 * u + 1] = t4.y; vv[4 * u + 2] = t4.z; vv[4 * u + 3] = t4.w;
      }
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const float p = tc::ex2_mixed(__uint_as_float(r[c][i + u]) + mneg, u);
        if (u & 1) l2 += p; else l += p;
#pragma unroll
        for (int e = 0; e < DVH; ++e) {
          const float val = (TAIL && c * 32 + i + u >= nvalid) ? 0.f : vv[u * DVH + e];
          acc[e] = fmaf(p, val, acc[e]);
        }
      }
    }
  l += l2;
}

// ================================================================================================
// Persistent CTAs.  One CTA per SM walks a static list of work items (item = blockIdx.x + i * gridDim.x; an item is one
// stationary tile of one (batch, head) pair).  All rings (streamed-tile stages, TMEM score slots, warpgroup rotation)
// run on a GLOBAL tile counter across items, so the TMA warp streams the next item's tiles while the math warpgroups
// finish the current one, the stationary operand is double-buffered in TMEM, and the only per-item serial work left is
// the accumulator drain.  Measured before (profiles/r01_c_head.md + tools/attn_timeline.py): one CTA per item spent
// ~2.4 k cycles before its first MMA, ~4 k after its last and ~5 k between CTAs, out of ~30 k per item.
// ================================================================================================
__device__ __forceinline__ void bulk_s2g(void* gdst, const void* smem_src, uint32_t bytes) {
  asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gdst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
  asm volatile("cp.async.bulk.commit_group;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }

// ================================================================================================
// forward
// ================================================================================================
// Measured A/B on B200 (T1, B = 16; profiles/r02_attn_ab.md): 128-key tiles with three 128-column score slots and two
// tcgen05.ld in flight per half tile (this configuration) 132 us; 64-key tiles with six 64-column slots (two per warpgroup)
// 142 us; four warpgroups (96 registers) 140 us; S' read in four software-pipelined 32-column chunks 136 us.  The kernel is
// bound by the per-warp dependent-issue rate (ncu: issue slots 61 % busy, MUFU pipe 67 %, 7.7 instructions per exponential),
// not by TMEM latency, slot count or the number of MMA k-steps (2 k-steps instead of 7: 127 us).
constexpr int CF_BM = 128, CF_BN = 128, CF_SLOTS = 3;
// three softmax warpgroups (global tile t -> warpgroup t % 3), one TMA warp, one score-MMA issuer (+TMEM alloc)
constexpr int CF_NWG = 3, CF_W_TMA = 4 * CF_NWG, CF_W_S = CF_W_TMA + 1, CF_THREADS = 32 * (CF_W_S + 1);
template <int KATOMS> struct CfStages { static constexpr int value = KATOMS >= 3 ? 3 : 4; };
// Qa buffers in TMEM: two when they fit next to the score slots
template <int KATOMS> struct CfQBuf { static constexpr int value = (2 * KATOMS * 32 + CF_SLOTS * CF_BN <= 512) ? 2 : 1; };

template <int KATOMS, int DVH>
struct __align__(1024) CfSmem {
  static constexpr int ST = CfStages<KATOMS>::value;
  bf16 q[KATOMS][CF_BM * 64];
  bf16 k[ST][KATOMS][CF_BN * 64];
  float vt[ST][CF_BN * DVH];                  // fp32 values of the key tile
  float xch[2][CF_NWG][CF_BM][4];             // per tile class (j % 3): partial (m, l, o[0..DVH)), double-buffered by item parity
  uint64_t bar_q, bar_q_free, bar_a_ready, bar_final, bar_full[ST], bar_empty[ST], bar_s_full[CF_SLOTS], bar_slot_free[CF_SLOTS];
  uint32_t tmem_base;
};

template <int KATOMS, int NKS, class Smem>
__device__ __forceinline__ void cf_score_loop(Smem& sm, uint32_t tmem, int ntiles, int my_items) {
  constexpr int ST = Smem::ST, NS = CF_SLOTS, QB = CfQBuf<KATOMS>::value;
  constexpr uint32_t COL_SLOT0 = QB * KATOMS * 32;
  constexpr uint32_t idesc_s = tc::idesc_bf16_f32(CF_BM, CF_BN);
  constexpr uint32_t K_ATOM = (CF_BN * 128) >> 4, K_STAGE = KATOMS * K_ATOM;
  const uint32_t k_lo = tc::desc_lo_k(smem_u32(sm.k[0][0]));
  Ring rst, rsl;
  int filled = 0;                                // the first NS tiles find their slot free
  for (int it = 0; it < my_items; ++it) {
    tc::mbar_wait(&sm.bar_a_ready, it & 1);
    tc::tc_fence_after();
    const uint32_t qa = tmem + (uint32_t)((it & (QB - 1)) * KATOMS * 32);
    for (int j = 0; j < ntiles; ++j, rst.next(ST), rsl.next(NS)) {
      const int st = rst.i, slot = rsl.i;
      tc::mbar_wait(&sm.bar_full[st], rst.ph);
      if (filled >= NS) tc::mbar_wait(&sm.bar_slot_free[slot], rsl.ph ^ 1);
      else ++filled;
      tc::tc_fence_after();
      if (tc::elect_one()) {
        tc::issue_ts_ksteps<NKS, 0, K_ATOM>(tmem + COL_SLOT0 + 128 * slot, 0u, qa, k_lo + st * K_STAGE, idesc_s);
        tc::mma_commit(&sm.bar_s_full[slot]);
        tc::mma_commit(&sm.bar_empty[st]);        // the K tile is free once these MMAs are done (+128 arrivals for vt)
        if (QB == 1 && j == ntiles - 1) tc::mma_commit(&sm.bar_final);   // single Qa buffer: refill only after the item's last MMA
      }
      __syncwarp();
    }
  }
}

template <int KATOMS, int DVH>
__global__ void __launch_bounds__(CF_THREADS, 1) attn_fwd_cc_kernel(
    const __grid_constant__ CUtensorMap tm_q, const __grid_constant__ CUtensorMap tm_k, const float* __restrict__ v,
    float* __restrict__ o, float* __restrict__ lse, int L, int C1, int nqt, int nitems, int dbg) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  typedef CfSmem<KATOMS, DVH> Smem;
  Smem& sm = *reinterpret_cast<Smem*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int ST = Smem::ST, NS = CF_SLOTS, QB = CfQBuf<KATOMS>::value;
  constexpr uint32_t COL_SLOT0 = QB * KATOMS * 32;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ntiles = (L + CF_BN - 1) / CF_BN;
  const int my_items = (nitems - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;

  if (warp == CF_W_TMA && lane == 0) {   // barrier set-up + the first Q tile load before the CTA-wide sync
    tc::mbar_init(&sm.bar_q, 1);
    tc::mbar_init(&sm.bar_q_free, 128);
    tc::mbar_init(&sm.bar_a_ready, 128);
    tc::mbar_init(&sm.bar_final, 1);
    for (int s = 0; s < ST; ++s) { tc::mbar_init(&sm.bar_full[s], 1); tc::mbar_init(&sm.bar_empty[s], 129); }
    for (int s = 0; s < NS; ++s) { tc::mbar_init(&sm.bar_s_full[s], 1); tc::mbar_init(&sm.bar_slot_free[s], 128); }
    tc::fence_barrier_init();
    const int item = blockIdx.x, bn = item / nqt, q0 = (item - bn * nqt) * CF_BM;
    tc::mbar_arrive_expect_tx(&sm.bar_q, KATOMS * CF_BM * 64 * 2);
    for (int a = 0; a < KATOMS; ++a) tc::tma_load_3d(sm.q[a], &tm_q, &sm.bar_q, a * 64, q0, bn);
    tc::tma_prefetch_desc(&tm_k);
  }
  if (warp == CF_W_S) tc::tmem_alloc<512>(&sm.tmem_base);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
  const uint32_t tmem = sm.tmem_base;

  if (warp == CF_W_TMA) {
    if (lane == 0) {
      Ring rg;
      const int jq = ntiles / 2;                    // see cb_producer
      for (int it = 0; it < my_items; ++it) {
        const int item = blockIdx.x + it * gridDim.x, bn = item / nqt;
        for (int j = 0; j < ntiles; ++j, rg.next(ST)) {
          if (j == jq && it + 1 < my_items) {          // next item's Q tile: its staging buffer is free once WG0 has moved
            const int nitem = item + gridDim.x, nbn = nitem / nqt, nq0 = (nitem - nbn * nqt) * CF_BM;   // this item's to TMEM
            tc::mbar_wait(&sm.bar_q_free, it & 1);
            tc::mbar_arrive_expect_tx(&sm.bar_q, KATOMS * CF_BM * 64 * 2);
            for (int a = 0; a < KATOMS; ++a) tc::tma_load_3d(sm.q[a], &tm_q, &sm.bar_q, a * 64, nq0, nbn);
          }
          const int s = rg.i;
          const int nvalid = min(CF_BN, L - j * CF_BN);
          tc::mbar_wait(&sm.bar_empty[s], rg.ph ^ 1);
          tc::mbar_arrive_expect_tx(&sm.bar_full[s], KATOMS * CF_BN * 64 * 2 + nvalid * DVH * 4);
          for (int a = 0; a < KATOMS; ++a) tc::tma_load_3d(sm.k[s][a], &tm_k, &sm.bar_full[s], a * 64, j * CF_BN, bn);
          bulk_g2s(sm.vt[s], v + ((size_t)bn * L + (size_t)j * CF_BN) * DVH, nvalid * DVH * 4, &sm.bar_full[s]);
        }
      }
    }
  } else if (warp == CF_W_S) {
    const int nks = C1 >> 4;
    switch (nks) {      // dispatched once, outside the loops
      case 1: cf_score_loop<KATOMS, 1>(sm, tmem, ntiles, my_items); break;
      case 2: cf_score_loop<KATOMS, 2>(sm, tmem, ntiles, my_items); break;
      case 3: cf_score_loop<KATOMS, 3>(sm, tmem, ntiles, my_items); break;
      case 4: cf_score_loop<KATOMS, 4>(sm, tmem, ntiles, my_items); break;
      case 5: cf_score_loop<KATOMS, 5>(sm, tmem, ntiles, my_items); break;
      case 6: cf_score_loop<KATOMS, 6>(sm, tmem, ntiles, my_items); break;
      case 7: cf_score_loop<KATOMS, 7>(sm, tmem, ntiles, my_items); break;
      case 8: cf_score_loop<KATOMS, 8>(sm, tmem, ntiles, my_items); break;
      case 9: cf_score_loop<KATOMS, 9>(sm, tmem, ntiles, my_items); break;
      case 10: cf_score_loop<KATOMS, 10>(sm, tmem, ntiles, my_items); break;
      default: cf_score_loop<KATOMS, 11>(sm, tmem, ntiles, my_items); break;
    }
  } else {
    // ===================== softmax warpgroups (thread == query row == TMEM lane) =====================
    const int wg = warp >> 2;
    const int rowi = (warp & 3) * 32 + lane;
    const uint32_t tlane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    auto stage_q = [&](int it) {                      // WG0: Q tile of item `it` -> its TMEM buffer
      tc::mbar_wait(&sm.bar_q, it & 1);
      stationary_to_tmem<KATOMS>(sm.q, tlane + (uint32_t)((it & (QB - 1)) * KATOMS * 32), rowi);
      tc::mbar_arrive(&sm.bar_a_ready);
      tc::mbar_arrive(&sm.bar_q_free);
    };
    if (wg == 0) stage_q(0);
    uint32_t r[2][32];
    Ring rst, rsl;
    int tcur = 0;                                     // global tile index the rings stand at
    for (int it = 0; it < my_items; ++it) {
      const int item = blockIdx.x + it * gridDim.x, bn = item / nqt, qt = item - bn * nqt, q0 = qt * CF_BM;
      float m = -INFINITY, l = 0.f, acc[DVH];
#pragma unroll
      for (int e = 0; e < DVH; ++e) acc[e] = 0.f;
      // GLOBAL tile t belongs to warpgroup t % 3, so a warpgroup meets a given score slot at a fixed stride and observes its
      // barrier phases in order (an item-dependent map let a warpgroup jump 4-5 tiles at an item boundary and mistake
      // an unfinished phase for a finished one: parity waits only tell neighbours apart).  Inside the item the warpgroup
      // therefore owns the tiles of ONE class j % 3 = cls; partial results are stored and merged BY CLASS, in class order,
      // so the output does not depend on where or when the item runs (batch independence bit for bit).
      const int cls = (wg + CF_NWG - (it * ntiles) % CF_NWG) % CF_NWG;
      for (int j = cls; j < ntiles; j += CF_NWG) {
        for (const int t = it * ntiles + j; tcur < t; ++tcur) { rst.next(ST); rsl.next(NS); }
        const int slot = rsl.i, st = rst.i;
        const uint32_t tslot = tlane + COL_SLOT0 + 128 * slot;
        const int nvalid = L - j * CF_BN;           // >= CF_BN for every tile but (possibly) the last
        const uint32_t vt = smem_u32(sm.vt[st]);
        tc::mbar_wait(&sm.bar_s_full[slot], rsl.ph);
        tc::tc_fence_after();
        tc::tmem_ld_x32(tslot + 0, r[0]);
        tc::tmem_ld_x32(tslot + 32, r[1]);
        tc::tmem_ld_wait();
        if (dbg & 8) l += __uint_as_float(r[0][0]);
        else if (nvalid < 64) fwd_cc_half<DVH, true>(r, vt, nvalid, m, l, acc);
        else fwd_cc_half<DVH, false>(r, vt, nvalid, m, l, acc);
        tc::tmem_ld_x32(tslot + 64, r[0]);
        tc::tmem_ld_x32(tslot + 96, r[1]);
        tc::tmem_ld_wait();
        tc::tc_fence_before();
        tc::mbar_arrive(&sm.bar_slot_free[slot]);   // all scores of the tile have been read: the slot can be refilled
        if (dbg & 8) l += __uint_as_float(r[0][0]);
        else if (nvalid < CF_BN) { if (nvalid > 64) fwd_cc_half<DVH, true>(r, vt + 64 * DVH * 4, nvalid - 64, m, l, acc); }
        else fwd_cc_half<DVH, false>(r, vt + 64 * DVH * 4, nvalid - 64, m, l, acc);
        tc::mbar_arrive(&sm.bar_empty[st]);          // value tile consumed
      }
      // the next item's Q tile goes to TMEM as early as possible: with two buffers right away (the score issuer then
      // runs ahead while the warpgroups merge), with one buffer after the item's last score MMA
      if (wg == 0 && it + 1 < my_items) {
        if (QB == 1) { tc::mbar_wait(&sm.bar_final, it & 1); tc::tc_fence_after(); }
        stage_q(it + 1);
      }
      // ---- merge the warpgroups' partial results ----
      float(*xch)[CF_BM][4] = sm.xch[it & 1];
      {
        float* x = xch[cls][rowi];
        x[0] = m;
        x[1] = l;
#pragma unroll
        for (int e = 0; e < DVH; ++e) x[2 + e] = acc[e];
      }
      asm volatile("bar.sync 1, %0;" ::"n"(128 * CF_NWG) : "memory");
      if (wg == 0) {
        float mm = -INFINITY;
#pragma unroll
        for (int g = 0; g < CF_NWG; ++g) mm = fmaxf(mm, xch[g][rowi][0]);
        float lt = 0.f, ot[DVH];
#pragma unroll
        for (int e = 0; e < DVH; ++e) ot[e] = 0.f;
#pragma unroll
        for (int g = 0; g < CF_NWG; ++g) {            // classes in order 0, 1, 2
          const float mg = xch[g][rowi][0];
          const float ag = (mg == -INFINITY) ? 0.f : tc::ex2f(mg - mm);
          lt = fmaf(ag, xch[g][rowi][1], lt);
#pragma unroll
          for (int e = 0; e < DVH; ++e) ot[e] = fmaf(ag, xch[g][rowi][2 + e], ot[e]);
        }
        const int qi = q0 + rowi;
        if (qi < L) {
          const float inv = 1.f / lt;
          const size_t row = (size_t)bn * L + qi;
#pragma unroll
          for (int e = 0; e < DVH; ++e) o[row * DVH + e] = ot[e] * inv;
          lse[row] = (mm + log2f(lt)) * 0.6931471805599453f;
        }
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == CF_W_S) tc::tmem_dealloc<512>(tmem);
}

// ================================================================================================
// backward
// ================================================================================================
constexpr int CB_BM = 128, CB_BN = 64, CB_MAXSLOTS = 7;
// three math warpgroups (global tile t -> warpgroup t % 3): three warps per scheduler keep the MUFU pipe busy while the others sit
// in TMEM load / store / barrier latencies;  then one TMA warp, the score-MMA issuer (+TMEM alloc) and the gradient-MMA issuer
// (warp CB_W_G), and TWO score-MMA issuers (CB_W_S even global tiles + TMEM alloc, CB_W_S2 odd ones): the timeline showed a
// single score issuer busy back to back (~600 cycles of waits + issue per tile) with every warpgroup waiting on it
constexpr int CB_NWG = 3, CB_W_TMA = 4 * CB_NWG, CB_W_S = CB_W_TMA + 1, CB_W_G = CB_W_TMA + 2, CB_W_S2 = CB_W_TMA + 3,
              CB_THREADS = 32 * (CB_W_S2 + 1);
// Streamed-tile stages.  A stage is held from its TMA issue until the tile's GRADIENT MMA has completed (~3.5 tiles of
// pipeline), so the prefetch lead is ST - 4.5 tiles; with 6 stages the score issuer waited 400-900 cycles per tile for the
// K tile to land (timeline).  The dQa kernel also holds a 24-88 KB staging tile (sized by OUTW >= KD), the dK/dV kernel does not.
template <int KATOMS, int OUT_FLOATS, int NSTAT = 1> struct CbStages {   // as many as fit beside the stationary tile(s) and the staging tile
  static constexpr int fixed = 1024 /*alignment slack*/ + (NSTAT > 1 ? 8192 : 4096) /*side rows, barriers*/ + (NSTAT > 1 ? 4096 : 2048) /*static dV exchange*/;
  static constexpr int avail = 232448 - fixed - NSTAT * KATOMS * CB_BM * 128 - OUT_FLOATS * 4;
  static constexpr int fit = avail / (KATOMS * CB_BN * 128);
  static constexpr int value = fit > 10 ? 10 : fit;
  static_assert(value >= 3, "not enough shared memory for three streamed stages");
};

// TMEM plan of a backward kernel whose accumulator needs ACC columns: QB stationary buffers, NS score slots of 64 columns
// The pipeline is latency-bound by (tiles in flight) / (S' MMA + TMEM round trip + math + gradient MMA ~ 2700 cycles), i.e. by
// the number of score slots: the stationary operand gets ONE buffer (it is refilled right after the item's last score MMA,
// which is when a second buffer would have been filled too) and every remaining column goes to slots.
// Phase-parity invariant of the two score issuers: with an odd stage count a stage alternates between the issuers, so each
// of them skips every other phase of bar_full[stage] and a parity wait cannot tell phase u from u+2.  It is still exact
// as long as the skipped phase (the other issuer's tile t+ST) is complete before the issuer reaches tile t+2*ST, which its
// slot wait (gradient MMA of tile t+2*ST-NS done) guarantees iff ST >= NS.  Hence NS <= ST for odd ST (an even ST keeps
// every stage with one issuer).  The 512-pixel dQa kernel (3 stages) deadlocked with 4 slots before this rule.
// Two score issuers when there are enough stages for both to have a tile in flight; one otherwise.
// (and an item of a single tile would leave one issuer without a commit on bar_s_done for that item)
__host__ __device__ constexpr int cb_issuers(int stages, int ntiles) { return (stages >= 4 && ntiles >= 2) ? 2 : 1; }
struct CbPlan { int QB, NS; uint32_t col_slot0, col_acc; };
// qb = 1: the stationary operand lives in TMEM (TS-mode score MMAs, at most 5 slots); qb = 0: it stays in shared memory
// (SS-mode, double-buffered by item parity) and its columns become score slots
__device__ __forceinline__ CbPlan cb_plan(int katoms, int acc_cols, int stages, int ntiles, int qb = 1) {
  CbPlan p;
  p.QB = qb;
  p.NS = min(qb ? 5 : CB_MAXSLOTS, (512 - p.QB * katoms * 32 - acc_cols) / 64);
  if (stages & 1) p.NS = min(p.NS, stages);
  // Math warpgroups: global tile t belongs to warpgroup t % 3, so before waiting for S'(t) on slot t % NS a warpgroup has
  // seen S'(t-3) complete; the slot's previous phase is S'(t-NS).  With ONE issuer the score MMAs complete in order and
  // NS >= 3 suffices; with TWO issuers (even / odd tiles) t-NS and t-3 must come from the same issuer, i.e. NS must be odd
  // (3 or 5).  NS = 4 with two issuers (512-px dQa kernel with 4 stages) let a warpgroup run ahead of the lagging issuer.
  if (cb_issuers(stages, ntiles) == 2 && !(p.NS & 1)) p.NS -= 1;
  p.col_slot0 = p.QB * katoms * 32;
  p.col_acc = p.col_slot0 + 64 * p.NS;
  return p;
}

template <int KATOMS, int SIDE_FLOATS, int OUT_FLOATS, int ROW_FLOATS, int NSTAT = 1>
struct __align__(1024) CbSmem {
  static constexpr int ST = CbStages<KATOMS, OUT_FLOATS, NSTAT>::value;
  static constexpr int NST = NSTAT;
  bf16 stat[NSTAT * KATOMS][CB_BM * 64];         // NSTAT = 2 (SS mode): buffer (item parity) * KATOMS + atom
  bf16 strm[ST][KATOMS][CB_BN * 64];
  float side[ST][SIDE_FLOATS];                 // fp32 side tile: v (dq kernel) or dO | delta (dkv kernel)
  float rowside[2][CB_BM * ROW_FLOATS];        // fp32 rows of the stationary tile (dO | delta, or v), by item parity
  float out[OUT_FLOATS > 0 ? OUT_FLOATS : 4];  // accumulator staging for the bulk store (dq kernel)
  uint64_t bar_stat, bar_stat_free, bar_a_ready, bar_s_done, bar_final, bar_acc_free, bar_dv, bar_full[ST], bar_empty[ST];
  uint64_t bar_s_full[CB_MAXSLOTS], bar_p_ready[CB_MAXSLOTS], bar_slot_free[CB_MAXSLOTS];
  uint32_t tmem_base;
};

// CTA set-up.  The TMA lane initialises the barriers itself and issues the first stationary-tile load right away, so
// that its latency runs under the TMEM allocation and the CTA-wide sync instead of after them.
// stationary tile of item (bn, row0) + its fp32 row data (r0: RW0 floats per row, r1: RW1 floats per row or NULL) -> bar_stat
template <int KATOMS, class Smem>
__device__ __forceinline__ void cb_load_stat(Smem& sm, const CUtensorMap* m_stat, const float* r0, int RW0, const float* r1, int RW1,
                                             int L, int bn, int row0, int parity) {
  const int nrows = min(CB_BM, L - row0);
  const size_t g0 = (size_t)bn * L + row0;
  tc::mbar_arrive_expect_tx(&sm.bar_stat, KATOMS * CB_BM * 64 * 2 + nrows * (RW0 + RW1) * 4);
  const int sb = (Smem::NST > 1 ? (parity & 1) : 0) * KATOMS;
  for (int a = 0; a < KATOMS; ++a) tc::tma_load_3d(sm.stat[sb + a], m_stat, &sm.bar_stat, a * 64, row0, bn);
  bulk_g2s(sm.rowside[parity], r0 + g0 * RW0, nrows * RW0 * 4, &sm.bar_stat);
  if (RW1) bulk_g2s(sm.rowside[parity] + CB_BM * RW0, r1 + g0 * RW1, nrows * RW1 * 4, &sm.bar_stat);
}

template <int KATOMS, class Smem>
__device__ __forceinline__ void cb_init(Smem& sm, int warp, int lane, const CUtensorMap* m_stat, const CUtensorMap* m_strm, int nqt,
                                        const float* r0, int RW0, const float* r1, int RW1, int L) {
  if (warp == CB_W_TMA && lane == 0) {
    tc::mbar_init(&sm.bar_stat, 1);
    tc::mbar_init(&sm.bar_stat_free, 128 * CB_NWG);   // every math thread has read its row data (WG0: and moved the tile to TMEM)
    tc::mbar_init(&sm.bar_a_ready, 128);
    tc::mbar_init(&sm.bar_s_done, cb_issuers(Smem::ST, (L + CB_BN - 1) / CB_BN));   // every score issuer commits its last tile of the item
    tc::mbar_init(&sm.bar_final, 1);
    tc::mbar_init(&sm.bar_acc_free, 128);             // warpgroup 0 drains the accumulator
    tc::mbar_init(&sm.bar_dv, 128 * CB_NWG);
    for (int s = 0; s < Smem::ST; ++s) { tc::mbar_init(&sm.bar_full[s], 1); tc::mbar_init(&sm.bar_empty[s], 129); }
    for (int s = 0; s < CB_MAXSLOTS; ++s) {
      tc::mbar_init(&sm.bar_s_full[s], 1);
      tc::mbar_init(&sm.bar_p_ready[s], 128);
      tc::mbar_init(&sm.bar_slot_free[s], 1);
    }
    tc::fence_barrier_init();
    const int item = blockIdx.x, bn = item / nqt, row0 = (item - bn * nqt) * CB_BM;
    cb_load_stat<KATOMS>(sm, m_stat, r0, RW0, r1, RW1, L, bn, row0, 0);
    tc::tma_prefetch_desc(m_strm);
  }
  if (warp == CB_W_S) tc::tmem_alloc<512>(&sm.tmem_base);
  tc::tc_fence_before();
  __syncthreads();
  tc::tc_fence_after();
}

// TMA producer of both backward kernels: per item the stationary tile (once its staging buffer is free), then the streamed
// tiles with their fp32 side rows (side0: SW0 floats per row, side1: SW1 floats per row or NULL)
template <int KATOMS, class Smem>
__device__ __forceinline__ void cb_producer(Smem& sm, const CUtensorMap* m_stat, const CUtensorMap* m_strm, const float* side0,
                                            int SW0, const float* side1, int SW1, const float* r0, int RW0, const float* r1, int RW1,
                                            int L, int nqt, int ntiles, int my_items, int dbg, long long* tl = nullptr) {
  Ring rg;
  // the next item's stationary tile is requested half-way through the item: by then every warpgroup has started the item
  // (bar_stat_free), so this wait never holds up the tile stream, and the tile still lands long before it is needed
  const int jq = ntiles / 2;
  for (int it = 0; it < my_items; ++it) {
    const int item = blockIdx.x + it * gridDim.x, bn = item / nqt;
    for (int j = 0; j < ntiles; ++j, rg.next(Smem::ST)) {
      if (j == jq && it + 1 < my_items) {              // next item's stationary tile: the staging buffer is free once WG0
        const int nitem = item + gridDim.x, nbn = nitem / nqt, nrow0 = (nitem - nbn * nqt) * CB_BM;   // has moved this item's to TMEM
        tc::hb(1, it * 1000 + j);
        tc::mbar_wait(&sm.bar_stat_free, it & 1);
        if (Smem::NST > 1 && it > 0) tc::mbar_wait(&sm.bar_s_done, (it - 1) & 1);   // SS mode: item it-1's score MMAs have read stat[(it+1)&1]
        tc::hb(1, 500000 + it * 1000 + j);
        cb_load_stat<KATOMS>(sm, m_stat, r0, RW0, r1, RW1, L, nbn, nrow0, (it + 1) & 1);
      }
      const int s = rg.i;
      const int nvalid = min(CB_BN, L - j * CB_BN);
      const size_t r0 = (size_t)bn * L + (size_t)j * CB_BN;
      tc::hb(0, it * 1000 + j);
      tc::mbar_wait(&sm.bar_empty[s], rg.ph ^ 1);
      TL_STAMP(tl, 14, it * ntiles + j);
      if ((dbg & 2) && (it > 0 || j >= Smem::ST)) { tc::mbar_arrive(&sm.bar_full[s]); continue; }     // ablation: no global traffic
      tc::mbar_arrive_expect_tx(&sm.bar_full[s], KATOMS * CB_BN * 64 * 2 + nvalid * (SW0 + SW1) * 4);
      for (int a = 0; a < KATOMS; ++a) tc::tma_load_3d(sm.strm[s][a], m_strm, &sm.bar_full[s], a * 64, j * CB_BN, bn);
      bulk_g2s(sm.side[s], side0 + r0 * SW0, nvalid * SW0 * 4, &sm.bar_full[s]);
      if (SW1) bulk_g2s(sm.side[s] + CB_BN * SW0, side1 + r0 * SW1, nvalid * SW1 * 4, &sm.bar_full[s]);
    }
  }
}

template <int KATOMS, int NKS, class Smem>
__device__ __forceinline__ void cb_score_loop(Smem& sm, uint32_t tmem, CbPlan pl, int ntiles, int my_items, int sidx, long long* tl) {
  const int nstep = cb_issuers(Smem::ST, ntiles);  // tiles sidx, sidx + nstep, ...
  if (sidx >= nstep) return;
  constexpr uint32_t idesc_s = tc::idesc_bf16_f32(CB_BM, CB_BN);
  constexpr uint32_t STRM_ATOM = (CB_BN * 128) >> 4, STAGE = KATOMS * STRM_ATOM;
  const uint32_t strm_lo = tc::desc_lo_k(smem_u32(sm.strm[0][0]));
  const int NS = pl.NS, total = my_items * ntiles;
  Ring rst, rsl;
  for (int i = 0; i < sidx; ++i) { rst.next(Smem::ST); rsl.next(NS); }
  int it = 0, j = sidx, a_it = -1;
  uint32_t a_tmem = tmem, a_smem = 0;
  constexpr uint32_t STAT_ATOM = (CB_BM * 128) >> 4;
  for (int t = sidx; t < total; t += nstep) {
    while (j >= ntiles) { j -= ntiles; ++it; }
    if (it != a_it) {                              // first tile of an item for this issuer: its stationary operand is in TMEM
      if (Smem::NST > 1) {                           // (SS mode: in shared memory buffer it & 1, landed with bar_stat)
        tc::mbar_wait(&sm.bar_stat, it & 1);
        a_smem = tc::desc_lo_k(smem_u32(sm.stat[(it & 1) * KATOMS]));
      } else {
        tc::mbar_wait(&sm.bar_a_ready, it & 1);
        a_tmem = tmem + (uint32_t)((it & (pl.QB - 1)) * KATOMS * 32);
      }
      a_it = it;
    }
    const int st = rst.i, slot = rsl.i;
    TL_STAMP(tl, 0, t);
    if (lane_id() == 0) tc::hb(2 + sidx, it * 1000 + j);
    tc::mbar_wait(&sm.bar_full[st], rst.ph);
    TL_STAMP(tl, 1, t);
    if (t >= NS) tc::mbar_wait(&sm.bar_slot_free[slot], rsl.ph ^ 1);
    tc::tc_fence_after();
    TL_STAMP(tl, 2, t);
    if (tc::elect_one()) {
      if (Smem::NST > 1) tc::issue_ss_ksteps<NKS, STAT_ATOM, STRM_ATOM>(tmem + pl.col_slot0 + 64 * slot, a_smem, strm_lo + st * STAGE, idesc_s);
      else tc::issue_ts_ksteps<NKS, 0, STRM_ATOM>(tmem + pl.col_slot0 + 64 * slot, 0u, a_tmem, strm_lo + st * STAGE, idesc_s);
      tc::mma_commit(&sm.bar_s_full[slot]);
      if (j + nstep >= ntiles) tc::mma_commit(&sm.bar_s_done);   // this issuer's last tile of the item
    }
    __syncwarp();
    if (lane_id() == 0) tc::hb(2 + sidx, 500000 + it * 1000 + j);
    TL_STAMP(tl, 3, t);
    j += nstep;
    for (int i = 0; i < nstep; ++i) { rst.next(Smem::ST); rsl.next(NS); }
  }
}
// score-MMA issuer shared by both backward kernels: S'(t) -> slot t % NS as soon as the K/Q tile has landed and the
// slot's previous gradient MMAs are done.  The k-step count is dispatched ONCE, outside the loops (an indirect
// branch per tile costs hundreds of cycles on the issuing warp, which is the critical resource).
template <int KATOMS, class Smem>
__device__ __forceinline__ void cb_score_issuer(Smem& sm, uint32_t tmem, CbPlan pl, int nks, int ntiles, int my_items, int sidx,
                                                long long* tl = nullptr) {
  switch (nks) {
    case 1: cb_score_loop<KATOMS, 1>(sm, tmem, pl, ntiles, my_items, sidx, tl); break;
    case 2: cb_score_loop<KATOMS, 2>(sm, tmem, pl, ntiles, my_items, sidx, tl); break;
    case 3: cb_score_loop<KATOMS, 3>(sm, tmem, pl, ntiles, my_items, sidx, tl); break;
    case 4: cb_score_loop<KATOMS, 4>(sm, tmem, pl, ntiles, my_items, sidx, tl); break;
    case 5: cb_score_loop<KATOMS, 5>(sm, tmem, pl, ntiles, my_items, sidx, tl); break;
    case 6: cb_score_loop<KATOMS, 6>(sm, tmem, pl, ntiles, my_items, sidx, tl); break;
    case 7: cb_score_loop<KATOMS, 7>(sm, tmem, pl, ntiles, my_items, sidx, tl); break;
    case 8: cb_score_loop<KATOMS, 8>(sm, tmem, pl, ntiles, my_items, sidx, tl); break;
    case 9: cb_score_loop<KATOMS, 9>(sm, tmem, pl, ntiles, my_items, sidx, tl); break;
    case 10: cb_score_loop<KATOMS, 10>(sm, tmem, pl, ntiles, my_items, sidx, tl); break;
    default: cb_score_loop<KATOMS, 11>(sm, tmem, pl, ntiles, my_items, sidx, tl); break;
  }
}

// gradient-MMA issuer shared by both backward kernels: acc (+)= dS(t)[TMEM slot] . streamed tile (MN-major view), N = n_acc
template <int KATOMS, class Smem>
__device__ __forceinline__ void cb_grad_issuer(Smem& sm, uint32_t tmem, CbPlan pl, uint32_t idesc, int ntiles, int my_items, int dbg,
                                               long long* tl = nullptr) {
  constexpr uint32_t STRM_ATOM = (CB_BN * 128) >> 4, STAGE = KATOMS * STRM_ATOM;
  const uint32_t b_lo = tc::desc_lo_mn(smem_u32(sm.strm[0][0]), CB_BN * 128);
  const int NS = pl.NS;
  Ring rst, rsl;
  for (int it = 0; it < my_items; ++it) {
    for (int jj = 0; jj < ntiles; ++jj, rst.next(Smem::ST), rsl.next(NS)) {
      const int st = rst.i, slot = rsl.i;
      const uint32_t tslot = tmem + pl.col_slot0 + 64 * slot;
      TL_STAMP(tl, 4, it * ntiles + jj);
      if (lane_id() == 0) tc::hb(4, it * 1000 + jj);
      tc::mbar_wait(&sm.bar_p_ready[slot], rsl.ph);
      if (jj == 0 && it > 0) tc::mbar_wait(&sm.bar_acc_free, (it - 1) & 1);   // previous item's accumulator has been drained
      tc::tc_fence_after();
      TL_STAMP(tl, 5, it * ntiles + jj);
      if (tc::elect_one()) {
        const uint32_t bb = b_lo + st * STAGE;
#pragma unroll
        for (int ks = 0; ks < CB_BN / 16; ++ks)
          if (!(dbg & 4) || jj == 0) tc::mma_ts(tmem + pl.col_acc, tslot + ks * 8, tc::desc64(bb + ks * 128), idesc, (jj > 0 || ks > 0) ? 1u : 0u);
        tc::mma_commit(&sm.bar_empty[st]);
        tc::mma_commit(&sm.bar_slot_free[slot]);
        if (jj == ntiles - 1) tc::mma_commit(&sm.bar_final);
      }
      __syncwarp();
      if (lane_id() == 0) tc::hb(4, 500000 + it * 1000 + jj);
      TL_STAMP(tl, 6, it * ntiles + jj);
    }
  }
}

// 32 keys (chunk C of a 64-key tile) of the dQa kernel: dS = 2^S' (dO.v[k] - delta) for this thread's query row, packed to bf16
template <int DVH, bool TAIL, int C>
__device__ __forceinline__ void dq_cc_chunk(const uint32_t (&rs)[32], uint32_t (&pd)[32], uint32_t vt, int nvalid,
                                            const float (&go)[DVH], float ndelta) {
#pragma unroll
  for (int i = 0; i < 32; i += 4) {
    float vv[4 * DVH];
#pragma unroll
    for (int u = 0; u < DVH; ++u) {
      const float4 t4 = lds128(vt + ((C * 32 + i) * DVH + 4 * u) * 4);
      vv[4 * u] = t4.x; vv[4 * u + 1] = t4.y; vv[4 * u + 2] = t4.z; vv[4 * u + 3] = t4.w;
    }
    float ds[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      float dp = ndelta;
#pragma unroll
      for (int e = 0; e < DVH; ++e) dp = fmaf(go[e], vv[u * DVH + e], dp);
      ds[u] = tc::ex2_mixed(__uint_as_float(rs[i + u]), u) * dp;
      if (TAIL && C * 32 + i + u >= nvalid) ds[u] = 0.f;     // zero-filled keys past L
    }
    pd[C * 16 + (i >> 1)] = tc::pack_bf16x2(ds[0], ds[1]);
    pd[C * 16 + (i >> 1) + 1] = tc::pack_bf16x2(ds[2], ds[3]);
  }
}

// 32 queries (chunk C of a 64-query tile) of the dK/dV kernel for this thread's key row: p = 2^S'^T, dV += p dO[q] (registers),
// dS^T = p (dO[q].v - delta[q])
template <int DVH, bool TAIL, int C>
__device__ __forceinline__ void dkv_cc_chunk(const uint32_t (&rs)[32], uint32_t (&pd)[32], uint32_t dot, uint32_t dlt, int nvalid,
                                             const float (&vk)[DVH], float (&dvacc)[DVH]) {
#pragma unroll
  for (int i = 0; i < 32; i += 4) {
    float gg[4 * DVH];
#pragma unroll
    for (int u = 0; u < DVH; ++u) {
      const float4 t4 = lds128(dot + ((C * 32 + i) * DVH + 4 * u) * 4);
      gg[4 * u] = t4.x; gg[4 * u + 1] = t4.y; gg[4 * u + 2] = t4.z; gg[4 * u + 3] = t4.w;
    }
    const float4 dl = lds128(dlt + (C * 32 + i) * 4);
    const float dls[4] = {dl.x, dl.y, dl.z, dl.w};
    float ds[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      float dp = -dls[u];
#pragma unroll
      for (int e = 0; e < DVH; ++e) dp = fmaf(gg[u * DVH + e], vk[e], dp);
      float p = tc::ex2_mixed(__uint_as_float(rs[i + u]), u);
      const bool dead = TAIL && C * 32 + i + u >= nvalid;    // zero-filled queries past L: the side tile holds stale data there
      if (dead) { p = 0.f; dp = 0.f; }
#pragma unroll
      for (int e = 0; e < DVH; ++e) dvacc[e] = fmaf(p, dead ? 0.f : gg[u * DVH + e], dvacc[e]);
      ds[u] = p * dp;
    }
    pd[C * 16 + (i >> 1)] = tc::pack_bf16x2(ds[0], ds[1]);
    pd[C * 16 + (i >> 1) + 1] = tc::pack_bf16x2(ds[2], ds[3]);
  }
}

// ---- query-stationary: dQa ------------------------------------------------------------------------
// TMEM: Qa buffers [0, QB*32K); slot s: S' at col_slot0 + 64 s (dS, bf16, over its first 32 columns); dQa behind the slots.
template <int KATOMS, int DVH, int OUTW>
__global__ void __launch_bounds__(CB_THREADS, 1) attn_bwd_dq_cc_kernel(
    const __grid_constant__ CUtensorMap tm_q_stat, const __grid_constant__ CUtensorMap tm_k_strm,
    const float* __restrict__ v, const float* __restrict__ d_o, const float* __restrict__ delta, float* __restrict__ dqa, int L,
    int KD, int NQ, int C1, int nqt, int nitems, int dbg, long long* __restrict__ tl_buf) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  typedef CbSmem<KATOMS, CB_BN * DVH, CB_BM * OUTW, DVH + 1> Smem;
  Smem& sm = *reinterpret_cast<Smem*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int ST = Smem::ST;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ntiles = (L + CB_BN - 1) / CB_BN;
  const int my_items = (nitems - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const CbPlan pl = cb_plan(KATOMS, NQ, ST, ntiles);
  // clock timeline of one CTA (tools/attn_timeline.py): lane 0 of the issuing warps and of each warpgroup's first warp
  long long* const tl = (tl_buf != nullptr && blockIdx.x == TL_CTA && lane == 0) ? tl_buf : nullptr;

  cb_init<KATOMS>(sm, warp, lane, &tm_q_stat, &tm_k_strm, nqt, d_o, DVH, delta, 1, L);
  const uint32_t tmem = sm.tmem_base;

  if (warp == CB_W_TMA) {
    if (lane == 0)
      cb_producer<KATOMS>(sm, &tm_q_stat, &tm_k_strm, v, DVH, nullptr, 0, d_o, DVH, delta, 1, L, nqt, ntiles, my_items, dbg, tl);
  } else if (warp == CB_W_S || warp == CB_W_S2) {
    cb_score_issuer<KATOMS>(sm, tmem, pl, C1 >> 4, ntiles, my_items, warp == CB_W_S ? 0 : 1, warp == CB_W_S ? tl : nullptr);
  } else if (warp == CB_W_G) {
    cb_grad_issuer<KATOMS>(sm, tmem, pl, tc::idesc_bf16_f32(CB_BM, NQ) | (1u << 16), ntiles, my_items, dbg, tl);
  } else {
    const int wg = warp >> 2;
    const int rowi = (warp & 3) * 32 + lane;
    const uint32_t tlane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const int NS = pl.NS;
    auto stage_stat = [&](int it) {                   // WG0: stationary tile of item `it` -> its TMEM buffer
      tc::mbar_wait(&sm.bar_stat, it & 1);
      stationary_to_tmem<KATOMS>(sm.stat, tlane + (uint32_t)((it & (pl.QB - 1)) * KATOMS * 32), rowi);
      tc::mbar_arrive(&sm.bar_a_ready);
    };
    if (wg == 0) stage_stat(0);
    uint32_t rs[2][32], pd[32];
    Ring rst, rsl;
    int tcur = 0;                                     // global tile index the rings stand at
    const bool bulk_out = (KD & 3) == 0 && !(dbg & 32);
    for (int it = 0; it < my_items; ++it) {
      const int item = blockIdx.x + it * gridDim.x, bn = item / nqt, qt = item - bn * nqt, q0 = qt * CB_BM;
      const int qi = q0 + rowi;
      const size_t row = (size_t)bn * L + qi;
      // this row's dO and delta came with the stationary tile (a global load here would sit on the item's critical path)
      if (wg != 0) tc::mbar_wait(&sm.bar_stat, it & 1);
      float go[DVH], ndelta = 0.f;
      {
        const float* rsd = sm.rowside[it & 1];
#pragma unroll
        for (int e = 0; e < DVH; ++e) go[e] = qi < L ? rsd[rowi * DVH + e] : 0.f;
        if (qi < L) ndelta = -rsd[CB_BM * DVH + rowi];
      }
      tc::mbar_arrive(&sm.bar_stat_free);
      for (int j = (wg + CB_NWG - (it * ntiles) % CB_NWG) % CB_NWG; j < ntiles; j += CB_NWG) {   // global tile t -> warpgroup t % 3
        {
          const int t = it * ntiles + j, dlt = t - tcur;             // 3 inside an item, 1..5 across an item boundary
          if (dlt == CB_NWG && ST >= CB_NWG && NS >= CB_NWG) { rst.advance(CB_NWG, ST); rsl.advance(CB_NWG, NS); }
          else for (int i = 0; i < dlt; ++i) { rst.next(ST); rsl.next(NS); }
          tcur = t;
        }
        const int slot = rsl.i, st = rst.i;
        const uint32_t tslot = tlane + pl.col_slot0 + 64 * slot;
        const int nvalid = L - j * CB_BN;
        const bool tail = nvalid < CB_BN;
        long long* const tw = (warp & 3) == 0 ? tl : nullptr;
        TL_STAMP(tw, 7, it * ntiles + j);
        if (lane == 0) tc::hb(8 + warp, it * 1000 + j);
        tc::mbar_wait(&sm.bar_s_full[slot], rsl.ph);
        tc::tc_fence_after();
        TL_STAMP(tw, 8, it * ntiles + j);
        // S' leaves TMEM in two 32-column chunks: the second load is in flight while the first chunk is exponentiated
        tc::tmem_ld_x32(tslot, rs[0]);
        tc::tmem_ld_wait();
        tc::tmem_ld_landed(rs[0]);
        tc::tmem_ld_x32(tslot + 32, rs[1]);
        TL_STAMP(tw, 9, it * ntiles + j);
        const uint32_t vt = smem_u32(sm.side[st]);
        if (dbg & 9) {
          tc::tmem_ld_wait();
          tc::tmem_ld_landed(rs[1]);
          if (dbg & 8) {
#pragma unroll
            for (int i = 0; i < 32; ++i) pd[i] = rs[0][i];
          } else {
#pragma unroll
            for (int i = 0; i < 32; ++i) pd[i] = tc::pack_bf16x2(__uint_as_float(rs[0][i]) * ndelta, __uint_as_float(rs[1][i]) * go[0]);
          }
        } else {
          if (tail) dq_cc_chunk<DVH, true, 0>(rs[0], pd, vt, nvalid, go, ndelta);
          else dq_cc_chunk<DVH, false, 0>(rs[0], pd, vt, nvalid, go, ndelta);
          tc::tmem_ld_wait();
          tc::tmem_ld_landed(rs[1]);
          if (tail) dq_cc_chunk<DVH, true, 1>(rs[1], pd, vt, nvalid, go, ndelta);
          else dq_cc_chunk<DVH, false, 1>(rs[1], pd, vt, nvalid, go, ndelta);
        }
        TL_STAMP(tw, 10, it * ntiles + j);
        tc::tmem_st_x32(tslot, pd);                    // dS (bf16) over S'[0,32): all of S' is in registers
        tc::tmem_st_wait();
        tc::tc_fence_before();
        tc::mbar_arrive(&sm.bar_p_ready[slot]);
        tc::mbar_arrive(&sm.bar_empty[st]);            // value tile consumed
        if (lane == 0) tc::hb(8 + warp, 500000 + it * 1000 + j);
        TL_STAMP(tw, 11, it * ntiles + j);
      }
      // ---- drain dQa (warpgroup 0 alone; the others go straight on with the next item's tiles, so the score slots are full
      //      again when the accumulator is released): TMEM -> shared staging tile -> one bulk store of nrows x KD floats ----
      if (wg == 0) {
        TL_STAMP(tl, 12, it * 4 + 0);
        if (lane == 0) tc::hb(24 + warp, 1000 + it);
        if (it + 1 < my_items) {                       // single stationary buffer: refill once the item's score MMAs are done
          tc::mbar_wait(&sm.bar_s_done, it & 1);
          tc::tc_fence_after();
          if (lane == 0) tc::hb(24 + warp, 2000 + it);
          stage_stat(it + 1);
        }
        if (lane == 0) tc::hb(24 + warp, 3000 + it);
        tc::mbar_wait(&sm.bar_final, it & 1);
        tc::tc_fence_after();
        if (lane == 0) tc::hb(24 + warp, 4000 + it);
        TL_STAMP(tl, 12, it * 4 + 1);
        if (bulk_out) {
          if (threadIdx.x == 0) bulk_wait_read();      // the previous item's store has finished reading the staging tile
          asm volatile("bar.sync 1, 128;" ::: "memory");
          for (int c0 = 0; c0 < NQ; c0 += 64) {        // two TMEM loads in flight
            tc::tmem_ld_x32(tlane + pl.col_acc + c0, rs[0]);
            if (c0 + 32 < NQ) tc::tmem_ld_x32(tlane + pl.col_acc + c0 + 32, rs[1]);
            tc::tmem_ld_wait();
#pragma unroll
            for (int h = 0; h < 2; ++h) {
              const uint32_t dst = smem_u32(sm.out + rowi * KD + c0 + 32 * h);
#pragma unroll
              for (int e = 0; e < 32; e += 4)
                if (c0 + 32 * h + e < KD)
                  asm volatile("st.shared.v4.b32 [%0], {%1,%2,%3,%4};" ::"r"(dst + e * 4), "r"(rs[h][e]), "r"(rs[h][e + 1]),
                               "r"(rs[h][e + 2]), "r"(rs[h][e + 3]) : "memory");
            }
          }
          tc::tc_fence_before();
          tc::mbar_arrive(&sm.bar_acc_free);           // the accumulator columns may be overwritten by the next item
          TL_STAMP(tl, 12, it * 4 + 2);
          tc::fence_proxy_async();
          asm volatile("bar.sync 1, 128;" ::: "memory");
          if (threadIdx.x == 0) bulk_s2g(dqa + ((size_t)bn * L + q0) * KD, sm.out, (uint32_t)(min(CB_BM, L - q0) * KD * 4));
          if (lane == 0) tc::hb(24 + warp, 5000 + it);
          TL_STAMP(tl, 12, it * 4 + 3);
        } else {
          for (int c0 = 0; c0 < NQ; c0 += 32) {
            tc::tmem_ld_x32(tlane + pl.col_acc + c0, rs[0]);
            tc::tmem_ld_wait();
            if (qi < L) {
#pragma unroll
              for (int e = 0; e < 32; ++e)
                if (c0 + e < KD) dqa[row * KD + c0 + e] = __uint_as_float(rs[0][e]);
            }
          }
          tc::tc_fence_before();
          tc::mbar_arrive(&sm.bar_acc_free);
        }
      }
    }
    if (threadIdx.x == 0) bulk_wait_read();
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == CB_W_S) tc::tmem_dealloc<512>(tmem);
}

// ---- key-stationary: dK, dV ------------------------------------------------------------------------
// TMEM: Ka buffers [0, QB*32K); slot s: S'^T at col_slot0 + 64 s (dS^T, bf16, over its first 32 columns); dK (32) behind the slots.
// SS = 1: the stationary Ka tile stays in shared memory (SS-mode score MMAs, double-buffered by item parity); its TMEM columns
// become score slots: 7 instead of 5 (the pipeline is bound by tiles in flight / chain latency, see cb_plan).
template <int KATOMS, int DVH, int SS>
__global__ void __launch_bounds__(CB_THREADS, 1) attn_bwd_dkv_cc_kernel(
    const __grid_constant__ CUtensorMap tm_k_stat, const __grid_constant__ CUtensorMap tm_q_strm,
    const float* __restrict__ v, const float* __restrict__ d_o, const float* __restrict__ delta, float* __restrict__ dk,
    float* __restrict__ dv, bf16* __restrict__ dqkvh, int KPq, int nh, int L, int dkh, int C1, int nqt, int nitems) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  typedef CbSmem<KATOMS, CB_BN * (DVH + 1), 0, DVH, SS ? 2 : 1> Smem;
  Smem& sm = *reinterpret_cast<Smem*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
  constexpr int ST = Smem::ST;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ntiles = (L + CB_BN - 1) / CB_BN;
  const int my_items = (nitems - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x;
  const CbPlan pl = cb_plan(KATOMS, 32, ST, ntiles, SS ? 0 : 1);
  __shared__ float dv_xch[2][CB_NWG][CB_BM][DVH];       // dV partial of every tile class (j % 3), by item parity

  cb_init<KATOMS>(sm, warp, lane, &tm_k_stat, &tm_q_strm, nqt, v, DVH, nullptr, 0, L);
  const uint32_t tmem = sm.tmem_base;

  if (warp == CB_W_TMA) {
    if (lane == 0)
      cb_producer<KATOMS>(sm, &tm_k_stat, &tm_q_strm, d_o, DVH, delta, 1, v, DVH, nullptr, 0, L, nqt, ntiles, my_items, 0);
  } else if (warp == CB_W_S || warp == CB_W_S2) {
    cb_score_issuer<KATOMS>(sm, tmem, pl, C1 >> 4, ntiles, my_items, warp == CB_W_S ? 0 : 1);
  } else if (warp == CB_W_G) {
    cb_grad_issuer<KATOMS>(sm, tmem, pl, tc::idesc_bf16_f32(CB_BM, 32) | (1u << 16), ntiles, my_items, 0);
  } else {
    const int wg = warp >> 2;
    const int rowi = (warp & 3) * 32 + lane;
    const uint32_t tlane = tmem + ((uint32_t)((warp & 3) * 32) << 16);
    const int NS = pl.NS;
    auto stage_stat = [&](int it) {
      tc::mbar_wait(&sm.bar_stat, it & 1);
      if (!SS) {
        stationary_to_tmem<KATOMS>(sm.stat, tlane + (uint32_t)((it & (pl.QB - 1)) * KATOMS * 32), rowi);
        tc::mbar_arrive(&sm.bar_a_ready);
      }
    };
    if (wg == 0) stage_stat(0);
    uint32_t rs[2][32], pd[32];
    Ring rst, rsl;
    int tcur = 0;                                        // global tile index the rings stand at
    const float LN2 = 0.6931471805599453f;               // Qa carries log2(e)*q
    for (int it = 0; it < my_items; ++it) {
      const int item = blockIdx.x + it * gridDim.x, bn = item / nqt, qt = item - bn * nqt, k0 = qt * CB_BM;
      const int kj = k0 + rowi;
      const size_t row = (size_t)bn * L + kj;
      if (wg != 0 || SS) tc::mbar_wait(&sm.bar_stat, it & 1);   // this row's v came with the stationary tile
      float vk[DVH], dvacc[DVH];
#pragma unroll
      for (int e = 0; e < DVH; ++e) { vk[e] = kj < L ? sm.rowside[it & 1][rowi * DVH + e] : 0.f; dvacc[e] = 0.f; }
      tc::mbar_arrive(&sm.bar_stat_free);
      // global tile t -> warpgroup t % 3 (see the forward kernel); the dV partials are kept per tile class j % 3 = cls and
      // summed in class order, so they do not depend on where the item runs
      const int cls = (wg + CB_NWG - (it * ntiles) % CB_NWG) % CB_NWG;
      for (int j = cls; j < ntiles; j += CB_NWG) {
        {
          const int t = it * ntiles + j, dlt = t - tcur;             // 3 inside an item, 1..5 across an item boundary
          if (dlt == CB_NWG && ST >= CB_NWG && NS >= CB_NWG) { rst.advance(CB_NWG, ST); rsl.advance(CB_NWG, NS); }
          else for (int i = 0; i < dlt; ++i) { rst.next(ST); rsl.next(NS); }
          tcur = t;
        }
        const int slot = rsl.i, st = rst.i;
        const uint32_t tslot = tlane + pl.col_slot0 + 64 * slot;
        const int nvalid = L - j * CB_BN;
        const bool tail = nvalid < CB_BN;
        tc::mbar_wait(&sm.bar_s_full[slot], rsl.ph);
        tc::tc_fence_after();
        tc::tmem_ld_x32(tslot, rs[0]);
        tc::tmem_ld_wait();
        tc::tmem_ld_landed(rs[0]);
        tc::tmem_ld_x32(tslot + 32, rs[1]);           // in flight under the first chunk's math
        const uint32_t dot = smem_u32(sm.side[st]), dlt = dot + CB_BN * DVH * 4;
        if (tail) dkv_cc_chunk<DVH, true, 0>(rs[0], pd, dot, dlt, nvalid, vk, dvacc);
        else dkv_cc_chunk<DVH, false, 0>(rs[0], pd, dot, dlt, nvalid, vk, dvacc);
        tc::tmem_ld_wait();
        tc::tmem_ld_landed(rs[1]);
        if (tail) dkv_cc_chunk<DVH, true, 1>(rs[1], pd, dot, dlt, nvalid, vk, dvacc);
        else dkv_cc_chunk<DVH, false, 1>(rs[1], pd, dot, dlt, nvalid, vk, dvacc);
        tc::tmem_st_x32(tslot, pd);                    // dS^T (bf16) over S'^T[0,32): all of S'^T is in registers
        tc::tmem_st_wait();
        tc::tc_fence_before();
        tc::mbar_arrive(&sm.bar_p_ready[slot]);
        tc::mbar_arrive(&sm.bar_empty[st]);
      }
      // every warpgroup hands its dV partial over; 1 and 2 go on with the next item, warpgroup 0 finishes this one
#pragma unroll
      for (int e = 0; e < DVH; ++e) dv_xch[it & 1][cls][rowi][e] = dvacc[e];
      tc::mbar_arrive(&sm.bar_dv);
      if (wg > 0) continue;
      if (!SS && it + 1 < my_items) {                  // single stationary TMEM buffer: refill once the item's score MMAs are done
        tc::mbar_wait(&sm.bar_s_done, it & 1);
        tc::tc_fence_after();
        stage_stat(it + 1);
      }
      tc::mbar_wait(&sm.bar_final, it & 1);
      tc::tc_fence_after();
      tc::mbar_wait(&sm.bar_dv, it & 1);
      const int b = bn / nh, n = bn - b * nh;
      bf16* prow = dqkvh ? dqkvh + ((size_t)b * L + kj) * KPq : nullptr;
      tc::tmem_ld_x32(tlane + pl.col_acc, rs[0]);
      tc::tmem_ld_wait();
      tc::tc_fence_before();
      tc::mbar_arrive(&sm.bar_acc_free);               // dK is in registers: the accumulator may be overwritten
      if (kj < L) {
        if (prow) {
          bf16* dst = prow + nh * dkh + n * dkh;
          if (((dkh | KPq) & 3) == 0) {
#pragma unroll
            for (int e = 0; e < 32; e += 4)
              if (e < dkh) {
                uint2 w;
                w.x = tc::pack_bf16x2(__uint_as_float(rs[0][e]) * LN2, __uint_as_float(rs[0][e + 1]) * LN2);
                w.y = tc::pack_bf16x2(__uint_as_float(rs[0][e + 2]) * LN2, __uint_as_float(rs[0][e + 3]) * LN2);
                *reinterpret_cast<uint2*>(dst + e) = w;
              }
          } else {
#pragma unroll
            for (int e = 0; e < 32; ++e)
              if (e < dkh) dst[e] = __float2bfloat16(__uint_as_float(rs[0][e]) * LN2);
          }
        } else {
#pragma unroll
          for (int e = 0; e < 32; ++e)
            if (e < dkh) dk[row * dkh + e] = __uint_as_float(rs[0][e]) * LN2;
        }
#pragma unroll
        for (int e = 0; e < DVH; ++e) {                  // dV: the three class partials in class order
          float t = 0.f;
#pragma unroll
          for (int g = 0; g < CB_NWG; ++g) t += dv_xch[it & 1][g][rowi][e];
          if (prow) prow[2 * nh * dkh + n * DVH + e] = __float2bfloat16(t);
          else dv[row * DVH + e] = t;
        }
      }
    }
  }
  tc::tc_fence_before();
  __syncthreads();
  if (warp == CB_W_S) tc::tmem_dealloc<512>(tmem);
}

int sm_count() {
  static int n = 0;
  if (n == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0)
      n = 148;
  }
  return n;
}

int make_aug_map(const Dims& d, const void* t, int KP, uint32_t box_rows, CUtensorMap* out) {
  const uint64_t dims[3] = {(uint64_t)KP, (uint64_t)d.L, (uint64_t)d.BN};
  const uint64_t strides[2] = {(uint64_t)KP * 2, (uint64_t)d.L * KP * 2};
  const uint32_t box[3] = {64, box_rows, 1};
  return make_tmap_bf16(out, t, 3, dims, strides, box, nullptr);
}

template <int KATOMS, int DVH>
int launch_fwd_cc(const Dims& d, const AugLayout& a, const void* qa, const void* ka, const float* v, float* o, float* lse,
                  cudaStream_t st) {
  CUtensorMap tq, tk;
  AACONV_TRY(make_aug_map(d, qa, a.KP, CF_BM, &tq));
  AACONV_TRY(make_aug_map(d, ka, a.KP, CF_BN, &tk));
  const size_t smem = sizeof(CfSmem<KATOMS, DVH>) + 1024;
  auto kern = attn_fwd_cc_kernel<KATOMS, DVH>;
  AACONV_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  const int nqt = cdiv(d.L, CF_BM), nitems = nqt * d.BN;
  kern<<<std::min(nitems, sm_count()), CF_THREADS, smem, AACONV_ST(st)>>>(tq, tk, v, o, lse, d.L, a.C1, nqt, nitems, g_attn_dbg_mode);
  AACONV_LAUNCH_OK("attn_fwd_cc");
  return 0;
}

template <int KATOMS, int DVH, int OUTW>
int launch_bwd_dq_cc(const Dims& d, const AugLayout& a, const CUtensorMap& tq_stat, const CUtensorMap& tk_strm, const float* v,
                     const float* d_o, const float* delta, float* dqa, int nqt, int nitems, int grid, cudaStream_t st) {
  const size_t smem = sizeof(CbSmem<KATOMS, CB_BN * DVH, CB_BM * OUTW, DVH + 1>) + 1024;
  auto kern = attn_bwd_dq_cc_kernel<KATOMS, DVH, OUTW>;
  AACONV_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  kern<<<grid, CB_THREADS, smem, AACONV_ST(st)>>>(tq_stat, tk_strm, v, d_o, delta, dqa, d.L, a.KD, a.NQ, a.C1, nqt, nitems, g_attn_dbg_mode, g_attn_dbg);
  AACONV_LAUNCH_OK("attn_bwd_dq_cc");
  return 0;
}

// the dQa staging tile is OUTW >= KD floats wide; a narrower one leaves room for one more streamed stage at 3 atoms
template <int KATOMS> struct CcOutw {
  static constexpr int MAX = KATOMS * 64 - 16, MID = KATOMS == 3 ? 152 : MAX;
};

template <int KATOMS, int DVH>
int launch_bwd_cc(const Dims& d, const AugLayout& a, const void* qa, const void* ka, const float* v, const float* d_o,
                  const float* delta, float* dqa, float* dk, float* dv, void* dqkvh, int KPq, cudaStream_t st) {
  CUtensorMap tq_stat, tk_strm, tk_stat, tq_strm;
  AACONV_TRY(make_aug_map(d, qa, a.KP, CB_BM, &tq_stat));
  AACONV_TRY(make_aug_map(d, ka, a.KP, CB_BN, &tk_strm));
  AACONV_TRY(make_aug_map(d, ka, a.KP, CB_BM, &tk_stat));
  AACONV_TRY(make_aug_map(d, qa, a.KP, CB_BN, &tq_strm));
  const int nqt = cdiv(d.L, CB_BM), nitems = nqt * d.BN;
  const int grid = std::min(nitems, sm_count());
  static const bool dkv_ss = [] { const char* e = getenv("AACONV_DKV_SS"); return e ? atoi(e) != 0 : false; }();   // A/B (profiles/r02_attn_ab.md): SS mode measured slower (167 vs 162 us), default off
  if (dkv_ss && KATOMS <= 2) {
    const size_t smem = sizeof(CbSmem<KATOMS, CB_BN * (DVH + 1), 0, DVH, 2>) + 1024;
    auto kern = attn_bwd_dkv_cc_kernel<KATOMS, DVH, 1>;
    AACONV_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, CB_THREADS, smem, AACONV_ST(st)>>>(tk_stat, tq_strm, v, d_o, delta, dk, dv, static_cast<bf16*>(dqkvh), KPq, d.nh, d.L, d.dkh, a.C1,
                                         nqt, nitems);
    AACONV_LAUNCH_OK("attn_bwd_dkv_cc");
  } else {
    const size_t smem = sizeof(CbSmem<KATOMS, CB_BN * (DVH + 1), 0, DVH>) + 1024;
    auto kern = attn_bwd_dkv_cc_kernel<KATOMS, DVH, 0>;
    AACONV_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    kern<<<grid, CB_THREADS, smem, AACONV_ST(st)>>>(tk_stat, tq_strm, v, d_o, delta, dk, dv, static_cast<bf16*>(dqkvh), KPq, d.nh, d.L, d.dkh, a.C1,
                                         nqt, nitems);
    AACONV_LAUNCH_OK("attn_bwd_dkv_cc");
  }
  typedef CcOutw<KATOMS> W;
  if (a.KD <= W::MID) return launch_bwd_dq_cc<KATOMS, DVH, W::MID>(d, a, tq_stat, tk_strm, v, d_o, delta, dqa, nqt, nitems, grid, st);
  return launch_bwd_dq_cc<KATOMS, DVH, W::MAX>(d, a, tq_stat, tk_strm, v, d_o, delta, dqa, nqt, nitems, grid, st);
}

// every kernel one (KATOMS, DVH) instance launches at this KD (forward, dK/dV, dQa) gets its dynamic shared memory next to
// its static shared memory within the per-block limit
template <class Kern>
bool smem_fits(Kern kern, size_t dyn) {
  static int optin = 0;
  if (optin == 0) {
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev) != cudaSuccess)
      optin = 232448;
  }
  cudaFuncAttributes fa;
  if (cudaFuncGetAttributes(&fa, kern) != cudaSuccess) { (void)cudaGetLastError(); return false; }
  return fa.sharedSizeBytes + dyn <= (size_t)optin;
}

template <int KATOMS, int DVH>
bool cc_smem_fits(int KD) {
  typedef CcOutw<KATOMS> W;
  static int ok[2] = {-1, -1};                     // per dQa staging width; the answer does not change within a process
  int& r = ok[KD > W::MID];
  if (r < 0) {
    const bool dq = KD <= W::MID
                        ? smem_fits(attn_bwd_dq_cc_kernel<KATOMS, DVH, W::MID>, sizeof(CbSmem<KATOMS, CB_BN * DVH, CB_BM * W::MID, DVH + 1>) + 1024)
                        : smem_fits(attn_bwd_dq_cc_kernel<KATOMS, DVH, W::MAX>, sizeof(CbSmem<KATOMS, CB_BN * DVH, CB_BM * W::MAX, DVH + 1>) + 1024);
    r = dq && smem_fits(attn_fwd_cc_kernel<KATOMS, DVH>, sizeof(CfSmem<KATOMS, DVH>) + 1024) &&
        smem_fits(attn_bwd_dkv_cc_kernel<KATOMS, DVH, 0>, sizeof(CbSmem<KATOMS, CB_BN * (DVH + 1), 0, DVH>) + 1024);
  }
  return r;
}

}  // namespace

// value width 1..2, 16-byte-aligned fp32 side tiles (L % 4 == 0), and every kernel of the instance within the 227 KB of
// shared memory a block can have (dv/nh = 2 at three operand atoms is not: its dK/dV kernel needs more; the tc kernels run it)
int cc_attn_supported(const Dims& d) {
  if (aug_supported(d)) return AACONV_E_UNSUPPORTED;
  if (d.dvh < 1 || d.dvh > 2 || (d.L & 3)) return AACONV_E_UNSUPPORTED;
  const AugLayout a = aug_layout(d);
  const int K = a.KP / 64;
  const bool fits = d.dvh == 1 ? (K == 1 ? cc_smem_fits<1, 1>(a.KD) : K == 2 ? cc_smem_fits<2, 1>(a.KD) : cc_smem_fits<3, 1>(a.KD))
                               : (K == 1 ? cc_smem_fits<1, 2>(a.KD) : K == 2 ? cc_smem_fits<2, 2>(a.KD) : cc_smem_fits<3, 2>(a.KD));
  if (!fits) return AACONV_E_UNSUPPORTED;
  return 0;
}

// ablation (tools/attn_ablate.py; results are WRONG): AACONV_ABL_NKS = score k-steps, AACONV_ABL_NQ = width of the dQa accumulator
static AugLayout ablated(AugLayout a) {
  if (const char* e = getenv("AACONV_ABL_NKS")) a.C1 = 16 * atoi(e);
  if (const char* e = getenv("AACONV_ABL_NQ")) a.NQ = atoi(e);
  return a;
}

int cc_attn_fwd(const Dims& d, const void* qa, const void* ka, const float* v, float* o, float* lse, cudaStream_t st) {
  AACONV_TRY(cc_attn_supported(d));
  const AugLayout a = ablated(aug_layout(d));
  const int K = a.KP / 64;
  if (d.dvh == 1) {
    if (K == 1) return launch_fwd_cc<1, 1>(d, a, qa, ka, v, o, lse, st);
    if (K == 2) return launch_fwd_cc<2, 1>(d, a, qa, ka, v, o, lse, st);
    return launch_fwd_cc<3, 1>(d, a, qa, ka, v, o, lse, st);
  }
  if (K == 1) return launch_fwd_cc<1, 2>(d, a, qa, ka, v, o, lse, st);
  if (K == 2) return launch_fwd_cc<2, 2>(d, a, qa, ka, v, o, lse, st);
  return launch_fwd_cc<3, 2>(d, a, qa, ka, v, o, lse, st);
}

int cc_attn_bwd(const Dims& d, const void* qa, const void* ka, const float* v, const float* d_o, const float* delta, float* dqa,
                float* dk, float* dv, void* dqkvh, int KPq, cudaStream_t st) {
  AACONV_TRY(cc_attn_supported(d));
  const AugLayout a = ablated(aug_layout(d));
  const int K = a.KP / 64;
  if (d.dvh == 1) {
    if (K == 1) return launch_bwd_cc<1, 1>(d, a, qa, ka, v, d_o, delta, dqa, dk, dv, dqkvh, KPq, st);
    if (K == 2) return launch_bwd_cc<2, 1>(d, a, qa, ka, v, d_o, delta, dqa, dk, dv, dqkvh, KPq, st);
    return launch_bwd_cc<3, 1>(d, a, qa, ka, v, d_o, delta, dqa, dk, dv, dqkvh, KPq, st);
  }
  if (K == 1) return launch_bwd_cc<1, 2>(d, a, qa, ka, v, d_o, delta, dqa, dk, dv, dqkvh, KPq, st);
  if (K == 2) return launch_bwd_cc<2, 2>(d, a, qa, ka, v, d_o, delta, dqa, dk, dv, dqkvh, KPq, st);
  return launch_bwd_cc<3, 2>(d, a, qa, ka, v, d_o, delta, dqa, dk, dv, dqkvh, KPq, st);
}

}  // namespace aaconv
