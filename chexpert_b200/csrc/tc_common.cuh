// sm_100a building blocks: mbarrier, TMA (cp.async.bulk.tensor), tcgen05 (alloc / mma / commit / ld / st),
// UMMA shared-memory and instruction descriptors.  Raw inline PTX; no CUTLASS dependency.
#pragma once
#include <cuda.h>          // CUtensorMap type + enums only (the driver entry point is fetched at run time)
#include <cuda_bf16.h>
#include "common.cuh"

namespace aaconv {
namespace tc {

// ------------------------------------------------------------------------------------------------
// generic helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ bool elect_one() {
  uint32_t pred = 0;
  asm volatile(
      "{\n\t.reg .pred P;\n\telect.sync _|P, 0xffffffff;\n\tselp.b32 %0, 1, 0, P;\n\t}\n"
      : "=r"(pred));
  return pred != 0;
}

// ------------------------------------------------------------------------------------------------
// mbarrier
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
// Arrive that cannot ISSUE before the registers feeding `dep_zero` have been written.  A consumer that releases a shared-memory
// stage after ld.shared'ing it must use this when nothing else consumes the loaded registers before the arrive: the loads
// are asynchronous (only a later USE of their destination registers waits for them), the arrive is not ordered behind them,
// and the producer's TMA write may then overwrite the stage while the last loads are still queued -- seen as run-to-run
// differences in the last-loaded 16-byte chunks of rel_bwd_tc's rows (single-stage configuration, 512 px).
// dep_zero = (xor of the loaded registers) & zmask with zmask == 0 at run time but unknown to the compiler.  The kernels that
// use it (aug_build_tc_kernel, rel_bwd_tc_kernel) take zmask as their last argument, `uint32_t dep_zero`, which every launch
// passes as 0.  It must stay a kernel argument: with a literal 0 (or anything else the compiler can prove is 0) the fold is
// deleted and the arrive issues right after the last ld.shared again; as a parameter it reaches the arrive's operand through
// a LOP3 of the loaded registers and the parameter (cuobjdump -sass: LOP3.LUT -> VIADD -> SYNCS.ARRIVE.TRANS64).
__device__ __forceinline__ void mbar_arrive_after(uint64_t* bar, uint32_t dep_zero) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(1u + dep_zero) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 P, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, P;\n\t}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
// Bounded wait: a protocol bug traps (-> launch error at the next sync) instead of hanging the GPU.  In "soft" mode
// (aaconv_debug_set_mode bit 16; debugging only) a timed-out wait is logged to a device buffer and treated as satisfied, so
// the kernel ends and the host can read WHICH barriers were stuck (aaconv_debug_read_mbar_log).
constexpr uint32_t MBAR_SPIN_LIMIT = 1u << 26;
static __device__ unsigned long long* g_mbar_log = nullptr;   // mapped pinned host memory: [0] = count, [1..64] = records
static __device__ unsigned g_mbar_soft = 0;                   // (survives a later fault of the kernel)
static __device__ __noinline__ void mbar_timeout(uint32_t bar, uint32_t parity) {
  if (g_mbar_soft && g_mbar_log) {
    const unsigned long long k = atomicAdd(g_mbar_log, 1ull);
    if (k < 64) g_mbar_log[1 + k] = ((unsigned long long)bar << 32) | ((unsigned long long)parity << 31) | ((unsigned long long)blockIdx.x << 12) | threadIdx.x;
    __threadfence_system();
    return;
  }
  printf("aaconv: mbarrier timeout block (%d,%d) thread %d bar 0x%x parity %u\n", blockIdx.x, blockIdx.y, threadIdx.x,
         bar, parity);
  __trap();
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0xFFFFFu) == 0 && (spins >= MBAR_SPIN_LIMIT || g_mbar_soft)) {   // flag read once per 2^20 polls
      mbar_timeout(smem_u32(bar), parity);
      break;
    }
  }
}
// Same, for waiters that are not on the critical path (math warpgroups, TMA producer): back off between polls so that
// many spinning warps do not crowd the barrier unit the MMA-issuing warps depend on.
__device__ __forceinline__ void mbar_wait_relaxed(uint64_t* bar, uint32_t parity) {
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    __nanosleep(40);
    if (++spins > (MBAR_SPIN_LIMIT >> 4)) { mbar_timeout(smem_u32(bar), parity); break; }
  }
}

// ------------------------------------------------------------------------------------------------
// TMA
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
__device__ __forceinline__ void tma_load_4d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2, int c3) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
      : "memory");
}

// ------------------------------------------------------------------------------------------------
// tcgen05
// ------------------------------------------------------------------------------------------------
template <uint32_t NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* dst_smem) {   // whole warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "n"(NCOLS) : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <uint32_t NCOLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {    // whole warp
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T   (both operands K-major unless the idesc says otherwise)
__device__ __forceinline__ void mma_ss(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// D[tmem] (+)= A[tmem] * B[smem]^T
__device__ __forceinline__ void mma_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}\n"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// arrive on an mbarrier when every previously issued tcgen05.mma of this thread has completed
__device__ __forceinline__ void mma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// TMEM -> registers: this warp's 32 lanes x N consecutive 32-bit columns (thread i <-> lane base+i)
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// After tmem_ld_wait(): ties the 32 destination registers of an earlier tcgen05.ld to this point of the instruction stream, so
// that arithmetic on them cannot be scheduled above the wait (the load is asynchronous: the compiler only sees the asm that
// ISSUED it).  Needed once a load is kept in flight under unrelated math (software-pipelined S' reads); emits no instruction.
__device__ __forceinline__ void tmem_ld_landed(uint32_t (&r)[32]) {
  asm volatile(""
               : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]), "+r"(r[8]),
                 "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]), "+r"(r[16]),
                 "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]), "+r"(r[24]),
                 "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
               :
               : "memory");
}

__device__ __forceinline__ void tmem_st_x16(uint32_t taddr, const uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31,%32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ------------------------------------------------------------------------------------------------
// descriptors
// ------------------------------------------------------------------------------------------------
// K-major operand tile stored as rows of exactly 128 bytes (64 bf16) with the 128B swizzle TMA writes:
// 8-row groups are 1024 B apart (SBO), LBO unused for swizzled K-major layouts, descriptor version 1.
__device__ __forceinline__ uint64_t smem_desc_sw128_kmajor(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr & 0x3FFFF) >> 4);        // start address, bits [0,14)
  d |= (uint64_t)1 << 16;                          // leading byte offset (ignored), bits [16,30)
  d |= (uint64_t)(1024 >> 4) << 32;                // stride byte offset, bits [32,46)
  d |= (uint64_t)1 << 46;                          // descriptor version (Blackwell), bits [46,48)
  d |= (uint64_t)2 << 61;                          // layout type SWIZZLE_128B, bits [61,64)
  return d;
}
// The same descriptors as (lo, hi) halves: hi is constant for every SWIZZLE_128B tile with 1024 B row groups, so
// the MMA issue loop only does 32-bit adds on `lo` (start address >> 4 in bits [0,14), LBO >> 4 in bits [16,30)).
constexpr uint32_t DESC_HI_SW128 = (1024u >> 4) | (1u << 14) | (2u << 29);
__device__ __forceinline__ uint32_t desc_lo_k(uint32_t saddr) { return ((saddr & 0x3FFFF) >> 4) | (1u << 16); }
__device__ __forceinline__ uint32_t desc_lo_mn(uint32_t saddr, uint32_t lbo_bytes) {
  return ((saddr & 0x3FFFF) >> 4) | (((lbo_bytes >> 4) & 0x3FFF) << 16);
}
__device__ __forceinline__ uint64_t desc64(uint32_t lo) { return ((uint64_t)DESC_HI_SW128 << 32) | lo; }

// Fully unrolled score-MMA issue (A in TMEM, B K-major in shared memory, one 16-wide k-step per MMA).  The issue rate of the
// single issuing thread is the critical resource: with compile-time trip counts and offsets the tensor pipe runs at its
// N/2-cycle floor, with a runtime loop each MMA costs ~80 cycles of issue (tools/mma_bench.cu).  NKS = number of k-steps
// of the main accumulator; EXTRA = 1 issues one more k-step (index NKS) into a second accumulator.
template <int NKS, int EXTRA, uint32_t B_ATOM>
__device__ __forceinline__ void issue_ts_ksteps(uint32_t d_main, uint32_t d_extra, uint32_t a_tmem, uint32_t b_lo, uint32_t idesc) {
#pragma unroll
  for (int ks = 0; ks < NKS; ++ks)
    mma_ts(d_main, a_tmem + ks * 8, desc64(b_lo + (ks >> 2) * B_ATOM + (ks & 3) * 2), idesc, ks > 0 ? 1u : 0u);
  if (EXTRA) mma_ts(d_extra, a_tmem + NKS * 8, desc64(b_lo + (NKS >> 2) * B_ATOM + (NKS & 3) * 2), idesc, 0u);
}
template <int EXTRA, uint32_t B_ATOM>
__device__ __forceinline__ void issue_ts_ksteps_n(int nks, uint32_t d_main, uint32_t d_extra, uint32_t a_tmem, uint32_t b_lo, uint32_t idesc) {
  switch (nks) {   // warp-uniform
    case 1: issue_ts_ksteps<1, EXTRA, B_ATOM>(d_main, d_extra, a_tmem, b_lo, idesc); break;
    case 2: issue_ts_ksteps<2, EXTRA, B_ATOM>(d_main, d_extra, a_tmem, b_lo, idesc); break;
    case 3: issue_ts_ksteps<3, EXTRA, B_ATOM>(d_main, d_extra, a_tmem, b_lo, idesc); break;
    case 4: issue_ts_ksteps<4, EXTRA, B_ATOM>(d_main, d_extra, a_tmem, b_lo, idesc); break;
    case 5: issue_ts_ksteps<5, EXTRA, B_ATOM>(d_main, d_extra, a_tmem, b_lo, idesc); break;
    case 6: issue_ts_ksteps<6, EXTRA, B_ATOM>(d_main, d_extra, a_tmem, b_lo, idesc); break;
    case 7: issue_ts_ksteps<7, EXTRA, B_ATOM>(d_main, d_extra, a_tmem, b_lo, idesc); break;
    case 8: issue_ts_ksteps<8, EXTRA, B_ATOM>(d_main, d_extra, a_tmem, b_lo, idesc); break;
    case 9: issue_ts_ksteps<9, EXTRA, B_ATOM>(d_main, d_extra, a_tmem, b_lo, idesc); break;
    case 10: issue_ts_ksteps<10, EXTRA, B_ATOM>(d_main, d_extra, a_tmem, b_lo, idesc); break;
    default: issue_ts_ksteps<11, EXTRA, B_ATOM>(d_main, d_extra, a_tmem, b_lo, idesc); break;
  }
}

// advance the start address by `bytes` (a multiple of 16; used to step K by 16 bf16 = 32 B inside the atom)
__device__ __forceinline__ uint64_t desc_advance(uint64_t desc, uint32_t bytes) { return desc + (bytes >> 4); }

// kind::f16 instruction descriptor: bf16 x bf16 -> fp32, both operands K-major
__host__ __device__ constexpr uint32_t idesc_bf16_f32(int M, int N) {
  return (1u << 4)                      // D format  : F32
         | (1u << 7)                    // A format  : BF16
         | (1u << 10)                   // B format  : BF16
         | ((uint32_t)(N >> 3) << 17)   // N / 8
         | ((uint32_t)(M >> 4) << 24);  // M / 16
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
  uint32_t r;
  asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));   // upper half <- first source
  return r;
}
__device__ __forceinline__ float ex2f(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}


}  // namespace tc

// ------------------------------------------------------------------------------------------------
// host: TMA descriptor encode through the driver entry point (no link-time libcuda dependency)
// ------------------------------------------------------------------------------------------------
// bf16 tensor, `rank` dims (dim 0 contiguous), strides in bytes for dims 1..rank-1, 128B swizzle.
int make_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                   const uint32_t* box, const uint32_t* elem_strides);

}  // namespace aaconv
