// Thin inline-PTX layer for sm_100a: mbarrier, bulk async copy (TMA engine), tcgen05 (UMMA) and
// tensor memory.  Bit layouts of the descriptors follow the PTX ISA tables for tcgen05.mma
// (shared-memory matrix descriptor and instruction descriptor, kind::f16).
#pragma once
#include <cuda_bf16.h>
#include <stdint.h>

namespace sm100 {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier ---------------------------------------------------------------------------------
// Suspend-time hint of mbarrier.try_wait: the waiting thread may sleep in hardware until the phase completes (it is woken as soon as it
// does) instead of returning after the short default window.  Without it the role warps of the MLP kernels spent ~30 % of all issued
// instructions on try_wait / branch pairs (ncu source counters) -- issue slots the epilogue warps of the same scheduler need.
constexpr uint32_t MBAR_SUSPEND_HINT = 0x989680u;

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_mbar_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(ok)
        : "r"(smem_u32(bar)), "r"(parity), "r"(MBAR_SUSPEND_HINT)
        : "memory");
    return ok != 0;
}
// Waits until the phase with the given parity has completed.
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) {
    }
}

// ---- bulk async copy global -> shared (TMA engine, SASS UBLKCP), completion on an mbarrier --------
__device__ __forceinline__ void bulk_g2s(void* smem_dst, const void* gmem_src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(
                     smem_u32(smem_dst)),
                 "l"(gmem_src), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// ---- bulk async copy shared -> global (TMA store), tracked by the issuing thread's bulk groups ----------
__device__ __forceinline__ void bulk_s2g(void* gmem_dst, const void* smem_src, uint32_t bytes) {
    asm volatile("cp.async.bulk.global.shared::cta.bulk_group [%0], [%1], %2;" ::"l"(gmem_dst), "r"(smem_u32(smem_src)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
// every bulk group of this thread has finished READING its shared-memory source (the source may be overwritten)
__device__ __forceinline__ void bulk_wait_read_all() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
// all but the most recent bulk group of this thread have finished reading their shared-memory source
__device__ __forceinline__ void bulk_wait_read_but_one() { asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory"); }
// every bulk group of this thread has completed (writes performed)
__device__ __forceinline__ void bulk_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
// named barrier over `nthreads` threads of the CTA (id 0 is __syncthreads)
__device__ __forceinline__ void named_bar_sync(int id, int nthreads) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(nthreads) : "memory"); }

// generic-proxy smem writes -> visible to the async proxy (UMMA / TMA reads)
__device__ __forceinline__ void fence_proxy_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// ---- tensor memory ----------------------------------------------------------------------------
// warp-wide; writes the allocated base address to *smem_slot
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_slot, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "r"(ncols)
                 : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tmem_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// 32 lanes x 32 consecutive 32-bit columns: thread i of the warp receives row (lane base + i)
__device__ __forceinline__ void tmem_ld32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
          "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
          "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}

// ---- UMMA descriptors -------------------------------------------------------------------------
enum : uint32_t { SWIZZLE_NONE = 0, SWIZZLE_128B = 2, SWIZZLE_64B = 4, SWIZZLE_32B = 6 };

// Shared-memory matrix descriptor for a K-major operand whose rows are 128 B (64 bf16) wide and
// 128B-swizzled: 8-row groups are 1024 B apart (SBO); LBO is unused for swizzled K-major layouts.
//   [0,14) start>>4   [16,30) LBO>>4   [32,46) SBO>>4   [46,48) version=1   [61,64) swizzle mode
__device__ __forceinline__ uint64_t umma_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)SWIZZLE_128B << 61;
    return d;
}

// Instruction descriptor, kind::f16, A and B = bf16 (K-major), D = fp32.
//   [4,6) D fmt (1 = f32)  [7,10) A fmt (1 = bf16)  [10,13) B fmt  [15] A major  [16] B major
//   [17,23) N>>3   [24,29) M>>4
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

// D[tmem] (+)= A[smem] * B[smem]^T ; issued by ONE thread
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t adesc, uint64_t bdesc, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}" ::"r"(tmem_d),
        "l"(adesc), "l"(bdesc), "r"(idesc), "r"(accumulate)
        : "memory");
}

// mbarrier arrive once every previously issued tcgen05.mma of this thread has completed
// (implies tcgen05.fence::before_thread_sync)
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}

// ---- CTA pairs (cluster of 2, tcgen05 cta_group::2): one M = 256 MMA over both CTAs' 128 rows, the B operand split across the pair ----
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// arrive on the mbarrier at the same shared-memory offset in CTA `rank` of the cluster
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* local_bar, uint32_t rank) {
    asm volatile(
        "{\n\t.reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}" ::"r"(smem_u32(local_bar)), "r"(rank)
        : "memory");
}
// wait on a LOCAL mbarrier whose arrivals may come from the peer CTA (cluster-scope acquire)
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    do {
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2, %3;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(ok)
            : "r"(smem_u32(bar)), "r"(parity), "r"(MBAR_SUSPEND_HINT)
            : "memory");
    } while (!ok);
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_slot, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_slot)), "r"(ncols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
// arrive on the mbarrier at this offset in BOTH CTAs once every previously issued MMA of the pair has completed
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(smem_u32(bar)),
                 "h"((uint16_t)3)
                 : "memory");
}

// true in exactly one lane of the (fully active) warp
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile("{\n\t.reg .pred p;\n\telect.sync _|p, 0xffffffff;\n\tselp.u32 %0, 1, 0, p;\n\t}" : "=r"(pred));
    return pred != 0;
}

// 32 lanes x 16 consecutive 32-bit columns
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}

// tcgen05.mma with the two smem descriptors given as (lo, hi) halves: lo = the 14-bit start-address field (+ LBO bit), advanced with
// plain 32-bit adds of compile-time constants; hi is the same constant for both operands.  Issued by ONE thread.
__device__ __forceinline__ void umma_lohi(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t hi, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "mov.b64 da, {%1, %3};\n\tmov.b64 db, {%2, %3};\n\t"
        "setp.ne.b32 p, %5, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], da, db, %4, p;\n\t}" ::"r"(tmem_d),
        "r"(a_lo), "r"(b_lo), "r"(hi), "r"(idesc), "r"(accumulate)
        : "memory");
}
// The same for a CTA pair: M = 256 (128 rows from each CTA), the N rows of B split across the two CTAs; issued by the leader only.
__device__ __forceinline__ void umma_lohi_pair(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t hi, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t.reg .b64 da, db;\n\t"
        "mov.b64 da, {%1, %3};\n\tmov.b64 db, {%2, %3};\n\t"
        "setp.ne.b32 p, %5, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], da, db, %4, p;\n\t}" ::"r"(tmem_d),
        "r"(a_lo), "r"(b_lo), "r"(hi), "r"(idesc), "r"(accumulate)
        : "memory");
}
template <bool PAIR>
__device__ __forceinline__ void umma_any(uint32_t tmem_d, uint32_t a_lo, uint32_t b_lo, uint32_t hi, uint32_t idesc, uint32_t accumulate) {
    if constexpr (PAIR) umma_lohi_pair(tmem_d, a_lo, b_lo, hi, idesc, accumulate);
    else umma_lohi(tmem_d, a_lo, b_lo, hi, idesc, accumulate);
}
template <bool PAIR>
__device__ __forceinline__ void commit_any(uint64_t* bar) {
    if constexpr (PAIR) umma_commit_pair(bar);
    else umma_commit(bar);
}
// issuer-side wait on an event whose arrivals may come from the peer CTA
template <bool PAIR>
__device__ __forceinline__ void wait_ev(uint64_t* bar, uint32_t parity) {
    if constexpr (PAIR) mbar_wait_cluster(bar, parity);
    else mbar_wait(bar, parity);
}

// Descriptor halves of a K-major, NON-swizzled 16-column (K = 16) bf16 tile stored as [row/8][k/8][row%8][k%8]: 8x8 core matrices of
// 128 contiguous bytes, the two K halves 128 B apart (leading byte offset), 8-row groups 256 B apart (stride byte offset).
constexpr uint32_t HI_NOSWZ = (256u >> 4) | (1u << 14);
__device__ __forceinline__ uint32_t desc_lo_noswz(uint32_t smem_addr) { return ((smem_addr & 0x3FFFF) >> 4) | ((128u >> 4) << 16); }

// byte offset of element (row, col) of a [rows][64] bf16 K-major tile in the 128B-swizzled layout
__host__ __device__ __forceinline__ uint32_t sw128_offset(uint32_t row, uint32_t col) {
    return (row >> 3) * 1024 + (row & 7) * 128 + ((((col >> 3) ^ row) & 7) << 4) + (col & 7) * 2;
}

// ReLU that keeps NaN (F.relu does; fmaxf(x, 0) returns 0 for a NaN x): one FMNMX.NAN
__device__ __forceinline__ float relu_nan(float x) {
    float r;
    asm("max.NaN.f32 %0, %1, 0f00000000;" : "=f"(r) : "f"(x));
    return r;
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}
__device__ __forceinline__ uint32_t pack_bf16x2_relu(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.relu.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

}  // namespace sm100
