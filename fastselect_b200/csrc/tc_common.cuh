// tc_common.cuh -- sm_100a building blocks for the one-hot tensor-core kernels:
// mbarrier, TMA (cp.async.bulk.tensor), TMEM allocation, tcgen05.mma kind::i8,
// tcgen05.ld, and the shared-memory / instruction descriptors they need.
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace fs {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ------------------------------------------------------------------ mbarrier
__device__ __forceinline__ void mbar_init(uint64_t *bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t *bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "WAIT_LOOP:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
        "@p bra WAIT_DONE;\n\t"
        "bra WAIT_LOOP;\n\t"
        "WAIT_DONE:\n\t"
        "}\n" ::"r"(smem_u32(bar)), "r"(parity)
        : "memory");
}

// ----------------------------------------------------------------------- TMA
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap *m) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(m)) : "memory");
}
// 2-D tile load: c0 = coordinate along the contiguous (byte) dimension, c1 = row
__device__ __forceinline__ void tma_load_2d(void *smem_dst, const CUtensorMap *m, uint64_t *bar, int32_t c0, int32_t c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
        : "memory");
}

// L2 prefetches: a 4-D tile of a tensor map, and a run of bytes (16-byte aligned, size a multiple of 16)
__device__ __forceinline__ void tma_prefetch_4d(const CUtensorMap *m, int32_t c0, int32_t c1, int32_t c2, int32_t c3) {
    asm volatile("cp.async.bulk.prefetch.tensor.4d.L2.global [%0, {%1, %2, %3, %4}];" ::"l"(reinterpret_cast<uint64_t>(m)), "r"(c0),
                 "r"(c1), "r"(c2), "r"(c3)
                 : "memory");
}
__device__ __forceinline__ void bulk_prefetch_l2(const void *gptr, uint32_t bytes) {
    asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(__cvta_generic_to_global(gptr)), "r"(bytes) : "memory");
}

// 1-D bulk copy global -> shared (size a multiple of 16 bytes), completion on a local mbarrier
__device__ __forceinline__ void bulk_load_1d(void *smem_dst, const void *gsrc, uint32_t bytes, uint64_t *bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(smem_dst)),
                 "l"(reinterpret_cast<uint64_t>(gsrc)), "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}

// ---------------------------------------------------------------------- TMEM
template <int kCols>
__device__ __forceinline__ void tmem_alloc(uint32_t *dst_smem) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "n"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc(uint32_t addr) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(addr), "n"(kCols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// tcgen05.commit: the mbarrier is arrived on when all previously issued MMAs of this thread retire
__device__ __forceinline__ void tc_commit(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
                 : "memory");
}

// D[tmem] (+)= A[smem] * B[smem]^T, int8 operands, int32 accumulators
__device__ __forceinline__ void mma_i8(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}

// 32 lanes x 32 consecutive 32-bit columns -> 32 registers per thread (thread = lane)
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
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
// 32 lanes x 16 consecutive 32-bit columns
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
          "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
// 16 lanes x 256 bits (8 columns) of this warp's lane quarter, starting at the lane in the address
// (offset 0 or 16): thread t receives (lane t/4, columns 2(t%4), 2(t%4)+1) in r0, r1 and
// (lane t/4 + 8, the same columns) in r2, r3 -- measured, profiles/r02_tmem_frag_probe.txt
__device__ __forceinline__ void tmem_ld_16x256b(uint32_t taddr, uint32_t (&r)[4]) {
    asm volatile("tcgen05.ld.sync.aligned.16x256b.x1.b32 {%0, %1, %2, %3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(taddr)
                 : "memory");
}
// tcgen05.wait::ld that names the registers it makes valid, so that the compiler cannot move their
// first use above the wait
__device__ __forceinline__ void tmem_ld_wait_on(uint32_t (&a)[4], uint32_t (&b)[4], uint32_t (&c)[4], uint32_t (&d)[4]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(a[0]), "+r"(a[1]), "+r"(a[2]), "+r"(a[3]), "+r"(b[0]), "+r"(b[1]), "+r"(b[2]), "+r"(b[3]), "+r"(c[0]),
                   "+r"(c[1]), "+r"(c[2]), "+r"(c[3]), "+r"(d[0]), "+r"(d[1]), "+r"(d[2]), "+r"(d[3])
                 :
                 : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// one 32-bit column of this warp's 32 lanes
__device__ __forceinline__ void tmem_st_32x1(uint32_t taddr, uint32_t v) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(taddr), "r"(v) : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem]^T, e2m1 (FP4) operands with UE8M0 block scales (one per 32
// elements, read from TMEM), FP32 accumulators; K = 64 elements (32 bytes) per instruction, twice
// the int8 rate.  With all scales 1.0 and small-integer operands the FP32 sums are exact up to 2^24
// (measured on B200: tools/mxf4_probe.cu).
__device__ __forceinline__ void mma_mxf4(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t tmem_sfa,
                                         uint32_t tmem_sfb, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::mxf4.block_scale.block32 [%0], %1, %2, %3, [%5], [%6], p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(tmem_sfa), "r"(tmem_sfb)
        : "memory");
}
// Instruction descriptor for kind::mxf4: A = B = e2m1, K-major, UE8M0 scale factors (ids 0), dense K = 64.
__host__ __device__ constexpr uint32_t make_idesc_mxf4(int m, int n) {
    return (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | (1u << 23) | ((uint32_t)(m >> 4) << 24);
}
// exact float -> int for integral |x| < 2^22 without the conversion unit
__device__ __forceinline__ int f32_to_int_exact(uint32_t bits) {
    return __float_as_int(__uint_as_float(bits) + 12582912.0f) - 0x4B400000;
}

// 0xffffffff when byte b of x has its top bit set, else 0 (prmt sign-replicate mode; b is a constant)
__device__ __forceinline__ uint32_t byte_mask(uint32_t x, int b) {
    uint32_t r;
    asm("prmt.b32 %0, %1, %1, %2;" : "=r"(r) : "r"(x), "r"(0x8888u + 0x1111u * (uint32_t)b));
    return r;
}

// ------------------------------------------------------------- descriptors
// Shared-memory matrix descriptor, K-major operand, 128-byte swizzle, rows of
// exactly 128 bytes (one swizzle atom wide): 8-row groups are 1024 B apart (SBO);
// LBO is unused for swizzled K-major layouts (encoded as 1); version = 1 (sm_100).
__device__ __forceinline__ uint64_t make_smem_desc_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr >> 4) & 0x3FFFu);
    d |= (uint64_t)1 << 16;
    d |= (uint64_t)(1024 >> 4) << 32;
    d |= (uint64_t)1 << 46;
    d |= (uint64_t)2 << 61;
    return d;
}

// Instruction descriptor for kind::i8: D = S32, A = B = signed int8, both K-major.
__host__ __device__ constexpr uint32_t make_idesc_i8(int m, int n) {
    return (2u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// ----------------------------------------------------------- CTA pairs (cta_group::2)
// A cluster of two CTAs drives one tcgen05.mma.cta_group::2: M = 256 (128 rows per CTA), the B operand
// read from both CTAs' shared memory (each stages half of its rows); the leader (cluster rank 0) issues.
constexpr uint32_t kLeaderMask = 0xFEFFFFFFu;   // shared::cluster address of the same offset in CTA 0 of the pair

__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// 2-D tile load by either CTA of the pair; the bytes are credited to the LEADER's mbarrier
__device__ __forceinline__ void tma_load_2d_pair(void *smem_dst, const CUtensorMap *m, uint64_t *bar, int32_t c0, int32_t c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];" ::"r"(
            smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & kLeaderMask), "r"(c0), "r"(c1)
        : "memory");
}
// 4-D / 5-D tile loads, by either CTA of the pair: the outer box dimensions enumerate ROWS of the operand in a
// permuted order (the accumulation kernel's merged-plane epilogue); c0 = coordinate along the contiguous (byte) dimension
__device__ __forceinline__ void tma_load_4d_pair(void *smem_dst, const CUtensorMap *m, uint64_t *bar, int32_t c0, int32_t c1,
                                                 int32_t c2, int32_t c3) {
    asm volatile(
        "cp.async.bulk.tensor.4d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];" ::"r"(
            smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & kLeaderMask), "r"(c0), "r"(c1), "r"(c2), "r"(c3)
        : "memory");
}
__device__ __forceinline__ void tma_load_5d_pair(void *smem_dst, const CUtensorMap *m, uint64_t *bar, int32_t c0, int32_t c1,
                                                 int32_t c2, int32_t c3, int32_t c4) {
    asm volatile(
        "cp.async.bulk.tensor.5d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];" ::"r"(
            smem_u32(smem_dst)),
        "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar) & kLeaderMask), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
        : "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_alloc_pair(uint32_t *dst_smem) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(dst_smem)), "n"(kCols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
template <int kCols>
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t addr) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(addr), "n"(kCols) : "memory");
}
// arrives on the mbarrier at this shared-memory offset in BOTH CTAs when the pair's MMAs retire
__device__ __forceinline__ void tc_commit_pair(uint64_t *bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;" ::"r"(
                     smem_u32(bar)),
                 "h"((uint16_t)3)
                 : "memory");
}
__device__ __forceinline__ void mma_mxf4_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                              uint32_t tmem_sfa, uint32_t tmem_sfb, uint32_t accumulate) {
    asm volatile(
        "{\n\t"
        ".reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::mxf4.block_scale.block32 [%0], %1, %2, %3, [%5], [%6], p;\n\t"
        "}\n" ::"r"(tmem_d),
        "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(tmem_sfa), "r"(tmem_sfb)
        : "memory");
}
// arrive on the mbarrier at this offset in CTA `cta` of the cluster (release at cluster scope)
__device__ __forceinline__ void mbar_arrive_cluster(uint64_t *bar, uint32_t cta) {
    uint32_t remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(bar)), "r"(cta));
    asm volatile("mbarrier.arrive.release.cluster.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}
// the same without the cluster-scope release (which compiles to MEMBAR.ALL.GPU): for hand-offs whose payload is
// ordered by tcgen05.fence (TMEM reads completed), not by generic-proxy memory ordering
__device__ __forceinline__ void mbar_arrive_cluster_relaxed(uint64_t *bar, uint32_t cta) {
    uint32_t remote;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(remote) : "r"(smem_u32(bar)), "r"(cta));
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(remote) : "memory");
}

// The four K = 64 steps of one 128-byte K block (descriptor start address + 2 per step) and commits, executed by a
// CONVERGED warp: elect.sync picks the issuing lane inside the statement, so the operands stay warp-uniform.
template <bool kPair>
__device__ __forceinline__ void mma_mxf4_x4(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t tmem_sf,
                                            uint32_t accumulate) {
    if constexpr (kPair) {
        asm volatile(
            "{\n\t"
            ".reg .pred p, e;\n\t"
            ".reg .b64 a, b;\n\t"
            "elect.sync _|e, 0xffffffff;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "@e tcgen05.mma.cta_group::2.kind::mxf4.block_scale.block32 [%0], %1, %2, %3, [%5], [%5], p;\n\t"
            "setp.eq.b32 p, 0, 0;\n\t"
            "add.s64 a, %1, 2;\n\t"
            "add.s64 b, %2, 2;\n\t"
            "@e tcgen05.mma.cta_group::2.kind::mxf4.block_scale.block32 [%0], a, b, %3, [%5], [%5], p;\n\t"
            "add.s64 a, %1, 4;\n\t"
            "add.s64 b, %2, 4;\n\t"
            "@e tcgen05.mma.cta_group::2.kind::mxf4.block_scale.block32 [%0], a, b, %3, [%5], [%5], p;\n\t"
            "add.s64 a, %1, 6;\n\t"
            "add.s64 b, %2, 6;\n\t"
            "@e tcgen05.mma.cta_group::2.kind::mxf4.block_scale.block32 [%0], a, b, %3, [%5], [%5], p;\n\t"
            "}\n" ::"r"(tmem_d),
            "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(tmem_sf)
            : "memory");
    } else {
        asm volatile(
            "{\n\t"
            ".reg .pred p, e;\n\t"
            ".reg .b64 a, b;\n\t"
            "elect.sync _|e, 0xffffffff;\n\t"
            "setp.ne.b32 p, %4, 0;\n\t"
            "@e tcgen05.mma.cta_group::1.kind::mxf4.block_scale.block32 [%0], %1, %2, %3, [%5], [%5], p;\n\t"
            "setp.eq.b32 p, 0, 0;\n\t"
            "add.s64 a, %1, 2;\n\t"
            "add.s64 b, %2, 2;\n\t"
            "@e tcgen05.mma.cta_group::1.kind::mxf4.block_scale.block32 [%0], a, b, %3, [%5], [%5], p;\n\t"
            "add.s64 a, %1, 4;\n\t"
            "add.s64 b, %2, 4;\n\t"
            "@e tcgen05.mma.cta_group::1.kind::mxf4.block_scale.block32 [%0], a, b, %3, [%5], [%5], p;\n\t"
            "add.s64 a, %1, 6;\n\t"
            "add.s64 b, %2, 6;\n\t"
            "@e tcgen05.mma.cta_group::1.kind::mxf4.block_scale.block32 [%0], a, b, %3, [%5], [%5], p;\n\t"
            "}\n" ::"r"(tmem_d),
            "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate), "r"(tmem_sf)
            : "memory");
    }
}
// tcgen05.commit by one elected lane of a converged warp (pairs: multicast to both CTAs' barriers)
template <bool kPair>
__device__ __forceinline__ void tc_commit_elected(uint64_t *bar) {
    if constexpr (kPair) {
        asm volatile(
            "{\n\t"
            ".reg .pred e;\n\t"
            "elect.sync _|e, 0xffffffff;\n\t"
            "@e tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;\n\t"
            "}\n" ::"r"(smem_u32(bar)),
            "h"((uint16_t)3)
            : "memory");
    } else {
        asm volatile(
            "{\n\t"
            ".reg .pred e;\n\t"
            "elect.sync _|e, 0xffffffff;\n\t"
            "@e tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n\t"
            "}\n" ::"r"(smem_u32(bar))
            : "memory");
    }
}

__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t"
        ".reg .pred P;\n\t"
        "elect.sync _|P, 0xffffffff;\n\t"
        "selp.b32 %0, 1, 0, P;\n\t"
        "}\n"
        : "=r"(pred));
    return pred != 0;
}

}  // namespace tc

// Host (tc_dist.cu): 2-D uint8 tensor map, box = 128 bytes x box_rows, 128-byte swizzle.
CUtensorMap make_tmap_u8_sw128(const void *base, uint64_t row_bytes, uint64_t rows, uint64_t pitch_bytes,
                               uint32_t box_rows);
// Host: rank-`rank` (3..5) uint8 tensor map, 128-byte swizzle; dims[0] / box[0] along the contiguous bytes,
// strides[i] = byte stride of dimension i + 1.  Returns false (map untouched) when the driver refuses it.
bool make_tmap_u8_sw128_nd(CUtensorMap *out, const void *base, int rank, const uint64_t *dims, const uint64_t *strides,
                           const uint32_t *box);

}  // namespace fs
