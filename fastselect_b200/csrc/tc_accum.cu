// tc_accum.cu -- per-feature hit/miss weight accumulation for discrete columns as a
// (neighbour mask) x (one-hot) GEMM on the 5th-gen tensor cores (FP4 operands, exact integer
// results), with a fused select / scale / reduce epilogue.
//
// Replaces the discrete branch of the reference's accumulation loops and their
// normalisation (MultiSURF.py:218-251, SURF.py:165-195).  For a discrete feature f with
// value codes c_jf:
//     sum_j c_ij [x_if != x_jf] = sum_j c_ij - sum_j c_ij [c_jf = c_if],
// and with c_ij = -aH_i * mH_ij + aM_i * mM_ij (mH, mM in {-1, 0, 1}: near/far hit and
// miss masks, aH_i = 1/|H_i|, aM_i = 1/|M_i| or 1) the inner sums are the integer GEMMs
//     GH[(f,v), i] = sum_j At[(f,v), j] * mH[i, j],   GM likewise,
// over the REDUCED one-hot rows v < last_f (onehot.cu); the implied last plane follows from
// sum_v G[(f,v), i] = rs_i (the mask's row sum), so
//     W_i[f] = sum_{v<last} [c_if = v] * k_i (rs_i - G[(f,v), i])  +  [c_if = last] * k_i * sum_{v<last} G[(f,v), i]
// for each of the two masks (k_i = -aH_i or +aM_i).  The thread that owns one-hot row (f,v)
// therefore adds k_i (rs_i - G) for targets whose code is v and k_i G for targets whose
// code is the last one: no exchange between rows.
//
// Arithmetic.  At holds 0/1 and the masks -1/0/1, both exact in e2m1, so the GEMM runs on
// tcgen05 kind::mxf4 (unit UE8M0 block scales, FP32 accumulators): the sums are integers below
// 2^22 and therefore exact in FP32 (probed on B200, tools/mxf4_probe.cu) at twice the int8 MMA
// rate.  The per-target scaling k_i * t is accumulated exactly as well: k_i is a 52-bit
// fixed-point number in two 26-bit limbs, t an integer, the sums two int64 -- no float64
// instruction in the inner loop (FP64 and the tensor pipe did not overlap on B200).
//
// Two kernels.  tc_accum_merged_kernel (below, the default for 0/1/2 columns: clusters of two CTAs, both
// planes of a column in one epilogue thread, exact 64-bit column sums by atomics) and the older
// tc_accum_kernel for every other value count, described first:
//
// Kernel: persistent, one CTA per SM.  A work unit is 128 one-hot rows (UMMA M = TMEM
// lanes) x a group of tiles of <= 240 target rows (UMMA N); units are dealt
// round-robin and the TMA / MMA / epilogue pipelines run across unit boundaries without
// draining.  Tiles never straddle a class boundary (host-built descriptors, staged in
// shared memory).  Each tile is processed as two work items, "hit" and "miss", one mask
// and one 240-column TMEM accumulator each (double-buffered, so the epilogue of one item
// overlaps the MMAs of the next; 8 more TMEM columns hold the scale factors).  Warp 0: TMA
// producer (At tile + mask tile per K block of 256 samples = 128 bytes, 128B swizzle, 4-stage
// mbarrier ring); warp 1: one thread issues tcgen05.mma.cta_group::1.kind::mxf4 (M=128,
// N<=240, K=64); warps 2-13 (lane quarter x column third): epilogue -- tcgen05.ld the
// accumulator, test the target's own value code (codesT), scale, and add into the fixed-point
// sums of its one-hot row; the reduction over a tile's targets is a loop over TMEM columns
// inside one thread.
// Samples are class-sorted, so for a class-homogeneous target tile the hit mask is
// non-zero only in the K blocks of the tile's own class and the miss mask only outside:
// the other K blocks are skipped, which keeps the MMA work at 2 MAC per (pair, feature)
// for 3-valued genotypes.  Partials are written per (tile group, column part, one-hot row) and
// reduced in a fixed order.
#include <algorithm>
#include <cstring>

#include "common.cuh"
#include "tc_common.cuh"

namespace fs {

namespace {
constexpr int BM = 128;   // one-hot rows per work unit
constexpr int BN = 240;   // target rows per tile (2 accumulators x 240 + 8 scale-factor columns <= 512 TMEM columns)
constexpr int BK = 128;   // bytes of K per block ...
constexpr int KS = 256;   // ... = 256 samples (FP4 nibbles)
constexpr int STAGES = 4;
constexpr int A_BYTES = BM * BK;                  // 16 KB
constexpr int B_BYTES = BN * BK;                  // 30 KB
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;    // 46 KB (a multiple of 1024: swizzle-atom aligned)
constexpr int GROUP = 8;                          // target tiles per work unit
constexpr int MAX_TILES = 256;                    // tile descriptors per launch (staged in shared memory)
constexpr int DESC_BYTES = MAX_TILES * 32;
constexpr int BAR_BYTES = 512;
constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + 1024 + BAR_BYTES + DESC_BYTES;
constexpr int EPI_WARPS = 12;            // epilogue warps: 3 per TMEM lane quarter, one column part each
constexpr int EPI_THREADS = EPI_WARPS * 32;
constexpr int THREADS = 64 + EPI_THREADS; // TMA warp, MMA warp, epilogue warps
constexpr int HALF = BN / (EPI_WARPS / 4); // 80 target columns per epilogue thread
constexpr int PARTS = EPI_WARPS / 4;      // column parts = partial vectors per (group, one-hot row)
constexpr int TMEM_COLS = 512;            // 2 accumulator buffers x 240 columns + scale factors
constexpr int SF_COL = 2 * BN;            // 8 columns of UE8M0 1.0 (0x7f) for both operands' block scales
// CTA pairs (merged-plane kernel): tiles of <= 224 target rows, each CTA stages half of them (7 chunks of 16)
constexpr int CG2_BN = 224;
constexpr int CG2_B_BYTES = (CG2_BN / 2) * BK;   // 14 KB
constexpr int CG2_STAGES = 6;
constexpr int CG2_SMEM_BYTES = CG2_STAGES * (A_BYTES + CG2_B_BYTES) + 1024 + BAR_BYTES;
static_assert(CG2_B_BYTES % 1024 == 0 && CG2_SMEM_BYTES <= 232448, "pair stage shape");
// Permuted mask box of the merged kernel (see above the kernel): target rows (e, j, g, chunk) with row strides 1, 4, 2,
// 16; each CTA's box covers its half of a tile's chunks, the second CTA's from chunk CG2_BN / 32 on.
constexpr uint32_t kMaskStride[4] = {1, 4, 2, 16};
constexpr uint32_t kMaskBox[4] = {2, 4, 2, CG2_BN / 32};
// How far past a tile's first row a mask box reaches: BN - 1 rows for the 2-D box (which TMA also clips at the map's R
// rows), kMaskReach = 223 for the permuted box (not clipped: its row index is split over four dimensions).  The masks
// carry kAccumMaskPadRows rows of padding behind them for this.
constexpr uint32_t kMaskReach = (kMaskBox[0] - 1) * kMaskStride[0] + (kMaskBox[1] - 1) * kMaskStride[1] +
                                (kMaskBox[2] - 1) * kMaskStride[2] + (CG2_BN / 32 + kMaskBox[3] - 1) * kMaskStride[3];
static_assert(BN - 1 < kAccumMaskPadRows && kMaskReach < kAccumMaskPadRows, "mask box reaches past the mask padding");

// A tile of target rows and the K blocks (of 128 samples) its two masks can be non-zero in:
// hit mask: blocks [hb0, hb1); miss mask: blocks [0, ib0) and [ib1, num_k_blocks).
struct __align__(16) TileDesc {
    int32_t row0, rows;     // target rows [row0, row0 + rows) of this launch's R rows
    int32_t hb0, hb1, ib0, ib1;
    int32_t pad0, pad1;
};
static_assert(sizeof(TileDesc) == 32, "TileDesc layout");
// merged-plane kernel: the tile table travels as a kernel parameter (constant bank, uniform loads)
constexpr int MERGED_MAX_TILES = 112;
struct TileTable {
    TileDesc t[MERGED_MAX_TILES];
};
// 16 epilogue warps (four per TMEM lane quarter = four column parts; chunks of 16 targets are dealt to the parts
// round-robin, at most M_CHUNKS each), then the producer and the MMA issuer
constexpr int M_EPI_WARPS = 16, M_PARTS = M_EPI_WARPS / 4, M_CHUNKS = (BN / 16 + M_PARTS - 1) / M_PARTS;
constexpr int M_THREADS = 32 * (M_EPI_WARPS + 2);
constexpr int PRODUCER_WARP = M_EPI_WARPS, MMA_WARP = M_EPI_WARPS + 1;
// the kernel's parameters (three tensor maps, the table, ~15 scalars) must stay within the classic 4 KB
static_assert(sizeof(TileTable) <= 3584, "tile table too large for the kernel parameter space");
static_assert(STAGE_BYTES % 1024 == 0 && HALF % 16 == 0 && SF_COL + 8 <= TMEM_COLS, "tile shape");

// Fixed-point image of a per-target coefficient c (|c| <= 1): C = round(c * 2^52) split into a
// signed high limb and a 26-bit low limb, so that c * t for an integer t is accumulated EXACTLY
// in two int64 sums (sum t*Chi, sum t*Clo) with integer multiply-adds.  No float64 instruction
// is left in the epilogue's inner loop: on B200 DADD/DFMA and the tensor pipe could not be kept
// busy at the same time (ncu on the earlier float64 epilogue: math-pipe throttle on every FP64
// instruction while the MMA issuer waited for the epilogue; FP64 time and MMA time added up
// instead of overlapping).
constexpr int kLimbBits = 26;            // C = round(c * 2^52) = Chi * 2^26 + Clo
__device__ __forceinline__ int2 coef_limbs(double c) {
    const long long C = __double2ll_rn(c * 4503599627370496.0);       // 2^52
    return make_int2((int)(C >> kLimbBits), (int)(C & ((1LL << kLimbBits) - 1)));
}
}  // namespace

// Per-target constants of every work item, laid out per (tile, phase) with a stride of 256
// targets: limbs[.] = fixed-point (Chi, Clo) of the item's coefficient (-aH for the hit phase,
// +aM for the miss phase), rsum[.] = the mask's row sum.  Targets beyond the tile's rows get
// zeros.  Written once per launch so that the accumulation epilogue reads them with uniform
// (broadcast) loads instead of staging them through shared memory behind a barrier per item.
__global__ void __launch_bounds__(256) accum_consts_kernel(const TileDesc *__restrict__ tiles, int num_tiles,
                                                           const RowInfo *__restrict__ rinfo, int2 *__restrict__ limbs,
                                                           int32_t *__restrict__ rsum, int rsum_as_float) {
    const int t = blockIdx.x >> 1, phase = blockIdx.x & 1, e = threadIdx.x;
    if (t >= num_tiles) return;
    const TileDesc d = tiles[t];
    double c = 0.0;
    int rs = 0;
    if (e < d.rows) {
        const RowInfo ri = rinfo[d.row0 + e];
        c = phase == 0 ? ri.coef[FS_MASK_NEAR_HIT] : ri.coef[FS_MASK_NEAR_MISS];
        rs = phase == 0 ? ri.n_hit - ri.n_far_hit : ri.n_miss - ri.n_far_miss;
    }
    limbs[(size_t)blockIdx.x * 256 + e] = coef_limbs(c);
    // the paired epilogue works on the FP32 accumulators directly: |rs| <= n < 2^22 is exact in float;
    // the merged-plane epilogue (rsum_as_float = 2) wants it with the float -> int bias already added
    rsum[(size_t)blockIdx.x * 256 + e] =
        rsum_as_float == 2 ? __float_as_int((float)rs + 12582912.0f) : (rsum_as_float ? __float_as_int((float)rs) : rs);
}

// kPair: every active column has exactly three values, so one-hot rows 2c and 2c + 1 (two adjacent
// TMEM lanes = two adjacent threads of an epilogue warp) are the two reduced planes of column c.  Per
// (column, target) only ONE of rs - G0, rs - G1, G0 + G1 is needed, times the coefficient once: the two
// threads swap accumulators with one shuffle and each finishes half of the targets, instead of each
// paying the whole select / convert / scale sequence for every target of its own plane.
template <bool kPair>
__global__ void __launch_bounds__(THREADS, 1)
tc_accum_kernel(const __grid_constant__ CUtensorMap tmap_at, const __grid_constant__ CUtensorMap tmap_mh,
                const __grid_constant__ CUtensorMap tmap_mm, int num_k_blocks, int64_t R,
                const TileDesc *__restrict__ tiles, int num_tiles, int groups, int group_tiles, int m_blocks,
                const int64_t *__restrict__ ids, int contiguous, const int2 *__restrict__ limbs,
                const int32_t *__restrict__ rsum, const uint8_t *__restrict__ codesT, int64_t ldt,
                const uint32_t *__restrict__ krow, int64_t K_rows, double *__restrict__ tpartial) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    // pointer arithmetic only (no integer round trip), so the compiler keeps the shared address space
    unsigned char *smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem + STAGES * STAGE_BYTES);
    uint64_t *empty_bar = full_bar + STAGES;
    uint64_t *tfull_bar = empty_bar + STAGES;     // [2] accumulator buffer ready
    uint64_t *tempty_bar = tfull_bar + 2;         // [2] accumulator buffer drained
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty_bar + 2);
    // per-target constants of the work item being drained: [2][BN] x {double c; int rs}
    unsigned char *s_desc = smem + STAGES * STAGE_BYTES + BAR_BYTES;
    const TileDesc *s_tiles = reinterpret_cast<const TileDesc *>(s_desc);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int units = m_blocks * groups;

    for (int i = threadIdx.x; i < num_tiles * 2; i += THREADS)
        reinterpret_cast<uint4 *>(s_desc)[i] = reinterpret_cast<const uint4 *>(tiles)[i];
    if (warp == 0 && lane == 0) {
        tc::prefetch_tmap(&tmap_at);
        tc::prefetch_tmap(&tmap_mh);
        tc::prefetch_tmap(&tmap_mm);
        for (int s = 0; s < STAGES; ++s) {
            tc::mbar_init(&full_bar[s], 1);
            tc::mbar_init(&empty_bar[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            tc::mbar_init(&tfull_bar[b], 1);
            tc::mbar_init(&tempty_bar[b], EPI_THREADS);   // all epilogue threads arrive
        }
        tc::fence_barrier_init();
    }
    if (warp == 1) tc::tmem_alloc<TMEM_COLS>(tmem_slot);
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    // block scale factors of both operands: UE8M0 1.0 everywhere (8 columns cover M = 128 and N <= 256)
    if (warp >= 2 && warp < 6) {
        for (int c = 0; c < 8; ++c) tc::tmem_st_32x1(tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + SF_COL + c, 0x7f7f7f7fu);
        tc::tmem_st_wait();
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::tc_fence_after();

    if (warp == 0) {
        // ===== TMA producer =====
        if (tc::elect_one()) {   // one thread, and the compiler knows it: uniform-register issue code
            int it = 0;
            for (int u = blockIdx.x; u < units; u += gridDim.x) {
                const int m0 = (u / groups) * BM, g = u % groups;
                const int tile_end = (g + 1) * group_tiles < num_tiles ? (g + 1) * group_tiles : num_tiles;
                for (int t = g * group_tiles; t < tile_end; ++t) {
                    const TileDesc d = s_tiles[t];
                    for (int phase = 0; phase < 2; ++phase) {
                        const CUtensorMap *tm = phase == 0 ? &tmap_mh : &tmap_mm;
                        // phase 0: [hb0, hb1); phase 1: [0, ib0) then [ib1, nkb)
                        int kb = phase == 0 ? d.hb0 : (d.ib0 > 0 ? 0 : d.ib1);
                        const int kend = phase == 0 ? d.hb1 : num_k_blocks;
                        while (kb < kend) {
                            const int s = it % STAGES;
                            const uint32_t ph = (it / STAGES) & 1;
                            ++it;
                            tc::mbar_wait(&empty_bar[s], ph ^ 1);
                            unsigned char *st = smem + s * STAGE_BYTES;
                            tc::mbar_arrive_expect_tx(&full_bar[s], STAGE_BYTES);
                            tc::tma_load_2d(st, &tmap_at, &full_bar[s], kb * BK, m0);
                            tc::tma_load_2d(st + A_BYTES, tm, &full_bar[s], kb * BK, d.row0);
                            ++kb;
                            if (phase == 1 && kb == d.ib0) kb = d.ib1;
                        }
                    }
                }
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer =====
        if (tc::elect_one()) {   // one thread, and the compiler knows it: uniform-register issue code
            int it = 0, item = 0;
            for (int u = blockIdx.x; u < units; u += gridDim.x) {
                const int g = u % groups;
                const int tile_end = (g + 1) * group_tiles < num_tiles ? (g + 1) * group_tiles : num_tiles;
                for (int t = g * group_tiles; t < tile_end; ++t) {
                    const TileDesc d = s_tiles[t];
                    // a partial tile (class tail) only needs N = its row count rounded up to 16
                    const uint32_t idesc = tc::make_idesc_mxf4(BM, ((d.rows + 15) >> 4) << 4);
                    for (int phase = 0; phase < 2; ++phase) {
                        const int nblk = phase == 0 ? d.hb1 - d.hb0 : d.ib0 + (num_k_blocks - d.ib1);
                        if (nblk == 0) continue;                          // mask is all zero: nothing to add
                        const int buf = item & 1;
                        const uint32_t tph = (item >> 1) & 1;
                        ++item;
                        tc::mbar_wait(&tempty_bar[buf], tph ^ 1);     // epilogue has drained this buffer
                        tc::tc_fence_after();
                        const uint32_t acc = tmem_base + (uint32_t)(buf * BN);
                        uint32_t have = 0;
                        for (int b = 0; b < nblk; ++b) {
                            const int s = it % STAGES;
                            const uint32_t ph = (it / STAGES) & 1;
                            ++it;
                            tc::mbar_wait(&full_bar[s], ph);
                            tc::tc_fence_after();
                            const uint32_t sa = tc::smem_u32(smem + s * STAGE_BYTES);
                            const uint64_t da = tc::make_smem_desc_sw128(sa);
                            const uint64_t db = tc::make_smem_desc_sw128(sa + A_BYTES);
#pragma unroll
                            for (int k = 0; k < BK / 32; ++k) {
                                tc::mma_mxf4(acc, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, tmem_base + SF_COL,
                                             tmem_base + SF_COL, have);
                                have = 1;
                            }
                            tc::tc_commit(&empty_bar[s]);
                        }
                        tc::tc_commit(&tfull_bar[buf]);
                    }
                }
            }
        }
    } else {
        // ===== epilogue (warps 2..: lane quarter = warp % 4, column part = (warp - 2) / 4) =====
        // thread = one-hot row (TMEM lane) x one part of the work item's 256 target columns
        const int q = warp & 3;
        const int half = (warp - 2) >> 2;
        const int et = q * 32 + lane;                         // 0..127: TMEM lane / local one-hot row
        const uint32_t parity = (uint32_t)lane & 1u;          // kPair: plane of this one-hot row (row 2c + parity)
        const int64_t ids0 = contiguous ? ids[0] : 0;
        int item = 0;
        for (int u = blockIdx.x; u < units; u += gridDim.x) {
            const int g = u % groups;
            const int tile_end = (g + 1) * group_tiles < num_tiles ? (g + 1) * group_tiles : num_tiles;
            const int64_t mrow = (int64_t)(u / groups) * BM + et;
            const bool row_live = mrow < K_rows;
            // this one-hot row's column (codesT row), value code and the column's last code
            const uint32_t meta = row_live ? krow[mrow] : 0u;
            const uint8_t *at_row = codesT + (int64_t)(meta & 0xffffffu) * ldt;
            const uint32_t own4 = ((meta >> 24) & 0xfu) * 0x01010101u;
            const uint32_t last4 = (meta >> 28) * 0x01010101u;
            const uint32_t oth4 = own4 ^ 0x01010101u;            // kPair: the partner lane's plane (codes 0 <-> 1)
            long long ah0 = 0, ah1 = 0, al0 = 0, al1 = 0;     // exact fixed-point sums (two chains)
            for (int t = g * group_tiles; t < tile_end; ++t) {
                const TileDesc d = s_tiles[t];
                // value codes of this thread's 128 targets in its column (issued before the
                // accumulator wait so the loads overlap the MMAs); shared by both phases.
                // Targets beyond the tile's rows get whatever follows: their coefficient is 0.
                // kPair: only the targets this thread finishes -- of every 16-target chunk the even lane
                // takes targets 0..7, the odd lane 8..15 -- i.e. two words per chunk.
                uint32_t oh[kPair ? HALF / 8 : HALF / 4];
                if constexpr (kPair) {
                    const int64_t rbase = (int64_t)d.row0 + half * HALF + 8 * (int)parity;
                    if (contiguous) {
                        const int64_t id0 = ids0 + rbase;
                        if ((id0 & 7) == 0) {
#pragma unroll
                            for (int j = 0; j < HALF / 16; ++j) {
                                const uint2 a = *reinterpret_cast<const uint2 *>(at_row + id0 + 16 * j);
                                oh[2 * j] = a.x; oh[2 * j + 1] = a.y;
                            }
                        } else {
                            // unaligned start (class-aligned tiles): aligned words + funnel shift
                            const uint32_t *src = reinterpret_cast<const uint32_t *>(at_row + (id0 & ~(int64_t)3));
                            const uint32_t sh = (uint32_t)(id0 & 3) * 8u;
#pragma unroll
                            for (int j = 0; j < HALF / 16; ++j) {
                                const uint32_t w0 = src[4 * j], w1 = src[4 * j + 1], w2 = src[4 * j + 2];
                                oh[2 * j] = __funnelshift_r(w0, w1, sh);
                                oh[2 * j + 1] = __funnelshift_r(w1, w2, sh);
                            }
                        }
                    } else {
#pragma unroll
                        for (int w = 0; w < HALF / 8; ++w) {
                            uint32_t x = 0;
#pragma unroll
                            for (int b = 0; b < 4; ++b) {
                                const int64_t r = rbase + (w >> 1) * 16 + (w & 1) * 4 + b;
                                const uint32_t byte = r < R ? (uint32_t)at_row[ids[r]] : 0xffu;
                                x |= byte << (8 * b);
                            }
                            oh[w] = x;
                        }
                    }
                } else {
                    const int64_t rbase = (int64_t)d.row0 + half * HALF;
                    if (contiguous) {
                        const int64_t id0 = ids0 + rbase;
                        if ((id0 & 15) == 0) {
                            const uint4 *src = reinterpret_cast<const uint4 *>(at_row + id0);
#pragma unroll
                            for (int w = 0; w < HALF / 16; ++w) {
                                const uint4 a = src[w];
                                oh[4 * w] = a.x; oh[4 * w + 1] = a.y; oh[4 * w + 2] = a.z; oh[4 * w + 3] = a.w;
                            }
                        } else {
                            // unaligned start (class-aligned tiles): aligned words + funnel shift
                            const uint32_t *src = reinterpret_cast<const uint32_t *>(at_row + (id0 & ~(int64_t)3));
                            const uint32_t sh = (uint32_t)(id0 & 3) * 8u;
                            uint32_t prev = src[0];
#pragma unroll
                            for (int w = 0; w < HALF / 4; ++w) {
                                const uint32_t next = src[w + 1];
                                oh[w] = __funnelshift_r(prev, next, sh);
                                prev = next;
                            }
                        }
                    } else {
#pragma unroll
                        for (int w = 0; w < HALF / 4; ++w) {
                            uint32_t x = 0;
#pragma unroll
                            for (int b = 0; b < 4; ++b) {
                                const int64_t r = rbase + w * 4 + b;
                                const uint32_t byte = r < R ? (uint32_t)at_row[ids[r]] : 0xffu;
                                x |= byte << (8 * b);
                            }
                            oh[w] = x;
                        }
                    }
                }
                for (int phase = 0; phase < 2; ++phase) {
                    const int nblk = phase == 0 ? d.hb1 - d.hb0 : d.ib0 + (num_k_blocks - d.ib1);
                    if (nblk == 0) continue;
                    const int buf = item & 1;
                    const uint32_t tph = (item >> 1) & 1;
                    ++item;
                    // per-target constants of this work item (accum_consts_kernel): uniform loads
                    const int2 *s_c = limbs + ((size_t)t * 2 + phase) * 256;
                    const int32_t *s_rs = rsum + ((size_t)t * 2 + phase) * 256;
                    tc::mbar_wait(&tfull_bar[buf], tph);
                    tc::tc_fence_after();
                    const uint32_t tacc = tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)(buf * BN + half * HALF);
#pragma unroll
                    for (int c0 = 0; c0 < HALF; c0 += 16) {
                        uint32_t v[16];                    // FP32 accumulators holding exact integers
                        tc::tmem_ld_32x16(tacc + c0, v);
                        tc::tmem_ld_wait();
                        if constexpr (kPair) {
                            // even lane (plane 0) finishes targets c0 .. c0+7, odd lane (plane 1) c0+8 .. c0+15:
                            // each sends the partner the accumulators of the partner's targets
                            uint32_t mine[8], oth[8];
#pragma unroll
                            for (int e = 0; e < 8; ++e) {
                                const uint32_t snd = parity ? v[e] : v[8 + e];
                                mine[e] = parity ? v[8 + e] : v[e];
                                oth[e] = __shfl_xor_sync(0xffffffffu, snd, 1);
                            }
                            const int4 *cc = reinterpret_cast<const int4 *>(s_c + half * HALF + c0 + 8 * (int)parity);
                            const float4 *rr = reinterpret_cast<const float4 *>(s_rs + half * HALF + c0 + 8 * (int)parity);
#pragma unroll
                            for (int e = 0; e < 8; e += 4) {
                                const uint32_t w = oh[(c0 >> 3) + (e >> 2)];
                                // own: the target carries this lane's plane; otr: the partner's plane; else the last value
                                const uint32_t own = __vcmpeq4(w, own4), otr = __vcmpeq4(w, oth4);
                                const float4 rs4 = __ldg(rr + (e >> 2));
                                const int4 ca = __ldg(cc + (e >> 1)), cb = __ldg(cc + (e >> 1) + 1);
                                const float rsv[4] = {rs4.x, rs4.y, rs4.z, rs4.w};
                                int tt[4];
#pragma unroll
                                for (int b = 0; b < 4; ++b) {
                                    const float gm = __uint_as_float(mine[e + b]), go = __uint_as_float(oth[e + b]);
                                    // t = rs - G_code for codes 0 / 1, G_0 + G_1 (= rs - G_last) for the last code: exact in
                                    // FP32; branch-free select through the 0x00 / 0xff compare bytes widened to word masks
                                    const uint32_t mo = tc::byte_mask(own, b), mt = tc::byte_mask(otr, b);
                                    const uint32_t ta = __float_as_uint(rsv[b] - gm), tb = __float_as_uint(rsv[b] - go);
                                    const uint32_t tl = __float_as_uint(gm + go);
                                    const uint32_t t1 = (ta & mo) | (tl & ~mo);
                                    tt[b] = tc::f32_to_int_exact((tb & mt) | (t1 & ~mt));
                                }
                                ah0 += (long long)tt[0] * ca.x; al0 += (long long)tt[0] * ca.y;
                                ah1 += (long long)tt[1] * ca.z; al1 += (long long)tt[1] * ca.w;
                                ah0 += (long long)tt[2] * cb.x; al0 += (long long)tt[2] * cb.y;
                                ah1 += (long long)tt[3] * cb.z; al1 += (long long)tt[3] * cb.w;
                            }
                        } else {
                        const int4 *cc = reinterpret_cast<const int4 *>(s_c + half * HALF + c0);
                        const int4 *rr = reinterpret_cast<const int4 *>(s_rs + half * HALF + c0);
#pragma unroll
                        for (int e = 0; e < 16; e += 4) {
                            const uint32_t w = oh[(c0 + e) >> 2];
                            const uint32_t own = __vcmpeq4(w, own4), lst = __vcmpeq4(w, last4);
                            const int4 rs4 = __ldg(rr + (e >> 2));
                            const int4 ca = __ldg(cc + (e >> 1)), cb = __ldg(cc + (e >> 1) + 1);   // (Chi, Clo) of two targets each
                            // t = own ? rs - G : (last ? G : 0)
                            const int g0 = tc::f32_to_int_exact(v[e]), g1 = tc::f32_to_int_exact(v[e + 1]);
                            const int g2 = tc::f32_to_int_exact(v[e + 2]), g3 = tc::f32_to_int_exact(v[e + 3]);
                            const int t0 = (own & 0x000000ffu) ? rs4.x - g0 : ((lst & 0x000000ffu) ? g0 : 0);
                            const int t1 = (own & 0x0000ff00u) ? rs4.y - g1 : ((lst & 0x0000ff00u) ? g1 : 0);
                            const int t2 = (own & 0x00ff0000u) ? rs4.z - g2 : ((lst & 0x00ff0000u) ? g2 : 0);
                            const int t3 = (own & 0xff000000u) ? rs4.w - g3 : ((lst & 0xff000000u) ? g3 : 0);
                            ah0 += (long long)t0 * ca.x; al0 += (long long)t0 * ca.y;
                            ah1 += (long long)t1 * ca.z; al1 += (long long)t1 * ca.w;
                            ah0 += (long long)t2 * cb.x; al0 += (long long)t2 * cb.y;
                            ah1 += (long long)t3 * cb.z; al1 += (long long)t3 * cb.w;
                        }
                        }
                    }
                    tc::tc_fence_before();
                    tc::mbar_arrive(&tempty_bar[buf]);
                }
            }
            // PARTS column parts per one-hot row: partial layout [group][part][row]
            // |t| <= n < 2^22 (checked by the launcher), limbs < 2^27, at most 2^11 terms per thread
            // and unit: the sums stay below 2^60
            if (row_live)
                tpartial[((int64_t)g * PARTS + half) * K_rows + mrow] =
                    ((double)(ah0 + ah1) * (double)(1 << kLimbBits) + (double)(al0 + al1)) * (1.0 / 4503599627370496.0);
        }
    }
    __syncthreads();
    if (warp == 1) {
        tc::tc_fence_after();
        tc::tmem_dealloc<TMEM_COLS>(tmem_base);
    }
}


// ------------------------------------------------------------------------------------------------
// Merged-plane variant for 0/1/2 columns (every active column owns the two one-hot rows 2c, 2c + 1).
//
// The paired kernel above lets the two planes of a column meet through a shuffle; here they meet in
// ONE thread, because the operands are staged in a permuted row order and the accumulator is read with
// the 16x256b TMEM fragment (thread t <- lanes t/4 and t/4 + 8, columns 2(t%4), 2(t%4) + 1 of every
// group of 8; measured, profiles/r02_tmem_frag_probe.txt):
//   * At tile: 4-D tensor map (bytes, column mod 8, plane, column / 8): shared-memory row = TMEM lane
//     16 * (c / 8) + 8 * plane + c % 8 for the tile's column c < 64, so lanes L and L + 8 are the two planes
//     of one column;
//   * mask tile: 5-D tensor map (bytes, e, j, g, chunk) with row strides 1, 4, 2, 16: shared-memory row =
//     TMEM column 16 chunk + 8 g + 2 j + e holds target 16 chunk + 4 j + 2 g + e of the tile, so thread
//     j = t % 4 owns the four CONSECUTIVE targets 16 chunk + 4 j .. + 3 of every chunk (one aligned word of
//     codesT, two int4 of coefficient limbs, one float4 of row sums).
// Per (column, target) the thread then has G_0 and G_1 in registers and needs one of rs - G_0, rs - G_1,
// G_0 + G_1 (selected by the target's own code) times the coefficient: no shuffle, no swap of
// accumulators, the float -> int bias rides on the row sum, and a thread serves two columns (lane
// offsets 0 and 16), i.e. two independent dependency chains.  TMEM loads and the per-target constants
// are double-buffered in registers; the accumulator buffer is handed back to the MMA issuer as soon as
// the LAST chunk is in registers (before its arithmetic).  Chunks of 16 targets are dealt to the four
// column parts (16 epilogue warps: lane quarter x part) round-robin (part, part + 4, ...), so a class-tail
// tile of 80 rows costs two chunk times instead of four.  The four threads of a column fold their sums at the
// end of a work unit and add them, as exact 64-bit integers, into the column's two slots of the partial
// buffer (one-hot row 2c: high limbs, row 2c + 1: low limbs); merged_finish_kernel converts, and the reducer of
// the older kernels is reused unchanged.
constexpr float kMagic = 12582912.0f;          // 1.5 * 2^23: float(kMagic + t) has the bits kBias + t for |t| < 2^22
constexpr int kBias = 0x4B400000;

struct ChunkConsts {
    int4 ca, cb;      // (Chi, Clo) of targets 0, 1 and 2, 3 of the thread's four
    float4 rs;        // mask row sums + kMagic
};

//
// The kernel runs as CLUSTERS OF TWO CTAs (tcgen05.mma.cta_group::2, M = 256): the pair takes two adjacent
// blocks of 128 one-hot rows through the same tiles; each CTA stages its own At block and HALF of the mask
// tile (chunks [0, nch / 2) or [nch / 2, nch), N rounded up to 32), the leader issues the MMAs for both and waits
// for both epilogues.  One CTA staging a whole tile moved 46 KB from L2 into shared memory per four MMAs -- with
// the epilogue switched off it still ran C3 in 1.12 ms against 0.78 ms of MMA time (18.5 TB/s out of L2 over the
// GPU: the same ceiling the distance GEMM hit before it became CTA pairs) -- the pair moves 30 KB.
__global__ void __launch_bounds__(M_THREADS, 1)
tc_accum_merged_kernel(const __grid_constant__ CUtensorMap tmap_at, const __grid_constant__ CUtensorMap tmap_mh,
                       const __grid_constant__ CUtensorMap tmap_mm, int num_k_blocks, int64_t R,
                       const __grid_constant__ TileTable tt, int num_tiles, int groups, int group_tiles, int m_blocks, int group_span,
                       const int64_t *__restrict__ ids, int contiguous, const int2 *__restrict__ limbs,
                       const int32_t *__restrict__ rsum, const uint8_t *__restrict__ codesT, int64_t ldt,
                       const uint32_t *__restrict__ krow, int64_t K_rows, double *__restrict__ tpartial) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char *smem = smem_raw + ((1024u - (tc::smem_u32(smem_raw) & 1023u)) & 1023u);
    constexpr int kStages = CG2_STAGES;
    constexpr int kStageBytes = A_BYTES + CG2_B_BYTES;               // At block + the mask rows this CTA stages per K block
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem + kStages * kStageBytes);
    uint64_t *empty_bar = full_bar + kStages;
    uint64_t *tfull_bar = empty_bar + kStages;    // [2] accumulator buffer ready
    uint64_t *tempty_bar = tfull_bar + 2;         // [2] accumulator buffer drained (pairs: the leader's, for both CTAs)
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(tempty_bar + 2);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    // both CTAs of a cluster walk the same units; the CTA's block of one-hot rows is 2 * (u / groups) + rank
    const uint32_t crank = tc::cluster_ctarank();
    const int worker = (int)(blockIdx.x >> 1);
    const int workers = (int)(gridDim.x >> 1);
    // work units: (block of one-hot rows, group of tiles), walked in bands of `group_span` groups: inside a band the
    // blocks advance slowest-varying-last (unit = band, block, group within band), so that the workers running at one
    // time cover group_span groups x (workers / group_span) blocks -- their mask tiles AND their At rows stay in L2
    // (group_span = groups: all groups of a block together; 1: one group for all workers)
    const int m_units = (m_blocks + 1) / 2;
    const int units = m_units * groups;
    const int band_units = m_units * group_span;
    auto unit_block = [&](int u, int &g) {
        const int band = u / band_units, rem = u - band * band_units;
        const int span = groups - band * group_span < group_span ? groups - band * group_span : group_span;
        g = band * group_span + rem % span;
        return rem / span;
    };

    if (warp == PRODUCER_WARP && lane == 0) {
        tc::prefetch_tmap(&tmap_at);
        tc::prefetch_tmap(&tmap_mh);
        tc::prefetch_tmap(&tmap_mm);
        for (int s = 0; s < kStages; ++s) {
            tc::mbar_init(&full_bar[s], 1);
            tc::mbar_init(&empty_bar[s], 1);
        }
        for (int b = 0; b < 2; ++b) {
            tc::mbar_init(&tfull_bar[b], 1);
            // one lane per epilogue warp of BOTH CTAs arrives
            tc::mbar_init(&tempty_bar[b], 2 * M_EPI_WARPS);
        }
        tc::fence_barrier_init();
    }
    if (warp == MMA_WARP) tc::tmem_alloc_pair<TMEM_COLS>(tmem_slot);
    tc::tc_fence_before();
    __syncthreads();
    tc::cluster_sync_all();                           // the peer's barriers exist before anything signals them
    tc::tc_fence_after();
    // the kernel owns ALL 512 TMEM columns, so the allocation starts at column 0, lane 0: a constant the compiler
    // can keep in uniform registers (checked here, trapped otherwise)
    if (*tmem_slot != 0u) __trap();
    constexpr uint32_t tmem_base = 0u;
    if (warp < 4) {
        for (int c = 0; c < 8; ++c) tc::tmem_st_32x1(tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + SF_COL + c, 0x7f7f7f7fu);
        tc::tmem_st_wait();
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::cluster_sync_all();                           // both CTAs' scale factors are in place before the leader issues
    tc::tc_fence_after();

    if (warp == PRODUCER_WARP) {
        // ===== TMA producer: both operands in the permuted row order described above.  elect.sync rather than
        // lane == 0 (here and in the MMA issuer): it tells the compiler that ONE thread runs the loop, so the
        // operands of the TMA / tcgen05 instructions stay in uniform registers =====
        if (tc::elect_one()) {
            int it = 0;
            for (int u = worker; u < units; u += workers) {
                int g;
                const int ub = unit_block(u, g);
                const int m0 = (ub * 2 + (int)crank) * BM;
                const int tile_end = (g + 1) * group_tiles < num_tiles ? (g + 1) * group_tiles : num_tiles;
                for (int t = g * group_tiles; t < tile_end; ++t) {
                    const TileDesc d = tt.t[t];
                    // this CTA's half of the tile's chunks of 16 target rows (N is a multiple of 32)
                    const int c_half = (int)crank * ((d.rows + 31) >> 5);
                    for (int phase = 0; phase < 2; ++phase) {
                        const CUtensorMap *tm = phase == 0 ? &tmap_mh : &tmap_mm;
                        int kb = phase == 0 ? d.hb0 : (d.ib0 > 0 ? 0 : d.ib1);
                        const int kend = phase == 0 ? d.hb1 : num_k_blocks;
                        while (kb < kend) {
                            const int s = it % kStages;
                            const uint32_t ph = (it / kStages) & 1;
                            ++it;
                            tc::mbar_wait(&empty_bar[s], ph ^ 1);
                            unsigned char *st = smem + s * kStageBytes;
                            // both CTAs' bytes are credited to the LEADER's barrier
                            if (crank == 0) tc::mbar_arrive_expect_tx(&full_bar[s], 2 * kStageBytes);
                            tc::tma_load_4d_pair(st, &tmap_at, &full_bar[s], kb * BK, 0, 0, m0 >> 4);
                            tc::tma_load_5d_pair(st + A_BYTES, tm, &full_bar[s], kb * BK, d.row0, 0, 0, c_half);
                            ++kb;
                            if (phase == 1 && kb == d.ib0) kb = d.ib1;
                        }
                    }
                }
            }
        }
    } else if (warp == MMA_WARP) {
        // ===== MMA issuer: one thread of the leader CTA, for both.  Everything the tcgen05 instructions
        // take is derived from kernel parameters (the tile table is one) and loop counters, so that it stays in
        // uniform registers: with the table in shared memory every tcgen05.mma was wrapped in an elect / broadcast
        // sequence of ~20 instructions and the issuing thread, not the tensor pipe, set the pace. =====
        if (crank == 0 && tc::elect_one()) {
            int it = 0, item = 0;
            for (int u = worker; u < units; u += workers) {
                int g;
                (void)unit_block(u, g);
                const int tile_end = (g + 1) * group_tiles < num_tiles ? (g + 1) * group_tiles : num_tiles;
                for (int t = g * group_tiles; t < tile_end; ++t) {
                    const TileDesc d = tt.t[t];
                    const uint32_t idesc = tc::make_idesc_mxf4(2 * BM, ((d.rows + 31) >> 5) << 5);
                    for (int phase = 0; phase < 2; ++phase) {
                        const int nblk = phase == 0 ? d.hb1 - d.hb0 : d.ib0 + (num_k_blocks - d.ib1);
                        if (nblk == 0) continue;
                        const int buf = item & 1;
                        const uint32_t tph = (item >> 1) & 1;
                        ++item;
                        tc::mbar_wait(&tempty_bar[buf], tph ^ 1);
                        tc::tc_fence_after();
                        const uint32_t acc = tmem_base + (uint32_t)(buf * BN);
                        uint32_t have = 0;
                        for (int b = 0; b < nblk; ++b) {
                            const int s = it % kStages;
                            const uint32_t ph = (it / kStages) & 1;
                            ++it;
                            tc::mbar_wait(&full_bar[s], ph);
                            tc::tc_fence_after();
                            const uint32_t sa = tc::smem_u32(smem + s * kStageBytes);
                            const uint64_t da = tc::make_smem_desc_sw128(sa);
                            const uint64_t db = tc::make_smem_desc_sw128(sa + A_BYTES);
#pragma unroll
                            for (int k = 0; k < BK / 32; ++k) {
                                tc::mma_mxf4_pair(acc, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, tmem_base + SF_COL,
                                                  tmem_base + SF_COL, have);
                                have = 1;
                            }
                            tc::tc_commit_pair(&empty_bar[s]);
                        }
                        tc::tc_commit_pair(&tfull_bar[buf]);
                    }
                }
            }
        }
    } else {
        // ===== epilogue (warps 0 .. 11: lane quarter = warp % 4, column part = warp / 4).  The producer and the MMA
        // issuer are the LAST two warps: the schedulers favour the highest warp id, and these two must never
        // queue behind epilogue arithmetic. =====
        const int q = warp & 3;
        const int part = warp >> 2;
        const int j = lane & 3, r8 = lane >> 2;
        const int64_t ids0 = contiguous ? ids[0] : 0;
        const uint32_t tquarter = tmem_base + ((uint32_t)(q * 32) << 16);
        // hand an accumulator buffer back to the MMA issuer (this thread's TMEM loads have completed)
        auto release_acc = [&](uint64_t *bar) {
            tc::tc_fence_before();
            __syncwarp();
            if (lane == 0) tc::mbar_arrive_cluster_relaxed(bar, 0);   // no memory fence: TMEM reads are ordered by tcgen05.fence
        };
        int item = 0;
        for (int u = worker; u < units; u += workers) {
            int g;
            const int ub = unit_block(u, g);
            const int tile_end = (g + 1) * group_tiles < num_tiles ? (g + 1) * group_tiles : num_tiles;
            // this thread's two columns: the tile's columns (2q + h) * 8 + r8, h = 0, 1 (lane offsets 0, 16)
            const int64_t mrow0 = (int64_t)(ub * 2 + (int)crank) * BM + 2 * ((2 * q) * 8 + r8);
            const int64_t mrow1 = mrow0 + 16;
            const uint8_t *at0 = codesT + (int64_t)((mrow0 < K_rows ? krow[mrow0] : 0u) & 0xffffffu) * ldt;
            const uint8_t *at1 = codesT + (int64_t)((mrow1 < K_rows ? krow[mrow1] : 0u) & 0xffffffu) * ldt;
            unsigned long long ah0 = 0, al0 = 0, ah1 = 0, al1 = 0;   // exact fixed-point sums, one pair per column
            for (int t = g * group_tiles; t < tile_end; ++t) {
                const TileDesc d = tt.t[t];
                const int nch = ((d.rows + 31) >> 5) << 1;   // chunks of 16 targets in this tile (N rounded up to 32)
                const int n_my = nch > part ? (nch - part + M_PARTS - 1) / M_PARTS : 0;   // this part's chunks: part, part + M_PARTS, ...
                // value codes of the thread's targets in its two columns: one word per chunk and column
                // (issued before the accumulator wait; shared by both phases).  Targets beyond the tile's
                // rows get whatever follows: their coefficient is 0.
                uint32_t oh0[M_CHUNKS], oh1[M_CHUNKS];
                if (contiguous) {
                    const int64_t a0 = ids0 + d.row0 + 16 * part + 4 * j;   // chunk i: + 16 M_PARTS i
                    if ((a0 & 3) == 0) {
#pragma unroll
                        for (int i = 0; i < M_CHUNKS; ++i)
                            if (i < n_my) {
                                oh0[i] = *reinterpret_cast<const uint32_t *>(at0 + a0 + 16 * M_PARTS * i);
                                oh1[i] = *reinterpret_cast<const uint32_t *>(at1 + a0 + 16 * M_PARTS * i);
                            }
                    } else {
                        // unaligned start (class-aligned tiles): two aligned words + funnel shift
                        const uint32_t sh = (uint32_t)(a0 & 3) * 8u;
                        const int64_t ab = a0 & ~(int64_t)3;
#pragma unroll
                        for (int i = 0; i < M_CHUNKS; ++i)
                            if (i < n_my) {
                                const uint32_t *s0 = reinterpret_cast<const uint32_t *>(at0 + ab + 16 * M_PARTS * i);
                                const uint32_t *s1 = reinterpret_cast<const uint32_t *>(at1 + ab + 16 * M_PARTS * i);
                                oh0[i] = __funnelshift_r(s0[0], s0[1], sh);
                                oh1[i] = __funnelshift_r(s1[0], s1[1], sh);
                            }
                    }
                } else {
#pragma unroll
                    for (int i = 0; i < M_CHUNKS; ++i)
                        if (i < n_my) {
                            uint32_t x0 = 0, x1 = 0;
#pragma unroll
                            for (int b = 0; b < 4; ++b) {
                                const int64_t r = (int64_t)d.row0 + 16 * (part + M_PARTS * i) + 4 * j + b;
                                const int64_t id = r < R ? ids[r] : -1;
                                x0 |= (id >= 0 ? (uint32_t)at0[id] : 0xffu) << (8 * b);
                                x1 |= (id >= 0 ? (uint32_t)at1[id] : 0xffu) << (8 * b);
                            }
                            oh0[i] = x0;
                            oh1[i] = x1;
                        }
                }
                for (int phase = 0; phase < 2; ++phase) {
                    const int nblk = phase == 0 ? d.hb1 - d.hb0 : d.ib0 + (num_k_blocks - d.ib1);
                    if (nblk == 0) continue;
                    const int buf = item & 1;
                    const uint32_t tph = (item >> 1) & 1;
                    ++item;
                    // per-target constants of this work item (accum_consts_kernel), target 16 chunk + 4 j + b
                    const int2 *s_c = limbs + ((size_t)t * 2 + phase) * 256 + 16 * part + 4 * j;
                    const float *s_rs = reinterpret_cast<const float *>(rsum) + ((size_t)t * 2 + phase) * 256 + 16 * part + 4 * j;
                    ChunkConsts kc{}, kn{};
                    if (n_my > 0) {
                        kc.ca = __ldg(reinterpret_cast<const int4 *>(s_c));
                        kc.cb = __ldg(reinterpret_cast<const int4 *>(s_c + 2));
                        kc.rs = __ldg(reinterpret_cast<const float4 *>(s_rs));
                    }
                    kn = kc;
                    tc::mbar_wait(&tfull_bar[buf], tph);
                    tc::tc_fence_after();
                    const uint32_t tacc = tquarter + (uint32_t)(buf * BN + 16 * part);   // chunk i: + 16 M_PARTS i
                    // v[buffer][column h][group g of 8 TMEM columns][r0..r3]
                    uint32_t v[2][2][2][4];
                    if (n_my > 0) {
                        tc::tmem_ld_16x256b(tacc, v[0][0][0]);
                        tc::tmem_ld_16x256b(tacc + 8, v[0][0][1]);
                        tc::tmem_ld_16x256b(tacc + (16u << 16), v[0][1][0]);
                        tc::tmem_ld_16x256b(tacc + (16u << 16) + 8, v[0][1][1]);
                    } else {
                        release_acc(&tempty_bar[buf]);
                    }
#pragma unroll
                    for (int i = 0; i < M_CHUNKS; ++i) {
                        if (i < n_my) {
                            uint32_t (&vc)[2][2][4] = v[i & 1];
                            tc::tmem_ld_wait_on(vc[0][0], vc[0][1], vc[1][0], vc[1][1]);
                            if (i + 1 < n_my) {
                                uint32_t (&vn)[2][2][4] = v[(i + 1) & 1];
                                const uint32_t ta = tacc + 16 * M_PARTS * (i + 1);
                                tc::tmem_ld_16x256b(ta, vn[0][0]);
                                tc::tmem_ld_16x256b(ta + 8, vn[0][1]);
                                tc::tmem_ld_16x256b(ta + (16u << 16), vn[1][0]);
                                tc::tmem_ld_16x256b(ta + (16u << 16) + 8, vn[1][1]);
                                kn.ca = __ldg(reinterpret_cast<const int4 *>(s_c + 16 * M_PARTS * (i + 1)));
                                kn.cb = __ldg(reinterpret_cast<const int4 *>(s_c + 16 * M_PARTS * (i + 1) + 2));
                                kn.rs = __ldg(reinterpret_cast<const float4 *>(s_rs + 16 * M_PARTS * (i + 1)));
                            } else {
                                // the last chunk is in registers: the MMA issuer may reuse the buffer
                                release_acc(&tempty_bar[buf]);
                            }
                            const int chi[4] = {kc.ca.x, kc.ca.z, kc.cb.x, kc.cb.z};
                            const int clo[4] = {kc.ca.y, kc.ca.w, kc.cb.y, kc.cb.w};
                            const float rsb[4] = {kc.rs.x, kc.rs.y, kc.rs.z, kc.rs.w};
#pragma unroll
                            for (int h = 0; h < 2; ++h) {
                                const uint32_t w = h == 0 ? oh0[i] : oh1[i];
#pragma unroll
                                for (int b = 0; b < 4; ++b) {
                                    // target 4 j + b of the chunk sits in TMEM column 8 (b / 2) + 2 j + b % 2
                                    const float g0 = __uint_as_float(vc[h][b >> 1][b & 1]);
                                    const float g1 = __uint_as_float(vc[h][b >> 1][2 + (b & 1)]);
                                    const bool c1 = (w & (1u << (8 * b))) != 0;      // the target's code is 1
                                    const bool c2 = (w & (2u << (8 * b))) != 0;      // ... is 2 (the implied plane)
                                    // biased t: rs - G_code for codes 0 / 1, G_0 + G_1 (= rs - G_last) for code 2
                                    const float t01 = __fsub_rn(rsb[b], c1 ? g1 : g0);
                                    const float tl = __fadd_rn(__fadd_rn(g0, kMagic), g1);
                                    const int ti = __float_as_int(c2 ? tl : t01) - kBias;
                                    if (h == 0) {
                                        ah0 += (unsigned long long)((long long)ti * chi[b]);
                                        al0 += (unsigned long long)((long long)ti * clo[b]);
                                    } else {
                                        ah1 += (unsigned long long)((long long)ti * chi[b]);
                                        al1 += (unsigned long long)((long long)ti * clo[b]);
                                    }
                                }
                            }
                            kc = kn;
                        }
                    }
                }
            }
            // the four threads j of a column fold their sums; |t| <= n < 2^22 (checked by the launcher),
            // limbs < 2^27, at most 2^9 terms per thread and unit: no overflow
#pragma unroll
            for (int o = 1; o <= 2; o <<= 1) {
                ah0 += __shfl_xor_sync(0xffffffffu, ah0, o);
                al0 += __shfl_xor_sync(0xffffffffu, al0, o);
                ah1 += __shfl_xor_sync(0xffffffffu, ah1, o);
                al1 += __shfl_xor_sync(0xffffffffu, al1, o);
            }
            // exact integers, so the order of the additions does not matter: one pair of 64-bit sums per column for the
            // whole launch (slot of one-hot row 2c: high limbs, of row 2c + 1: low limbs), added with fire-and-forget
            // atomics; merged_finish_kernel turns them into doubles.  No float64 instruction in this kernel.
            if (j == 0) {
                unsigned long long *out = reinterpret_cast<unsigned long long *>(tpartial);
                if (mrow0 < K_rows) {
                    atomicAdd(out + mrow0, ah0);
                    atomicAdd(out + mrow0 + 1, al0);
                }
                if (mrow1 < K_rows) {
                    atomicAdd(out + mrow1, ah1);
                    atomicAdd(out + mrow1 + 1, al1);
                }
            }
        }
    }
    __syncthreads();
    tc::cluster_sync_all();                           // neither CTA leaves (or frees TMEM) while the pair is in flight
    if (warp == MMA_WARP) {
        tc::tc_fence_after();
        tc::tmem_dealloc_pair<TMEM_COLS>(tmem_base);
    }
}

// (sum of high limbs, sum of low limbs) of every column -> its weight as a double in the slot of one-hot row 2c, 0 in
// the slot of row 2c + 1: the layout reduce_tensor_partials_kernel expects (one partial vector)
__global__ void __launch_bounds__(256) merged_finish_kernel(double *__restrict__ tpartial, int64_t K_rows) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (2 * c + 1 >= K_rows) return;
    const long long hi = reinterpret_cast<const long long *>(tpartial)[2 * c];
    const long long lo = reinterpret_cast<const long long *>(tpartial)[2 * c + 1];
    tpartial[2 * c] = ((double)hi * (double)(1 << kLimbBits) + (double)lo) * (1.0 / 4503599627370496.0);
    tpartial[2 * c + 1] = 0.0;
}

// Host plan: class-aligned tiles of <= 256 target rows and the K blocks their masks need.
struct AccumPlan {
    std::vector<TileDesc> tiles;
    double blocks = 0;       // K blocks contracted per one-hot row block (both phases, all tiles), in units of full 256-column tiles
};

static AccumPlan make_plan(int64_t n, int64_t R, bool contiguous, const int64_t *h_ids, const int32_t *h_y,
                           const int64_t *h_cls_start, int bn, int n_round) {
    AccumPlan plan;
    const int nkb = (int)ceil_div(n, KS);
    auto add = [&](int64_t row0, int64_t rows, int64_t hs, int64_t he, bool mixed) {
        TileDesc d{};
        d.row0 = (int32_t)row0;
        d.rows = (int32_t)rows;
        if (mixed) {
            d.hb0 = 0; d.hb1 = nkb; d.ib0 = nkb; d.ib1 = nkb;      // both masks over every block
        } else {
            d.hb0 = (int32_t)(hs / KS);
            d.hb1 = (int32_t)ceil_div(he, KS);
            // blocks entirely inside [hs, he) hold no misses of this class
            d.ib0 = (int32_t)ceil_div(hs, KS);
            d.ib1 = he == n ? nkb : (int32_t)(he / KS);
            if (d.ib1 < d.ib0) d.ib1 = d.ib0;
        }
        // MMA N: the tile's rows rounded up to n_round (16; CTA pairs 32), in units of full 240-column tiles
        plan.blocks += (double)((d.hb1 - d.hb0) + d.ib0 + (nkb - d.ib1)) * (double)(ceil_div(rows, n_round) * n_round) / BN;
        plan.tiles.push_back(d);
    };
    if (!contiguous) {
        for (int64_t r = 0; r < R; r += bn) add(r, std::min<int64_t>(bn, R - r), 0, n, true);
        return plan;
    }
    const int64_t id0 = h_ids[0];
    int64_t r = 0;
    while (r < R) {
        const int c = h_y[id0 + r];
        const int64_t cls_end = std::min<int64_t>(h_cls_start[c + 1] - id0, R);   // first row past this class
        for (; r < cls_end; r += bn) add(r, std::min<int64_t>(bn, cls_end - r), h_cls_start[c], h_cls_start[c + 1], false);
        r = cls_end;
    }
    return plan;
}

// wsum[tout[c]] += sum over groups g and one-hot rows of column c of tpartial[g, row]
__global__ void __launch_bounds__(256) reduce_tensor_partials_kernel(const double *__restrict__ tpartial, int groups,
                                                                     int64_t K_rows, const int32_t *__restrict__ toff,
                                                                     const int64_t *__restrict__ tout, int64_t pt,
                                                                     double *__restrict__ wsum) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= pt) return;
    double s = 0.0;
    for (int g = 0; g < groups; ++g)
        for (int r = toff[c]; r < toff[c + 1]; ++r) s += tpartial[(int64_t)g * K_rows + r];
    wsum[tout[c]] += s;
}

void launch_accum_tensor(fs_dataset *ds, const WorkSet &ws, const int64_t *d_row_ids, const int64_t *h_row_ids,
                         bool contiguous, int64_t R, const int8_t *mask_h, const int8_t *mask_m, int64_t ldn,
                         const RowInfo *rinfo, double *wsum, cudaStream_t st, int *launches, double *ops) {
    const int64_t n = ds->n;
    // the accumulation operands hold the columns [a0, a1) of the active list (everything outside a
    // multi-GPU group; this rank's share inside one), one-hot rows numbered from 0
    const int64_t pa = ws.a1 - ws.a0, K_rows = ws.Ka_used;
    if (pa <= 0 || K_rows <= 0) return;
    ds->tile_desc.reserve(MAX_TILES * sizeof(TileDesc) / sizeof(int32_t));
    TileDesc *d_tiles = reinterpret_cast<TileDesc *>(ds->tile_desc.ptr);
    // K of this GEMM is the sample index; At and the masks hold FP4 nibbles: rows of (n + 1) / 2 bytes
    const uint64_t row_bytes = (uint64_t)((n + 1) / 2), pa_b = (uint64_t)(ws.ldt / 2), pm_b = (uint64_t)(ldn / 2);
    CUtensorMap tmap_at = make_tmap_u8_sw128(ws.At.ptr, row_bytes, (uint64_t)ws.Ka, pa_b, BM);
    CUtensorMap tmap_mh = make_tmap_u8_sw128(mask_h, row_bytes, (uint64_t)R, pm_b, BN);
    CUtensorMap tmap_mm = make_tmap_u8_sw128(mask_m, row_bytes, (uint64_t)R, pm_b, BN);
    // Kernel choice.  Every column with exactly three values (one-hot rows 2c, 2c + 1 are column c's two planes):
    // 3, the merged-plane kernel, whose operands are staged in a permuted row order (see above the kernel; the
    // default below n = 2^17, where its per-column 64-bit sums stay exact: n^2 * 2^27 < 2^63), or 1, the paired
    // epilogue (planes meet by shuffle).  Otherwise 0: one thread per one-hot row.  FS_B200_ACCUM_PAIR = 0 / 1 / 3
    // forces a mode for three-valued columns.
    int pair_mode = ws.all_v3 ? (n < (1 << 17) ? 3 : 1) : 0;
    if (const char *e = getenv("FS_B200_ACCUM_PAIR"))
        if (ws.all_v3 && (e[0] == '0' || e[0] == '1' || (e[0] == '3' && n < (1 << 17)))) pair_mode = e[0] - '0';
    if (pair_mode == 3) {
        const uint64_t da[4] = {row_bytes, 8, 2, (uint64_t)(ws.Ka / 16)}, sa[3] = {2 * pa_b, pa_b, 16 * pa_b};
        const uint32_t ba[4] = {BK, 8, 2, 8};
        const uint64_t dm[5] = {row_bytes, (uint64_t)R, 4, 2, CG2_BN / 16};
        const uint64_t sm[4] = {kMaskStride[0] * pm_b, kMaskStride[1] * pm_b, kMaskStride[2] * pm_b, kMaskStride[3] * pm_b};
        const uint32_t bm[5] = {BK, kMaskBox[0], kMaskBox[1], kMaskBox[2], kMaskBox[3]};
        CUtensorMap at4, mh5, mm5;
        if (make_tmap_u8_sw128_nd(&at4, ws.At.ptr, 4, da, sa, ba) && make_tmap_u8_sw128_nd(&mh5, mask_h, 5, dm, sm, bm) &&
            make_tmap_u8_sw128_nd(&mm5, mask_m, 5, dm, sm, bm)) {
            tmap_at = at4;
            tmap_mh = mh5;
            tmap_mm = mm5;
        } else {
            pair_mode = 1;   // the driver refused a permuted map: the 2-D maps and the paired epilogue still apply
        }
    }
    const bool merged = pair_mode == 3;
    auto kernel = pair_mode == 1 ? tc_accum_kernel<true> : tc_accum_kernel<false>;
    const int smem_bytes = merged ? CG2_SMEM_BYTES : SMEM_BYTES;
    if (merged) FS_CUDA(cudaFuncSetAttribute(tc_accum_merged_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    else FS_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_bytes));
    int dev = 0, sms = 0;
    FS_CUDA(cudaGetDevice(&dev));
    FS_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    FS_REQUIRE(n < (1LL << 22), FS_ERR_INVALID, "one-hot accumulation supports up to 2^22 samples (got %lld)", (long long)n);
    const AccumPlan plan = make_plan(n, R, contiguous, h_row_ids, ds->y_sorted.data(), ds->cls_start.data(),
                                     merged ? CG2_BN : BN, merged ? 32 : 16);
    const int m_blocks = (int)ceil_div(K_rows, BM);
    // Tile groups.  Work units (128 one-hot rows x one group) are dealt round-robin, so the ~sms
    // units resident at one time span sms / groups one-hot row blocks, each streaming its own
    // 128 x n bytes of At again for every tile of the group: keep that footprint within about half
    // of L2 (else every re-read goes to HBM and the kernel turns DRAM-bound for large n) by
    // cutting the tiles into more, smaller groups of equal size.
    // Merged kernel at large n (the two masks, n^2 bytes, no longer fit L2): groups of two tiles walked in bands of
    // twelve (see the kernel) keep the mask tiles and the At rows of the ~74 running clusters inside L2 -- measured
    // on a C5 cut (20 000 x 100 000): 226 -> 204 ms of accumulation per TuRF run
    // (profiles/r02_accum_l2_blocking_c5cut.txt).  Otherwise all groups of a block are walked together.
    const bool l2_bands = merged && n > 8192;
    auto groups_for = [&](int nt) {
        if (l2_bands) return (int)ceil_div(nt, 2);
        const int64_t want = ceil_div((int64_t)sms * BM * (n / 2), (int64_t)60 << 20);   // At rows are n / 2 bytes
        return (int)std::max<int64_t>(ceil_div(nt, GROUP), std::min<int64_t>(nt, want));
    };
    const size_t max_tiles = merged ? MERGED_MAX_TILES : MAX_TILES;
    int total_groups = 0;
    for (size_t t0 = 0; t0 < plan.tiles.size(); t0 += max_tiles)
        total_groups += groups_for((int)std::min<size_t>(max_tiles, plan.tiles.size() - t0));
    // merged kernel: one pair of exact 64-bit sums per column for the whole call (zeroed here, finished below)
    DevBuf<double> &tpartial = ds->tpartial;
    tpartial.reserve(merged ? (size_t)K_rows + 2 : (size_t)total_groups * PARTS * K_rows);
    if (merged) FS_CUDA(cudaMemsetAsync(tpartial.ptr, 0, (size_t)K_rows * sizeof(double), st));
    int groups_done = 0;
    // at most max_tiles tile descriptors per launch
    for (size_t t0 = 0; t0 < plan.tiles.size(); t0 += max_tiles) {
        const int nt = (int)std::min<size_t>(max_tiles, plan.tiles.size() - t0);
        // equal-sized groups (work units are dealt round-robin: unequal units would unbalance the SMs)
        const int group_tiles = (int)ceil_div(nt, groups_for(nt));
        const int groups = (int)ceil_div(nt, group_tiles);
        // pageable source: the copy is staged before cudaMemcpyAsync returns
        FS_CUDA(cudaMemcpyAsync(d_tiles, plan.tiles.data() + t0, nt * sizeof(TileDesc), cudaMemcpyHostToDevice, st));
        // per-item constants: [nt x 2 phases x 256] (Chi, Clo) pairs, then as many row sums
        ds->tile_consts.reserve((size_t)nt * 2 * 256 * 3 + 512);   // slack: the epilogue prefetches one item ahead
        int2 *limbs = reinterpret_cast<int2 *>(ds->tile_consts.ptr);
        int32_t *rsum = ds->tile_consts.ptr + (size_t)nt * 2 * 256 * 2;
        accum_consts_kernel<<<2 * nt, 256, 0, st>>>(d_tiles, nt, rinfo, limbs, rsum, merged ? 2 : pair_mode);
        ++*launches;
        if (merged) {
            // clusters of two CTAs: a cluster takes two adjacent blocks of one-hot rows through a group of tiles.
            // The tile table is a kernel parameter.
            TileTable table;
            memcpy(table.t, plan.tiles.data() + t0, (size_t)nt * sizeof(TileDesc));
            const int units = (m_blocks + 1) / 2 * groups;
            const int workers = sms / 2;
            const int group_span = l2_bands && 12 < groups ? 12 : groups;
            cudaLaunchConfig_t cfg{};
            cfg.gridDim = dim3((unsigned)(2 * (units < workers ? units : workers)));
            cfg.blockDim = dim3(M_THREADS);
            cfg.dynamicSmemBytes = (size_t)smem_bytes;
            cfg.stream = st;
            cudaLaunchAttribute attr{};
            attr.id = cudaLaunchAttributeClusterDimension;
            attr.val.clusterDim.x = 2;
            attr.val.clusterDim.y = 1;
            attr.val.clusterDim.z = 1;
            cfg.attrs = &attr;
            cfg.numAttrs = 1;
            FS_CUDA(cudaLaunchKernelEx(&cfg, tc_accum_merged_kernel, tmap_at, tmap_mh, tmap_mm, (int)ceil_div(n, KS), R, table,
                                       nt, groups, group_tiles, m_blocks, group_span, d_row_ids, contiguous ? 1 : 0,
                                       (const int2 *)limbs, (const int32_t *)rsum, ws.codesT.ptr, ws.ldt, ws.krow.ptr, K_rows, tpartial.ptr));
        } else {
            const int units = m_blocks * groups;
            const int grid = units < sms ? units : sms;
            kernel<<<grid, THREADS, smem_bytes, st>>>(
                tmap_at, tmap_mh, tmap_mm, (int)ceil_div(n, KS), R, d_tiles, nt,
                groups, group_tiles, m_blocks, d_row_ids, contiguous ? 1 : 0, limbs, rsum, ws.codesT.ptr, ws.ldt, ws.krow.ptr, K_rows,
                tpartial.ptr + (size_t)groups_done * PARTS * K_rows);
        }
        FS_CUDA(cudaGetLastError());
        ++*launches;
        groups_done += groups;
    }
    if (ops) *ops += 2.0 * BM * BN * KS * plan.blocks * (double)(merged ? (m_blocks + 1) / 2 * 2 : m_blocks);
    if (merged) {
        merged_finish_kernel<<<(unsigned)ceil_div(K_rows / 2 + 1, 256), 256, 0, st>>>(tpartial.ptr, K_rows);
        FS_CUDA(cudaGetLastError());
        ++*launches;
    }
    const int parts = merged ? 1 : PARTS * groups_done;
    reduce_tensor_partials_kernel<<<(unsigned)ceil_div(pa, 256), 256, 0, st>>>(tpartial.ptr, parts, K_rows, ws.atoff.ptr,
                                                                              ws.tout.ptr + ws.a0, pa, wsum);
    FS_CUDA(cudaGetLastError());
    ++*launches;
}

}  // namespace fs
