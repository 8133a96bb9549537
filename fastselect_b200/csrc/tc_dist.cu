// tc_dist.cu -- genotype / discrete mismatch distance on the 5th-gen tensor cores.
//
// Replaces the discrete branch of the reference's distance loops
// (MultiSURF.py:184-185, SURF.py:153-154, ReliefF.py:151-152):
//     d_ij = sum_f [x_if != x_jf] = s_i + s_j - sum_k U[i,k] * Wd[j,k],
// where U / Wd are the reduced one-hot images of the discrete columns (onehot.cu: V_f - 1
// int8 columns per feature, K = sum_f (V_f - 1)) and s_i counts the columns in which sample
// i does not carry its column's last value.  The contraction is a GEMM U * Wd^T over operands
// stored as e2m1 (FP4) nibbles -- entries 0/1 and 0/1/2 -- with unit UE8M0 block scales and FP32
// accumulation (tcgen05 kind::mxf4, twice the int8 rate): every product and every partial sum is a
// small integer, so the FP32 accumulators are exact up to 2^24 and the distances are exact.
//
// Kernel: one cluster of two CTAs (tcgen05 cta_group::2) per 256 x 256 super-block of D.  Warp 0
// of each CTA streams 128-byte-wide K slabs of its own 128 target rows and of HALF of the 256
// sample rows with TMA (128B swizzle) through a 6-stage mbarrier ring; one elected thread of the
// leader CTA's warp 1 issues tcgen05.mma.cta_group::2.kind::mxf4 (M=256, N=256, K=64) for the
// pair, which reads the B operand from both CTAs' shared memory, into a 256-column TMEM
// accumulator; commits are multicast to both CTAs' barriers.  Warps 2-5 of each CTA read its 128
// TMEM lanes back with tcgen05.ld (32 lanes x 32 columns per instruction), form s_i + s_j - acc
// and store int32 rows (each thread writes whole 128-byte lines).
// Pairs, because one CTA staging a whole 128 x 256 tile was bound by the operand feed from L2:
// about 190 cycles per M128 N256 K64 MMA against the 128 that tools/fp4_peak.cu reaches from
// resident operands.  Probed stand-alone first (tools/tc_dist_cg2_probe.cu,
// profiles/r02_tc_dist_cg2_probe_run1.txt: exact).
//
// Symmetric mode.  D is symmetric, so when the target rows of all ranks together cover every
// sample (one GPU scoring all rows, or one process per GPU each scoring its row shard) only
// half of the off-diagonal 256 x 256 super-blocks are computed: super-block (I, J), I != J, is
// computed on the rank that owns rows I iff ((I + J) even) == (J > I) -- a checkerboard that
// gives every rank the same share -- and each computed tile is stored twice: into the
// computing rank's slab, and transposed into the slab of the rank that owns rows J (a warp's 32
// lanes hold 32 consecutive rows of one column, so the mirrored store is one 128-byte line;
// for another rank it is a peer store over NVLink into that rank's slab, mapped through CUDA
// IPC).  The exchange is fused into the GEMM epilogue; a cross-rank barrier before the
// neighbour selection is all that follows.
// Tensor-pipe bound: 4 ops per (sample pair, feature) for 3-valued genotypes, half of
// that in symmetric mode.
#include "common.cuh"
#include "tc_common.cuh"

namespace fs {

// ---------------------------------------------------------------------------
// TMA descriptors (driver entry point fetched through the runtime: no -lcuda)
// ---------------------------------------------------------------------------
typedef CUresult (*EncodeTiledFn)(CUtensorMap *, CUtensorMapDataType, cuuint32_t, void *, const cuuint64_t *,
                                  const cuuint64_t *, const cuuint32_t *, const cuuint32_t *, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void *p = nullptr;
        cudaDriverEntryPointQueryResult q;
        FS_CUDA(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q));
        FS_REQUIRE(p != nullptr && q == cudaDriverEntryPointSuccess, FS_ERR_CUDA, "cuTensorMapEncodeTiled not available");
        fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

CUtensorMap make_tmap_u8_sw128(const void *base, uint64_t row_bytes, uint64_t rows, uint64_t pitch_bytes,
                               uint32_t box_rows) {
    CUtensorMap m;
    cuuint64_t dims[2] = {row_bytes, rows};
    cuuint64_t strides[1] = {pitch_bytes};
    cuuint32_t box[2] = {128, box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult rc = encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_UINT8, 2, const_cast<void *>(base), dims, strides, box, estr,
                              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                              CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    FS_REQUIRE(rc == CUDA_SUCCESS, FS_ERR_CUDA, "cuTensorMapEncodeTiled failed (%d): base=%p row_bytes=%llu rows=%llu pitch=%llu",
               (int)rc, base, (unsigned long long)row_bytes, (unsigned long long)rows, (unsigned long long)pitch_bytes);
    return m;
}

bool make_tmap_u8_sw128_nd(CUtensorMap *out, const void *base, int rank, const uint64_t *dims, const uint64_t *strides,
                           const uint32_t *box) {
    CUtensorMap m;
    cuuint64_t gd[5], gs[4];
    cuuint32_t bx[5], estr[5];
    for (int i = 0; i < rank; ++i) {
        gd[i] = dims[i];
        bx[i] = box[i];
        estr[i] = 1;
        if (i + 1 < rank) gs[i] = strides[i];
    }
    const CUresult rc = encode_fn()(&m, CU_TENSOR_MAP_DATA_TYPE_UINT8, (cuuint32_t)rank, const_cast<void *>(base), gd, gs, bx, estr,
                                    CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                                    CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (rc != CUDA_SUCCESS) return false;
    *out = m;
    return true;
}

namespace {
constexpr int BM = 128;        // target rows per CTA (half of UMMA M)
constexpr int BN = 256;        // sample columns per super-block (UMMA N)
constexpr int BK = 128;        // bytes of K per stage (one swizzle atom)
constexpr int STAGES = 6;
constexpr int A_BYTES = BM * BK;         // 16 KB
constexpr int B_BYTES = (BN / 2) * BK;   // 16 KB: this CTA's half of the sample rows
constexpr int SMEM_BYTES = STAGES * (A_BYTES + B_BYTES) + 1024 /*align*/ + 256 /*barriers*/;
constexpr int THREADS = 192;
constexpr int TMEM_COLS = 512;  // 256 accumulator columns + 8 scale-factor columns, rounded up to a power of two
constexpr int SF_COL = BN;      // 8 columns of UE8M0 1.0 (0x7f): block scales of both operands
constexpr int BAND = 8;         // super-block rows per rasterisation band
}  // namespace

// Symmetric mode: is super-block (sb_i, sb_j) computed on the side that owns rows sb_i?  Exactly
// one of (i, j) and (j, i) says yes.  Blocks are first grouped 2^coarse_shift x 2^coarse_shift:
// whole groups alternate (so that the tiles resident at one time are dense and share their
// operand slabs through L2 -- one GPU uses groups of 8, i.e. one rasterisation band), and inside
// a group on the diagonal the single super-blocks alternate.  Across GPUs the groups are single
// super-blocks, which balances the ranks' shares best.
// Between two RANKS the blocks go by distance on the ring of ranks: rank r computes every block against
// the ranks r+1 .. r+ceil(G/2)-1 (and none against the ranks that far behind it); with an even number of
// ranks the opposite rank's blocks are split by the checkerboard.  Every rank then needs the sample
// operand Wd only for its own samples and those of the floor(G/2) ranks after it (onehot.cu encodes no
// more), and the work stays balanced.
__host__ __device__ inline bool dist_row_side(int sb_i, int sb_j, int coarse_shift, int rank_i = 0, int rank_j = 0,
                                              int world = 1) {
    if (rank_i != rank_j) {
        const int d = (rank_j - rank_i + world) % world;
        if (2 * d < world) return true;
        if (2 * d > world) return false;
        return (((sb_i + sb_j) & 1) == 0) == (rank_j > rank_i);
    }
    if (sb_i == sb_j) return true;
    const int ci = sb_i >> coarse_shift, cj = sb_j >> coarse_shift;
    if (ci != cj) return (((ci + cj) & 1) == 0) == (cj > ci);
    return (((sb_i + sb_j) & 1) == 0) == (sb_j > sb_i);
}

// Epilogue of one 128 x 256 accumulator tile (this warp's 32 TMEM lanes = 32 target rows): distances
// s_i + s_j - acc, stored (or subtracted, incremental update) into the slab row and, for a mirrored
// tile, transposed into the slab of the rank that owns the samples as target rows.
__device__ __forceinline__ void dist_store_tile(uint32_t tmem_base, int q, int64_t row, int32_t s_i, int64_t R, int64_t n0,
                                                int64_t cend, const int32_t *__restrict__ srow, int64_t ldd, int subtract,
                                                bool mirror, int32_t *Dd, int32_t *Dm, int64_t owner_start,
                                                int64_t row_global0) {
#pragma unroll 1
        for (int c0 = 0; c0 < BN; c0 += 32) {
            const int64_t col = n0 + c0;
            if (col >= cend) continue;                         // warp-uniform
            uint32_t v[32];
            tc::tmem_ld_32x32(tmem_base + ((uint32_t)(q * 32) << 16) + (uint32_t)c0, v);
            tc::tmem_ld_wait();
            // distances of this thread's row to samples col .. col+31 (srow is padded to ldd;
            // col is a multiple of 4)
#pragma unroll
            for (int e = 0; e < 32; e += 4) {
                const int4 sj = *reinterpret_cast<const int4 *>(srow + col + e);
                v[e] = (uint32_t)(s_i + sj.x - __float2int_rn(__uint_as_float(v[e])));
                v[e + 1] = (uint32_t)(s_i + sj.y - __float2int_rn(__uint_as_float(v[e + 1])));
                v[e + 2] = (uint32_t)(s_i + sj.z - __float2int_rn(__uint_as_float(v[e + 2])));
                v[e + 3] = (uint32_t)(s_i + sj.w - __float2int_rn(__uint_as_float(v[e + 3])));
            }
            // subtract mode (incremental update): the operands are those of removed columns and
            // their mismatch count is taken off the resident slab.  All loads of a chunk are issued
            // before the first store (the slab pointers may alias, so the compiler would otherwise
            // order every load behind the previous store: 32 dependent round trips per chunk).
            if (row < R) {
                int32_t *dst = Dd + row * ldd + col;           // ldd multiple of 128, col multiple of 4: 16-byte aligned
                if (subtract) {
                    int4 old[8];
#pragma unroll
                    for (int e = 0; e < 32; e += 4)
                        old[e >> 2] = col + e < cend ? *reinterpret_cast<const int4 *>(dst + e) : make_int4(0, 0, 0, 0);
#pragma unroll
                    for (int e = 0; e < 32; e += 4)
                        if (col + e < cend)                    // cend is a multiple of 4 or the padded end
                            *reinterpret_cast<int4 *>(dst + e) =
                                make_int4(old[e >> 2].x - (int)v[e], old[e >> 2].y - (int)v[e + 1],
                                          old[e >> 2].z - (int)v[e + 2], old[e >> 2].w - (int)v[e + 3]);
                } else {
#pragma unroll
                    for (int e = 0; e < 32; e += 4)
                        if (col + e < cend)
                            *reinterpret_cast<int4 *>(dst + e) = make_int4((int)v[e], (int)v[e + 1], (int)v[e + 2], (int)v[e + 3]);
                }
            }
            if (mirror && row < R) {
                // transposed copy: row (col + e) of the owner's slab, column = this row's sample
                int32_t *m = Dm + (col - owner_start) * ldd + row_global0 + row;
                if (subtract) {
                    int32_t old[32];
#pragma unroll
                    for (int e = 0; e < 32; ++e) old[e] = col + e < cend ? m[e * ldd] : 0;
#pragma unroll
                    for (int e = 0; e < 32; ++e)
                        if (col + e < cend) m[e * ldd] = old[e] - (int32_t)v[e];
                } else {
#pragma unroll
                    for (int e = 0; e < 32; ++e)
                        if (col + e < cend) m[e * ldd] = (int32_t)v[e];
                }
            }
        }
}

// One cluster of two CTAs per super-block (see the header); a pair is exactly one super-block of the
// symmetric scheme.
__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(THREADS, 1)
tc_dist_pair_kernel(const __grid_constant__ CUtensorMap tmap_a, const __grid_constant__ CUtensorMap tmap_b,
                    int num_k_blocks, const int32_t *__restrict__ srow, const int64_t *__restrict__ ids, int64_t R,
                    int64_t n, int64_t ldd, int symmetric, int subtract, int pair_rows, int tiles_x,
                    const __grid_constant__ DistPeers peers) {
    const uint32_t crank = tc::cluster_ctarank();
    // L2-friendly rasterisation: bands of BAND super-block rows, walked column by column, so that the
    // ~74 concurrently resident pairs form a roughly square region and share their operand K-slabs
    // through L2 (8 x 256 target rows and ~9 x 256 sample rows per wave) instead of streaming a
    // different 256-row slab of the sample operand per pair.
    int pair_y, tile_x;
    {
        const int lin = (int)(blockIdx.x >> 1);
        const int band = lin / (BAND * tiles_x);
        const int band_rows = pair_rows - band * BAND < BAND ? pair_rows - band * BAND : BAND;
        const int in_band = lin - band * BAND * tiles_x;
        pair_y = band * BAND + in_band % band_rows;
        tile_x = in_band / band_rows;
    }
    int owner = 0;
    while (owner + 1 < peers.world && tile_x >= peers.sb_base[owner + 1]) ++owner;
    const int64_t n0 = peers.starts[owner] + (int64_t)(tile_x - peers.sb_base[owner]) * BN;
    const int64_t cend = n0 + BN < peers.starts[owner + 1] ? n0 + BN : peers.starts[owner + 1];
    const int sb_i = peers.sb_base[peers.rank] + pair_y, sb_j = tile_x;
    const bool diagonal = sb_i == sb_j;
    if (symmetric && !dist_row_side(sb_i, sb_j, peers.coarse_shift, peers.rank, owner, peers.world)) return;      // both CTAs of the pair take the same exit
    const bool mirror = symmetric && !diagonal;
    int32_t *Dd = peers.slab[peers.rank];
    int32_t *Dm = peers.slab[owner];
    const int64_t row_global0 = peers.starts[peers.rank];
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    unsigned char *smem = reinterpret_cast<unsigned char *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    unsigned char *smem_a = smem;
    unsigned char *smem_b = smem + STAGES * A_BYTES;
    uint64_t *full_bar = reinterpret_cast<uint64_t *>(smem + STAGES * (A_BYTES + B_BYTES));
    uint64_t *empty_bar = full_bar + STAGES;
    uint64_t *accum_bar = empty_bar + STAGES;
    uint32_t *tmem_slot = reinterpret_cast<uint32_t *>(accum_bar + 1);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int m0 = pair_y * (2 * BM) + (int)crank * BM;           // this CTA's 128 target rows

    if (warp == 0 && lane == 0) {
        tc::prefetch_tmap(&tmap_a);
        tc::prefetch_tmap(&tmap_b);
        for (int s = 0; s < STAGES; ++s) {
            tc::mbar_init(&full_bar[s], 1);       // the leader's producer arrives with the pair's byte count
            tc::mbar_init(&empty_bar[s], 1);      // the pair's MMA commit arrives (multicast)
        }
        tc::mbar_init(accum_bar, 1);
        tc::fence_barrier_init();
    }
    if (warp == 1) tc::tmem_alloc_pair<TMEM_COLS>(tmem_slot);
    tc::tc_fence_before();
    __syncthreads();
    tc::cluster_sync_all();                           // the peer's barriers exist before anything signals them
    tc::tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    if (warp >= 2) {
        for (int c = 0; c < 8; ++c) tc::tmem_st_32x1(tmem_base + ((uint32_t)((warp & 3) * 32) << 16) + SF_COL + c, 0x7f7f7f7fu);
        tc::tmem_st_wait();
    }
    tc::tc_fence_before();
    __syncthreads();
    tc::cluster_sync_all();                           // both CTAs' scale factors are in place before the leader issues
    tc::tc_fence_after();

    if (warp == 0) {
        // ===== TMA producer (one per CTA: own A rows, own half of the B rows) =====
        if (tc::elect_one()) {   // one thread, and the compiler knows it: uniform-register issue code
            for (int kb = 0; kb < num_k_blocks; ++kb) {
                const int s = kb % STAGES;
                const uint32_t ph = (kb / STAGES) & 1;
                tc::mbar_wait(&empty_bar[s], ph ^ 1);
                if (crank == 0) tc::mbar_arrive_expect_tx(&full_bar[s], 2 * (A_BYTES + B_BYTES));
                tc::tma_load_2d_pair(smem_a + s * A_BYTES, &tmap_a, &full_bar[s], kb * BK, m0);
                tc::tma_load_2d_pair(smem_b + s * B_BYTES, &tmap_b, &full_bar[s], kb * BK, (int32_t)(n0 + crank * (BN / 2)));
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: one thread of the leader CTA, for the pair =====
        if (crank == 0 && tc::elect_one()) {
            constexpr uint32_t idesc = tc::make_idesc_mxf4(2 * BM, BN);
            for (int kb = 0; kb < num_k_blocks; ++kb) {
                const int s = kb % STAGES;
                const uint32_t ph = (kb / STAGES) & 1;
                tc::mbar_wait(&full_bar[s], ph);
                tc::tc_fence_after();
                const uint64_t da = tc::make_smem_desc_sw128(tc::smem_u32(smem_a + s * A_BYTES));
                const uint64_t db = tc::make_smem_desc_sw128(tc::smem_u32(smem_b + s * B_BYTES));
#pragma unroll
                for (int k = 0; k < BK / 32; ++k)
                    tc::mma_mxf4_pair(tmem_base, da + (uint64_t)(2 * k), db + (uint64_t)(2 * k), idesc, tmem_base + SF_COL,
                                  tmem_base + SF_COL, (kb | k) != 0);
                tc::tc_commit_pair(&empty_bar[s]);
            }
            tc::tc_commit_pair(accum_bar);
        }
    } else {
        // ===== epilogue: this CTA's 128 TMEM lanes =====
        const int q = warp & 3;
        const int64_t row = (int64_t)m0 + q * 32 + lane;
        const int32_t s_i = row < R ? srow[ids[row]] : 0;
        tc::mbar_wait(accum_bar, 0);
        tc::tc_fence_after();
        dist_store_tile(tmem_base, q, row, s_i, R, n0, cend, srow, ldd, subtract, mirror, Dd, Dm, peers.starts[owner], row_global0);
        tc::tc_fence_before();
    }
    __syncthreads();
    tc::cluster_sync_all();                           // neither CTA leaves (or frees TMEM) while the pair is in flight
    if (warp == 1) {
        tc::tc_fence_after();
        tc::tmem_dealloc_pair<TMEM_COLS>(tmem_base);
    }
}

void launch_tc_dist(const int8_t *a, const int8_t *b, int64_t row_bytes, int64_t pitch, int64_t K, const int32_t *srow,
                    const int64_t *d_ids, int64_t R, int64_t n, int64_t ldd, bool symmetric, bool subtract,
                    const DistPeers &peers, cudaStream_t st, int *launches, double *ops) {
    const CUtensorMap tmap_a = make_tmap_u8_sw128(a, row_bytes, R, pitch, BM);
    const CUtensorMap tmap_b = make_tmap_u8_sw128(b, row_bytes, n, pitch, BN / 2);   // each CTA of a pair stages half of the sample rows
    const int tiles_x = peers.sb_base[peers.world], pair_rows = (int)ceil_div(R, 2 * BM);
    // per launch: the attribute belongs to the CURRENT device (several devices per process: fs_multi_*)
    FS_CUDA(cudaFuncSetAttribute(tc_dist_pair_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, SMEM_BYTES));
    tc_dist_pair_kernel<<<(unsigned)(2 * tiles_x * pair_rows), THREADS, SMEM_BYTES, st>>>(
        tmap_a, tmap_b, (int)(K / BK), srow, d_ids, R, n, ldd, symmetric ? 1 : 0, subtract ? 1 : 0, pair_rows, tiles_x, peers);
    FS_CUDA(cudaGetLastError());
    ++*launches;
    if (ops) {
        int64_t tiles = 0;
        for (int py = 0; py < pair_rows; ++py)
            for (int bx = 0; bx < tiles_x; ++bx) {
                int owner = 0;
                while (owner + 1 < peers.world && bx >= peers.sb_base[owner + 1]) ++owner;
                const int sb_i = peers.sb_base[peers.rank] + py;
                // a pair always runs both of its 128-row tiles
                tiles += (!symmetric || dist_row_side(sb_i, bx, peers.coarse_shift, peers.rank, owner, peers.world)) ? 2 : 0;
            }
        *ops += 2.0 * BM * BN * (2.0 * (double)K) * (double)tiles;      // K is the operand row length in bytes
    }
}

void launch_dist_tensor(fs_dataset *ds, const WorkSet &ws, int64_t r0_internal, const int64_t *h_row_ids,
                        const int64_t *d_row_ids, bool contiguous, int64_t R, int32_t *Dd, int64_t ldn,
                        cudaStream_t st, int *launches, double *ops) {
    // incremental update: the operands are those of the removed columns and the result is subtracted
    const bool incr = ws.dist_mode == kDistIncremental;
    const int8_t *Uop = incr ? ws.Ur.ptr : ws.U.ptr, *Wop = incr ? ws.Wdr.ptr : ws.Wd.ptr;
    const int32_t *sop = incr ? ws.srow_r.ptr : ws.srow.ptr;
    const int64_t K = (incr ? ws.Kr : ws.K) / 2;        // operand row bytes (FP4 nibbles)
    // every column adds at most 2 to an FP32 accumulator: exact while the sums stay below 2^24
    FS_REQUIRE(2 * ws.pt < (1LL << 24), FS_ERR_INVALID, "too many one-hot columns for exact FP32 accumulation (%lld)", (long long)ws.pt);
    const int8_t *a_rows;
    const int64_t u_lo = incr ? 0 : ws.u_lo;           // first sample row held by the target-side operand
    if (contiguous) {
        a_rows = Uop + (size_t)(r0_internal - u_lo) * K;
    } else {
        DevBuf<int8_t> &g = ds->a_gather;
        g.reserve((size_t)R * K);
        for (int64_t r = 0; r < R; ++r)
            FS_CUDA(cudaMemcpyAsync(g.ptr + (size_t)r * K, Uop + (size_t)(h_row_ids[r] - u_lo) * K, K,
                                    cudaMemcpyDeviceToDevice, st));
        a_rows = g.ptr;
    }
    // Symmetric mode: the target rows of all ranks together cover every sample, so half of the
    // off-diagonal super-blocks are computed and mirrored (see the file head).  One rank scoring all rows
    // is the trivial case; with peers configured (fs_dataset_set_peers) this rank's rows must be
    // exactly its shard and Dd its exported slab.  An incremental update across ranks stays
    // non-symmetric (it would need remote read-modify-writes).
    const bool own_shard = contiguous && ds->peers_on && Dd == ds->peer_slab && r0_internal == ds->peers.starts[ds->peers.rank] &&
                           R == ds->peers.starts[ds->peers.rank + 1] - ds->peers.starts[ds->peers.rank] && !incr;
    const DistPeers peers = own_shard ? ds->peers : single_rank_peers(Dd, ds->n);
    const bool symmetric = own_shard || (contiguous && r0_internal == 0 && R == ds->n);
    launch_tc_dist(a_rows, Wop, K, K, K, sop, d_row_ids, R, ds->n, ldn, symmetric, incr, peers, st, launches, ops);
    ds->last_dist_exchanged = symmetric && peers.world > 1;
}

}  // namespace fs
