// onehot.cu -- encoding of the active discrete columns into the operands of the one-hot
// tensor-core path (tc_dist.cu, tc_accum.cu) and of ReliefF's one-hot gather (accum_general.cu).
//
// K0 "encode" of the design: every active discrete column f with 2 <= V_f <= FS_DISTINCT_CAP
// distinct values becomes V_f - 1 reduced one-hot rows/columns (only equality matters,
// MultiSURF.py:184-185, so any injective value coding is exact), stored as e2m1 (FP4) nibbles --
// two entries per byte -- for the tcgen05 kind::mxf4 GEMMs:
//   U, Wd [n, K/2 bytes]   sample-major (one-hot index contiguous)  -> the two operands of the distance GEMM
//   At    [K, ldt/2 bytes] feature-major (sample index contiguous)   -> M operand of the accumulation GEMM
//   codesT [pt, ldt] feature-major value codes               -> accumulation epilogue
//   codes  [n, ldc]  sample-major value codes                -> ReliefF's sparse neighbour gather (only then)
// Samples are in the data set's class-sorted internal order.  HBM-bound streaming kernel:
// reads n*pt elements once, writes 1.5*n*K + n*pt bytes.
#include <algorithm>
#include <type_traits>

#include "common.cuh"

namespace fs {

// ---------------------------------------------------------------------------
// encode
// ---------------------------------------------------------------------------
// Reduced one-hot operands.  A column with V distinct values (codes 0..V-1) owns V - 1
// rows, one per code v < V - 1; the last code is implied because every sample carries
// exactly one code:
//   matches_f(i, j) = sum_v [c_i = v][c_j = v]
//                   = 1 - [c_i != last] - [c_j != last] + sum_{v < last} [c_i = v] ([c_j = v] + [c_j != last]),
// so with U[i,(f,v)] = [c_i = v], Wd[j,(f,v)] = [c_j = v] + [c_j != last] and
// s_i = #{f : c_if != last_f}:   d_ij = sum_f (1 - matches_f) = s_i + s_j - (U Wd^T)_ij   -- exact integers,
// with a contraction length of sum_f (V_f - 1) instead of sum_f V_f (2/3 of the MMA work for
// 0/1/2 genotypes).  The accumulation GEMM contracts the same reduced rows (At) and its
// epilogue recovers the implied plane from G_last = rowsum - sum_{v<last} G_v (tc_accum.cu).
//
// Tile: 128 samples x 64 columns per CTA.  Step 1 reads x and keeps the value codes in
// shared memory in both orientations; step 2 emits the U / Wd rows (one-hot index
// contiguous) and the per-sample counts s; step 3 the At and codesT rows (sample index
// contiguous).  One kernel template, onehot_encode_kernel<Tin, kLean>, does all three steps: its
// lean instantiation (one-byte 0/1/2 genotypes) writes every byte of the tile's footprint exactly
// once, so the host clears only the K padding of U / Wd; the general instantiations (any input
// type, up to FS_DISTINCT_CAP values) OR the words at unaligned tile edges into operands the host
// cleared whole (clear_dist_ops).  Where every column of a tile holds three values, both take the
// same 0/1/2 paths, whose global stores are 8- or 16-byte vectors.
constexpr int ENC_ROWS = 128;
constexpr int ENC_COLS = 64;
constexpr int ENC_CR_LD = ENC_ROWS + 4;                       // conflict-free transposed stores
constexpr int ENC_KMAX = ENC_COLS * (FS_DISTINCT_CAP - 1);

// FP4 (e2m1 nibble) images of 4 genotype codes: one byte per column -- low nibble = row v = 0,
// high nibble = row v = 1.  U: [c = v] -> 1.0 = 0x2.  Wd: [c = v] + [c != last] in {0, 1, 2} ->
// 0x0 / 0x2 / 0x4, i.e. the bytes 0x24 (code 0), 0x42 (code 1), 0x00 (code 2).
__device__ __forceinline__ void expand_v3_fp4(uint32_t cw, uint32_t &u, uint32_t &w, int &cnt) {
    const uint32_t e1 = cw & 0x01010101u, e2 = (cw >> 1) & 0x01010101u;
    const uint32_t ne = e2 ^ 0x01010101u;             // [code != last]
    const uint32_t e0 = ne ^ e1;                      // [code == 0]
    cnt += __popc(ne);
    u = (e0 << 1) | (e1 << 5);
    w = (e0 << 2) | (e0 << 5) | (e1 << 1) | (e1 << 6);
}

// At is stored as e2m1 (FP4) nibbles, two samples per byte (low nibble = even sample), for the
// tcgen05 kind::mxf4 accumulation GEMM: 1.0 is the nibble 0x2.  pack_fp4_flags turns four 0/1
// flag bytes (samples s..s+3) into two bytes of nibbles.
__device__ __forceinline__ uint32_t pack_fp4_flags(uint32_t e) {
    const uint32_t t = (e << 1) | (e >> 3);          // byte 0: b0<<1 | b1<<5,  byte 2: b2<<1 | b3<<5
    return __byte_perm(t, 0u, 0x4420);               // (t.b0, t.b2, 0, 0)
}
__device__ __forceinline__ uint2 pack_fp4_flags16(uint32_t e0, uint32_t e1, uint32_t e2, uint32_t e3) {
    return make_uint2(pack_fp4_flags(e0) | (pack_fp4_flags(e1) << 16), pack_fp4_flags(e2) | (pack_fp4_flags(e3) << 16));
}

// Sample rows (internal order) whose Wd rows somebody reads: everything on one GPU; inside a multi-GPU
// group the rank's own samples and those of the floor(G/2) ranks after it on the ring (tc_dist.cu), i.e.
// at most two ranges.
struct WdRows {
    int64_t lo0, hi0, lo1, hi1;
    __host__ __device__ bool has(int64_t r) const { return (r >= lo0 && r < hi0) || (r >= lo1 && r < hi1); }
    __host__ __device__ bool touches(int64_t a, int64_t b) const { return (a < hi0 && b > lo0) || (a < hi1 && b > lo1); }
};

// kLean: the instantiation for the case that matters most, one-byte input whose columns all hold exactly the
// values 0/1/2 (the value is its own code, two reduced rows per column).  It has no code tables and no per-column
// bookkeeping, so registers stay low enough for 6 CTAs per SM, which is what hides the perm -> x load chain of
// this streaming kernel.  It alone stages short column spans in shared memory (step 1) and writes a ragged column
// tile byte by byte (step 2); only the general instantiations translate values to codes and OR partial words in.
// (A minimum of 0 CTAs per SM sets none: the general instantiations' register allocation changes under a minimum of 1.)
template <typename Tin, bool kLean>
__global__ void __launch_bounds__(256, kLean ? 6 : 0) onehot_encode_kernel(
    const Tin *__restrict__ x, int64_t ldx, const int64_t *__restrict__ perm, const int64_t *__restrict__ tcol,
    const int32_t *__restrict__ toff, const double *__restrict__ vals, int as_f32, int64_t n, int64_t pt, int64_t K,
    int64_t ldt, int64_t ldc, int8_t *__restrict__ U, int8_t *__restrict__ Wd, int8_t *__restrict__ At,
    uint8_t *__restrict__ codesT, uint8_t *__restrict__ codes, int32_t *__restrict__ srow,
    uint32_t *__restrict__ krow, int all_ident, int64_t u_lo, int64_t u_hi, const int32_t *__restrict__ tpos, int uk0,
    WdRows wr) {
    // uk0: one-hot row of U / Wd that this launch's row 0 of `toff` stands for (a launch over a slice of the
    // columns numbers At / krow rows from 0 but addresses the distance operands globally)
    __shared__ __align__(16) uint8_t code_rc[ENC_ROWS][ENC_COLS];       // [sample][column]
    __shared__ __align__(16) uint8_t code_cr[ENC_COLS][ENC_CR_LD];      // [column][sample]
    __shared__ uint8_t kcol[ENC_KMAX];                                  // general: reduced row -> column in tile
    __shared__ uint8_t kval[ENC_KMAX];                                  // general: reduced row -> value code
    __shared__ uint8_t clast[ENC_COLS];                                 // general: last code of each column
    __shared__ int64_t sperm[ENC_ROWS];
    const int tid = threadIdx.x, lane = tid & 31;
    // row tiles vary fastest: the CTAs resident at one time cover every sample of a band of
    // columns, so the feature-major rows (At, codesT) are written as whole contiguous rows
    const int tiles_y = (int)((n + ENC_ROWS - 1) / ENC_ROWS);
    const int tile_x = (int)(blockIdx.x / tiles_y), tile_y = (int)(blockIdx.x % tiles_y);
    const int64_t c0 = (int64_t)tile_x * ENC_COLS, r0 = (int64_t)tile_y * ENC_ROWS;
    const int ncols = (int)(pt - c0 < ENC_COLS ? pt - c0 : ENC_COLS);
    const int nrows = (int)(n - r0 < ENC_ROWS ? n - r0 : ENC_ROWS);
    const int k0 = toff[c0], k1 = toff[c0 + ncols];
    // a distance-only launch has nothing to do for a row tile whose samples' Wd rows nobody reads
    if (At == nullptr && codes == nullptr && !wr.touches(r0, r0 + nrows)) return;
    if (tid < ENC_ROWS) sperm[tid] = tid < nrows ? perm[r0 + tid] : 0;

    // ---- step 1: value codes
    {
        const int c = tid & (ENC_COLS - 1);
        int64_t f = 0;
        int V = 0;
        bool ident = true;          // the code of a value is the value itself (sorted 0..V-1)
        // code table of this thread's column in the input's own type (values came from the
        // data, so the conversion back is exact); float64 input scored in float32 arithmetic
        // is compared after narrowing, as the reference compares x.astype(float32)
        Tin v[FS_DISTINCT_CAP];
        float vf[FS_DISTINCT_CAP];
        if (c < ncols) {
            f = tcol[c0 + c];
            const int off = kLean ? k0 + 2 * c : toff[c0 + c];
            V = kLean ? 3 : toff[c0 + c + 1] - off + 1;
            if constexpr (!kLean) {
                if (!all_ident) {
#pragma unroll
                    for (int q = 0; q < FS_DISTINCT_CAP; ++q) {
                        const double d = q < V ? vals[f * FS_DISTINCT_CAP + q] : 0.0;
                        v[q] = (Tin)d;
                        vf[q] = (float)d;
                        ident = ident && (q >= V || d == (double)q);
                    }
                }
            }
            if (tid < ENC_COLS) {
                if constexpr (!kLean) {
                    clast[c] = (uint8_t)(V - 1);
                    for (int q = 0; q < V - 1; ++q) {
                        kcol[off - k0 + q] = (uint8_t)c;
                        kval[off - k0 + q] = (uint8_t)q;
                    }
                }
                for (int q = 0; tile_y == 0 && krow && q < V - 1; ++q)
                    krow[off + q] = (uint32_t)(tpos ? tpos[c0 + c] : (int32_t)(c0 + c)) | ((uint32_t)q << 24) | ((uint32_t)(V - 1) << 28);
            }
        }
        // whole-tile fast path: one-byte input, identity codes, and the tile's 64 columns are 64
        // consecutive, 16-byte aligned bytes of every row of x -> 16-byte loads, no table look-ups
        const int64_t f0 = tcol[c0];
        const bool fast1 = __syncthreads_and(sizeof(Tin) == 1 && ncols == ENC_COLS && ident && f == f0 + c &&
                                             (ldx & 15) == 0 && ((reinterpret_cast<uintptr_t>(x) + f0) & 15) == 0);
        // lean second choice: the tile's columns lie within kSpan bytes of x (16-byte aligned base)
        constexpr int kSpan = 256, kSpanRows = 32;
        const int64_t fbase = f0 & ~(int64_t)15;
        const int64_t flast = tcol[c0 + ncols - 1];
        const bool span_ok = kLean && __syncthreads_and(!fast1 && (ldx & 15) == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 &&
                                                        flast - fbase < kSpan && (c >= ncols || (f >= fbase && f <= flast)));
        if (fast1) {
            // two 16-byte loads per thread, both in flight before either is used
            uint4 q[2];
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int rr = (tid + 256 * i) >> 2, ch = tid & 3;
                q[i] = rr < nrows ? *reinterpret_cast<const uint4 *>(reinterpret_cast<const uint8_t *>(x) + sperm[rr] * ldx + f0 + 16 * ch)
                                  : make_uint4(0u, 0u, 0u, 0u);
            }
#pragma unroll
            for (int i = 0; i < 2; ++i) {
                const int rr = (tid + 256 * i) >> 2, ch = tid & 3;
                if (codes && rr < nrows) *reinterpret_cast<uint4 *>(codes + (r0 + rr) * ldc + c0 + 16 * ch) = q[i];   // ldc, c0: multiples of 16
                *reinterpret_cast<uint4 *>(&code_rc[rr][16 * ch]) = q[i];
                const uint32_t qw[4] = {q[i].x, q[i].y, q[i].z, q[i].w};
#pragma unroll
                for (int b = 0; b < 16; ++b) code_cr[16 * ch + b][rr] = (uint8_t)(qw[b >> 2] >> (8 * (b & 3)));
            }
        } else if (!span_ok) {
            // gathered columns (TuRF iterations): one column per thread, 32 samples per thread (rows
            // tid/64 + 4i); the loads of a batch of 8 are issued before any of them is used, so 8
            // requests per thread are in flight
            constexpr int kBatch = 8;
            for (int i0 = 0; i0 < ENC_ROWS / 4; i0 += kBatch) {
                Tin xv[kBatch];
#pragma unroll
                for (int u = 0; u < kBatch; ++u) {
                    const int rr = (tid >> 6) + 4 * (i0 + u);
                    xv[u] = (c < ncols && rr < nrows) ? x[sperm[rr] * ldx + f] : (Tin)0;
                }
#pragma unroll
                for (int u = 0; u < kBatch; ++u) {
                    const int rr = (tid >> 6) + 4 * (i0 + u);
                    uint8_t code = 0;
                    if (c < ncols && rr < nrows) {
                        int found = 0;
                        if (ident) {
                            found = (int)xv[u];
                        } else if constexpr (!kLean) {
                            if (V <= 4) {                   // genotype-like columns: 3 compares, no loop
#pragma unroll
                                for (int q = 3; q >= 1; --q) {
                                    const bool eq = as_f32 ? ((float)xv[u] == vf[q]) : (xv[u] == v[q]);
                                    if (q < V && eq) found = q;
                                }
                                if (as_f32 ? ((float)xv[u] == vf[0]) : (xv[u] == v[0])) found = 0;   // lowest match wins
                            } else {
#pragma unroll
                                for (int q = FS_DISTINCT_CAP - 1; q >= 0; --q) {
                                    const bool eq = as_f32 ? ((float)xv[u] == vf[q]) : (xv[u] == v[q]);
                                    if (q < V && eq) found = q;
                                }
                            }
                        }
                        code = (uint8_t)found;
                        if (codes) codes[(r0 + rr) * ldc + c0 + c] = code;
                    }
                    code_rc[rr][c] = code;
                    code_cr[c][rr] = code;
                }
            }
        } else if constexpr (kLean) {
            // gathered columns whose span in x is short (TuRF's early iterations: ascending columns with
            // a few gaps): the span [fbase, fbase + kSpan) of 32 rows at a time is staged in shared memory
            // with coalesced 16-byte loads, and every thread picks its column's bytes from there
            __shared__ __align__(16) uint8_t raw[kSpanRows][kSpan];
            const int span_chunks = (int)((flast - fbase) >> 4) + 1;          // 16-byte chunks that hold a wanted column
            for (int rb = 0; rb < ENC_ROWS; rb += kSpanRows) {
                // fixed 16-chunk indexing (no division by the run-time chunk count); chunks past the span idle
                for (int item = tid; item < kSpanRows * (kSpan / 16); item += 256) {
                    const int rr = rb + (item >> 4), ch = item & 15;
                    if (ch >= span_chunks) continue;
                    uint4 q = make_uint4(0u, 0u, 0u, 0u);
                    if (rr < nrows && fbase + 16 * ch < ldx) q = *reinterpret_cast<const uint4 *>(x + sperm[rr] * ldx + fbase + 16 * ch);
                    *reinterpret_cast<uint4 *>(&raw[rr - rb][16 * ch]) = q;
                }
                __syncthreads();
#pragma unroll
                for (int u = 0; u < kSpanRows / 4; ++u) {
                    const int rl = (tid >> 6) + 4 * u, rr = rb + rl;
                    const uint8_t xv = (c < ncols && rr < nrows) ? raw[rl][(int)(f - fbase)] : (uint8_t)0;
                    if (codes && c < ncols && rr < nrows) codes[(r0 + rr) * ldc + c0 + c] = xv;
                    code_rc[rr][c] = xv;
                    code_cr[c][rr] = xv;
                }
                __syncthreads();
            }
        }
    }
    __syncthreads();

    // ---- step 2: U[r, k0..k1), Wd[r, k0..k1), s[r]
    const int kg0 = k0 + uk0, kg1 = k1 + uk0;          // the same rows in U / Wd
    // every column of the tile has 3 values (0/1/2 genotypes): two reduced rows per column, codes are the rows' bits
    bool all3 = true;
    if constexpr (!kLean) all3 = __syncthreads_and((tid >= ncols) || clast[tid < ncols ? tid : 0] == 2);
    if (U == nullptr) {
        // distance operands not wanted (the slab is updated incrementally from other columns)
    } else if (all3 && (kg0 & 31) == 0 && (ncols & 15) == 0) {
        // 16 columns per item: 16 code bytes -> 16 bytes of U and of Wd (one byte per column)
        const int ngroups = ncols >> 4;
#pragma unroll
        for (int it = 0; it < ENC_ROWS * 4 / 256; ++it) {                 // uniform trip count (shuffles below)
            const int item = tid + 256 * it, rr = item >> 2, g = item & 3;
            int cnt = 0;
            if (rr < nrows && g < ngroups) {
                const uint4 cw = *reinterpret_cast<const uint4 *>(&code_rc[rr][16 * g]);
                uint4 u, w;
                expand_v3_fp4(cw.x, u.x, w.x, cnt);
                expand_v3_fp4(cw.y, u.y, w.y, cnt);
                expand_v3_fp4(cw.z, u.z, w.z, cnt);
                expand_v3_fp4(cw.w, u.w, w.w, cnt);
                const int64_t o = (r0 + rr) * K + (kg0 >> 1) + 16 * g;     // K = row pitch in bytes
                // U holds only the rows [u_lo, u_hi) (the target rows of this rank)
                if (r0 + rr >= u_lo && r0 + rr < u_hi) *reinterpret_cast<uint4 *>(U + o - u_lo * K) = u;
                if (wr.has(r0 + rr)) *reinterpret_cast<uint4 *>(Wd + o) = w;
            }
            cnt += __shfl_xor_sync(0xffffffffu, cnt, 1);
            cnt += __shfl_xor_sync(0xffffffffu, cnt, 2);
            if (g == 0 && rr < nrows && cnt) atomicAdd(&srow[r0 + rr], cnt);
        }
    } else if constexpr (kLean) {
        // ragged last column tile: one (sample, column) byte per step
        for (int rr = tid >> 5; rr < ENC_ROWS; rr += 8) {
            int cnt = 0;
            if (rr < nrows)
                for (int cc = lane; cc < ncols; cc += 32) {
                    const uint32_t code = code_rc[rr][cc];
                    const int64_t o = (r0 + rr) * K + (kg0 >> 1) + cc;
                    if (r0 + rr >= u_lo && r0 + rr < u_hi)
                        U[o - u_lo * K] = (int8_t)(code == 0u ? 0x02u : code == 1u ? 0x20u : 0u);
                    if (wr.has(r0 + rr)) Wd[o] = (int8_t)(code == 0u ? 0x24u : code == 1u ? 0x42u : 0u);
                    cnt += code != 2u ? 1 : 0;
                }
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
            if (lane == 0 && rr < nrows && cnt) atomicAdd(&srow[r0 + rr], cnt);
        }
    } else {
        // general path: nibbles k0..k1 of the row; 32-bit words (8 nibbles) that belong to this tile
        // entirely are stored, the words at the unaligned edges are OR-ed in (the operands were
        // cleared by the host; a neighbouring tile owns the other nibbles of such a word)
        const int w0 = kg0 >> 3, w1 = (kg1 + 7) >> 3;             // word range covering [kg0, kg1)
        for (int rr = tid >> 5; rr < ENC_ROWS; rr += 8) {          // uniform trip count
            int cnt = 0;
            if (rr < nrows) {
                for (int w = w0 + lane; w < w1; w += 32) {
                    uint32_t uw = 0, ww = 0;
                    bool full = true;
#pragma unroll
                    for (int b = 0; b < 8; ++b) {
                        const int k = 8 * w + b;
                        if (k >= kg0 && k < kg1) {
                            const int col = kcol[k - kg0];
                            const uint32_t code = code_rc[rr][col];
                            const uint32_t on = code == kval[k - kg0] ? 1u : 0u;
                            uw |= (on << 1) << (4 * b);                                        // 1.0 = 0x2
                            ww |= ((on + (code != clast[col] ? 1u : 0u)) << 1) << (4 * b);      // 0 / 1.0 / 2.0 = 0x0 / 0x2 / 0x4
                        } else {
                            full = false;
                        }
                    }
                    const int64_t o = (r0 + rr) * K + 4 * (int64_t)w;         // K = row pitch in bytes
                    const bool in_u = r0 + rr >= u_lo && r0 + rr < u_hi;      // U holds only those rows
                    const bool in_w = wr.has(r0 + rr);
                    if (full) {
                        if (in_u) *reinterpret_cast<uint32_t *>(U + o - u_lo * K) = uw;
                        if (in_w) *reinterpret_cast<uint32_t *>(Wd + o) = ww;
                    } else {
                        if (in_u && uw) atomicOr(reinterpret_cast<unsigned int *>(U + o - u_lo * K), uw);
                        if (in_w && ww) atomicOr(reinterpret_cast<unsigned int *>(Wd + o), ww);
                    }
                }
                for (int c = lane; c < ncols; c += 32) cnt += code_rc[rr][c] != clast[c] ? 1 : 0;
            }
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
            if (lane == 0 && rr < nrows && cnt) atomicAdd(&srow[r0 + rr], cnt);
        }
    }
    // ---- step 3: At[k, r0..r0+128) and codesT[c, r0..r0+128): 16 samples per store
    if (At == nullptr) {
        // accumulation operands not wanted (columns that only update the distance slab)
    } else if (all3) {
        // one item = 16 samples of one column -> its two At rows and its codesT row
        for (int item = tid; item < ncols * 8; item += 256) {
            const int c = item >> 3, seg = item & 7;
            const uint32_t *src = reinterpret_cast<const uint32_t *>(&code_cr[c][16 * seg]);
            const uint4 w = make_uint4(src[0], src[1], src[2], src[3]);
            uint4 e0, e1;
            e1.x = w.x & 0x01010101u; e0.x = ((w.x >> 1) & 0x01010101u) ^ 0x01010101u ^ e1.x;
            e1.y = w.y & 0x01010101u; e0.y = ((w.y >> 1) & 0x01010101u) ^ 0x01010101u ^ e1.y;
            e1.z = w.z & 0x01010101u; e0.z = ((w.z >> 1) & 0x01010101u) ^ 0x01010101u ^ e1.z;
            e1.w = w.w & 0x01010101u; e0.w = ((w.w >> 1) & 0x01010101u) ^ 0x01010101u ^ e1.w;
            const int64_t o = r0 + 16 * seg;                                  // r0, ldt multiples of 128: aligned
            const int64_t lda = ldt >> 1;                                     // At: two samples per byte
            int8_t *a0 = At + (int64_t)(k0 + 2 * c) * lda + (o >> 1), *a1 = a0 + lda;
            uint8_t *ct = codesT ? codesT + (c0 + c) * ldt + o : nullptr;
            if (16 * seg + 16 <= nrows) {
                *reinterpret_cast<uint2 *>(a0) = pack_fp4_flags16(e0.x, e0.y, e0.z, e0.w);
                *reinterpret_cast<uint2 *>(a1) = pack_fp4_flags16(e1.x, e1.y, e1.z, e1.w);
                if (ct) *reinterpret_cast<uint4 *>(ct) = w;
            } else {
                // ragged last row tile: whole bytes only where a sample lives, zero nibbles past nrows
                for (int b = 0; b < 16 && 16 * seg + b < nrows; b += 2) {
                    const uint32_t ca = code_cr[c][16 * seg + b];
                    const bool two = 16 * seg + b + 1 < nrows;
                    const uint32_t cb = two ? code_cr[c][16 * seg + b + 1] : 3u;     // 3 matches no value
                    a0[b >> 1] = (int8_t)((ca == 0u ? 0x02u : 0u) | (cb == 0u ? 0x20u : 0u));
                    a1[b >> 1] = (int8_t)((ca == 1u ? 0x02u : 0u) | (cb == 1u ? 0x20u : 0u));
                    if (ct) {
                        ct[b] = (uint8_t)ca;
                        if (two) ct[b + 1] = (uint8_t)cb;
                    }
                }
            }
        }
    } else if constexpr (!kLean) {
        const int nk = k1 - k0;
        for (int item = tid; item < nk * 8; item += 256) {
            const int kk = item >> 3, seg = item & 7;
            const uint32_t *src = reinterpret_cast<const uint32_t *>(&code_cr[kcol[kk]][16 * seg]);
            const uint32_t val = kval[kk] * 0x01010101u;
            uint4 o;
            o.x = __vcmpeq4(src[0], val) & 0x01010101u;
            o.y = __vcmpeq4(src[1], val) & 0x01010101u;
            o.z = __vcmpeq4(src[2], val) & 0x01010101u;
            o.w = __vcmpeq4(src[3], val) & 0x01010101u;
            // two samples per byte (FP4 nibbles); r0, ldt multiples of 128: aligned
            int8_t *dst = At + (int64_t)(k0 + kk) * (ldt >> 1) + ((r0 + 16 * seg) >> 1);
            const uint2 pk = pack_fp4_flags16(o.x, o.y, o.z, o.w);
            if (16 * seg + 16 <= nrows) {
                *reinterpret_cast<uint2 *>(dst) = pk;
            } else {
                // ragged last row tile: flags of samples beyond nrows are zero (their codes are 0 in
                // shared memory but may match value 0: mask them), whole bytes only where a sample lives
                const uint32_t pw[2] = {pk.x, pk.y};
                for (int b = 0; b < 8; ++b) {
                    const int s0 = 16 * seg + 2 * b;
                    if (s0 >= nrows) break;
                    uint32_t byte = (pw[b >> 2] >> (8 * (b & 3))) & 0xffu;
                    if (s0 + 1 >= nrows) byte &= 0x0fu;
                    dst[b] = (int8_t)byte;
                }
            }
        }
        for (int item = tid; codesT != nullptr && item < ncols * 8; item += 256) {
            const int c = item >> 3, seg = item & 7;
            const uint32_t *src = reinterpret_cast<const uint32_t *>(&code_cr[c][16 * seg]);
            const uint4 o = make_uint4(src[0], src[1], src[2], src[3]);
            uint8_t *dst = codesT + (c0 + c) * ldt + r0 + 16 * seg;
            if (16 * seg + 16 <= nrows) {
                *reinterpret_cast<uint4 *>(dst) = o;
            } else {
                const uint32_t ow[4] = {o.x, o.y, o.z, o.w};
                for (int b = 0; b < 16; ++b)
                    if (16 * seg + b < nrows) dst[b] = (uint8_t)((ow[b >> 2] >> (8 * (b & 3))) & 0xffu);
            }
        }
    }
}

// The lean instantiation hard-codes 0/1/2 genotypes: identity codes AND exactly three values in EVERY column of a
// non-empty list (K_used == 2 * pt alone also holds for, say, one 2-valued plus one 4-valued column).
static bool lean_encode(bool all_ident, bool all_v3, int64_t pc) { return all_ident && all_v3 && pc > 0; }

// Clears what the encode launches that fill the distance operands U [u_rows, K/2 bytes] and Wd [n, K/2 bytes]
// do not write.  The lean kernel writes every byte of its columns, so only the K padding (reduced rows
// K_used..K); the general kernel ORs the words at unaligned tile edges in, so everything.
static void clear_dist_ops(bool lean, int8_t *U, int64_t u_rows, int8_t *Wd, int64_t n, int64_t K_used, int64_t K,
                           cudaStream_t st) {
    const size_t Kb = (size_t)K / 2;
    if (!lean) {
        FS_CUDA(cudaMemsetAsync(U, 0, (size_t)u_rows * Kb, st));
        FS_CUDA(cudaMemsetAsync(Wd, 0, (size_t)n * Kb, st));
    } else if (K > K_used) {
        FS_CUDA(cudaMemset2DAsync(U + K_used / 2, Kb, 0, (size_t)(K - K_used) / 2, (size_t)u_rows, st));
        FS_CUDA(cudaMemset2DAsync(Wd + K_used / 2, Kb, 0, (size_t)(K - K_used) / 2, (size_t)n, st));
    }
}

// One launch of the encode over the columns tcol[0, pc): the lean kernel (see lean_encode), else the general
// kernel in the input's type.  off: the columns' first reduced rows; uk0: the reduced row of U and Wd that off's
// row 0 stands for.  Null outputs are not written.
static void launch_encode(const fs_dataset *ds, bool lean, int all_ident, const int64_t *tcol, const int32_t *off, int64_t pc,
                          int64_t K, int64_t ldt, int64_t ldc, int8_t *U, int8_t *Wd, int8_t *At, uint8_t *codesT,
                          uint8_t *codes, int32_t *srow, uint32_t *krow, int64_t u_lo, int64_t u_hi, const int32_t *tpos,
                          int uk0, WdRows wr, cudaStream_t st, int *launches) {
    const int64_t n = ds->n;
    const unsigned grid = (unsigned)(ceil_div(pc, ENC_COLS) * ceil_div(n, ENC_ROWS));
    const int as_f32 = (ds->arith == FS_ARITH_F32 && ds->dtype == FS_F64) ? 1 : 0;
    auto encode = [&](auto type_tag, auto lean_tag) {
        using T = decltype(type_tag);
        onehot_encode_kernel<T, decltype(lean_tag)::value><<<grid, 256, 0, st>>>(
            static_cast<const T *>(ds->x), ds->ldx, ds->d_perm.ptr, tcol, off, ds->d_vals.ptr, as_f32, n, pc, K, ldt, ldc,
            U, Wd, At, codesT, codes, srow, krow, all_ident, u_lo, u_hi, tpos, uk0, wr);
    };
    if (lean) {
        encode(uint8_t{}, std::true_type{});      // FS_U8 and FS_I8 alike: the bytes are the codes 0/1/2
    } else {
        switch (ds->dtype) {
            case FS_U8: encode(uint8_t{}, std::false_type{}); break;
            case FS_I8: encode(int8_t{}, std::false_type{}); break;
            case FS_F32: encode(float{}, std::false_type{}); break;
            case FS_F64: encode(double{}, std::false_type{}); break;
        }
    }
    FS_CUDA(cudaGetLastError());
    ++*launches;
}

// Distance operands (Ur, Wdr, srow_r) of the columns removed since the cached slab was built.
static void build_removed(fs_dataset *ds, WorkSet &ws, int *launches) {
    Trace tr("    build_removed");
    const int64_t n = ds->n, pr = (int64_t)ws.removed.size();
    ws.p_rcol.reserve(pr);
    ws.p_roff.reserve(pr + 1);
    int64_t K = 0;
    unsigned ident = kColIdent;
    bool v3 = true;
    for (int64_t c = 0; c < pr; ++c) {
        const unsigned ci = ds->col_info[ws.removed[c]];
        v3 = v3 && (ci >> 4) == 2;
        ws.p_rcol.ptr[c] = ws.removed[c];
        ws.p_roff.ptr[c] = (int32_t)K;
        K += ci >> 4;
        ident &= ci;
    }
    ws.p_roff.ptr[pr] = (int32_t)K;
    ws.Kr_used = K;
    ws.Kr = round_up(K, 256);                 // elements (FP4 nibbles); rows are Kr / 2 bytes
    ws.rcol.reserve(pr);
    ws.roff.reserve(pr + 1);
    const size_t Kb = (size_t)ws.Kr / 2;
    ws.Ur.reserve((size_t)n * Kb);
    ws.Wdr.reserve((size_t)n * Kb);
    ws.srow_r.reserve(ws.ldt);
    cudaStream_t st = ds->stream;
    FS_CUDA(cudaMemcpyAsync(ws.rcol.ptr, ws.p_rcol.ptr, pr * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    FS_CUDA(cudaMemcpyAsync(ws.roff.ptr, ws.p_roff.ptr, (pr + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    FS_CUDA(cudaMemsetAsync(ws.srow_r.ptr, 0, ws.ldt * sizeof(int32_t), st));
    const int all_ident = (ident & kColIdent) ? 1 : 0;
    const bool lean = lean_encode(all_ident, v3, pr);
    clear_dist_ops(lean, ws.Ur.ptr, n, ws.Wdr.ptr, n, ws.Kr_used, ws.Kr, st);
    launch_encode(ds, lean, all_ident, ws.rcol.ptr, ws.roff.ptr, pr, (int64_t)Kb, ws.ldt, 0, ws.Ur.ptr, ws.Wdr.ptr, nullptr,
                  nullptr, nullptr, ws.srow_r.ptr, nullptr, 0, n, nullptr, 0, WdRows{0, n, 0, 0}, st, launches);
}

void build_onehot(fs_dataset *ds, WorkSet &ws, bool group_call, int *launches) {
    const int64_t n = ds->n, pt = ws.pt;
    // tcol / tout / toff, K_used, all_ident and the accumulation slice [a0, a1) were filled by build_lists
    ws.K = round_up(ws.K_used, 256);          // elements (FP4 nibbles); U / Wd rows are K / 2 bytes
    ws.ldt = round_up(n, 128);
    ws.ldc = round_up(pt, 16);
    FS_REQUIRE(pt < (1LL << 24), FS_ERR_INVALID, "too many one-hot columns (%lld)", (long long)pt);
    ws.tcol.reserve(pt);
    ws.tout.reserve(pt);
    ws.toff.reserve(pt + 1);
    const bool ops = ws.have_dist_ops;
    // accumulation operands: the slice [a0, a1) of the active columns (all of them outside a multi-GPU
    // group), one-hot rows numbered from 0
    const int64_t a0 = ws.a0, a1 = ws.a1, pa = a1 - a0;
    const bool split = ws.acc_split;
    ws.Ka_used = ws.p_toff.ptr[a1] - ws.p_toff.ptr[a0];
    ws.Ka = round_up(ws.Ka_used, 256);
    if (ops) {
        ws.U.reserve((size_t)(ws.u_hi - ws.u_lo) * (ws.K / 2));   // target rows of this call only
        ws.Wd.reserve((size_t)n * (ws.K / 2));
        ws.srow.reserve(ws.ldt);   // padded: the distance epilogue reads it in 16-byte vectors
    }
    ws.At.reserve((size_t)std::max<int64_t>(ws.Ka, 256) * (ws.ldt / 2));          // FP4 nibbles: two samples per byte
    // codesT (value codes, feature-major) depends on a column only, not on which other columns are
    // active: when every column of the slice already has a row in the resident codesT of an earlier, wider
    // encode (TuRF iterations), that table is kept and the one-hot rows point into it (krow)
    bool reuse_ct = ds->ct_valid;
    for (int64_t c = a0; c < a1 && reuse_ct; ++c) reuse_ct = ds->ct_pos[ws.p_tcol.ptr[c]] >= 0;
    if (reuse_ct) {
        ws.p_tpos.reserve(std::max<int64_t>(pa, 1));
        for (int64_t c = a0; c < a1; ++c) ws.p_tpos.ptr[c - a0] = ds->ct_pos[ws.p_tcol.ptr[c]];
        ws.tpos.reserve(std::max<int64_t>(pa, 1));
    } else {
        ws.codesT.reserve((size_t)pa * ws.ldt + 512);   // slack: the accumulation epilogue reads whole 128-byte runs
        if (ds->ct_version != ws.lists_version || (int64_t)ds->ct_pos.size() != ds->p) {
            ds->ct_pos.assign(ds->p, -1);
            for (int64_t c = a0; c < a1; ++c) ds->ct_pos[ws.p_tcol.ptr[c]] = (int32_t)(c - a0);
            ds->ct_version = ws.lists_version;
        }
        ds->ct_valid = true;
    }
    if (ws.have_codes) ws.codes.reserve((size_t)n * ws.ldc);
    ws.krow.reserve(std::max<int64_t>(ws.Ka, 256));
    cudaStream_t st = ds->stream;
    if (reuse_ct && pa > 0) FS_CUDA(cudaMemcpyAsync(ws.tpos.ptr, ws.p_tpos.ptr, pa * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    if (!ws.lists_uploaded) {
        // (skipped when the cached lists of an all-columns call are already on the device)
        FS_CUDA(cudaMemcpyAsync(ws.tcol.ptr, ws.p_tcol.ptr, pt * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        FS_CUDA(cudaMemcpyAsync(ws.tout.ptr, ws.p_tout.ptr, pt * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        FS_CUDA(cudaMemcpyAsync(ws.toff.ptr, ws.p_toff.ptr, (pt + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        // slice-local row offsets (the general encoder and the final reduction read them)
        ws.p_atoff.reserve(pa + 1);
        for (int64_t c = 0; c <= pa; ++c) ws.p_atoff.ptr[c] = ws.p_toff.ptr[a0 + c] - ws.p_toff.ptr[a0];
        ws.atoff.reserve(pa + 1);
        FS_CUDA(cudaMemcpyAsync(ws.atoff.ptr, ws.p_atoff.ptr, (pa + 1) * sizeof(int32_t), cudaMemcpyHostToDevice, st));
        ws.lists_uploaded = true;
    }
    const size_t Kb = (size_t)ws.K / 2;
    const bool lean = lean_encode(ws.all_ident, ws.all_v3, pt);
    if (ops) {
        FS_CUDA(cudaMemsetAsync(ws.srow.ptr, 0, ws.ldt * sizeof(int32_t), st));
        clear_dist_ops(lean, ws.U.ptr, ws.u_hi - ws.u_lo, ws.Wd.ptr, n, ws.K_used, ws.K, st);
    }
    // the encode writes every used byte of At and codesT exactly once; only the K padding (reduced rows
    // Ka_used..Ka) has to be cleared.  Sample padding of the feature-major rows (columns n..ldt) is never
    // read (the TMA maps are n bytes wide).
    if (ws.Ka > ws.Ka_used)
        FS_CUDA(cudaMemsetAsync(ws.At.ptr + (size_t)ws.Ka_used * (ws.ldt / 2), 0, (size_t)(ws.Ka - ws.Ka_used) * (ws.ldt / 2), st));
    const int all_ident = ws.all_ident ? 1 : 0;
    // One fused launch when the accumulation operands cover the same columns as the distance operands;
    // in a multi-GPU group two: the distance operands of ALL active columns (every rank needs Wd of all
    // samples), then the accumulation operands of this rank's slice only.
    // Wd rows this rank's distance kernel reads (see WdRows)
    WdRows wr{0, n, 0, 0};
    if (group_call) {
        const DistPeers &pr = ds->peers;
        const int G = pr.world, r = pr.rank, last = r + G / 2;          // ranks r .. r + floor(G / 2) on the ring
        if (last < G) {
            wr = WdRows{pr.starts[r], pr.starts[last + 1], 0, 0};
        } else {
            wr = WdRows{pr.starts[r], n, 0, pr.starts[last - G + 1]};
        }
    }
    auto launch = [&](int64_t c_lo, int64_t c_hi, bool want_dist, bool want_acc, bool want_codes) {
        const int64_t pc = c_hi - c_lo;
        if (pc <= 0 || (!want_dist && !want_acc && !want_codes)) return;
        // slice-local offsets: one-hot rows from 0, codesT rows from 0
        const bool local_rows = want_acc && c_lo == a0;        // At / krow rows numbered from the slice's first column
        const int32_t *off = local_rows ? ws.atoff.ptr : ws.toff.ptr + c_lo;
        const int uk0 = local_rows ? ws.p_toff.ptr[a0] : 0;    // where those rows sit in U / Wd
        int8_t *Uo = want_dist ? ws.U.ptr : nullptr, *Wo = want_dist ? ws.Wd.ptr : nullptr;
        int8_t *Ao = want_acc ? ws.At.ptr : nullptr;
        uint8_t *Co = want_acc && !reuse_ct ? ws.codesT.ptr : nullptr;
        uint32_t *Ko = want_acc ? ws.krow.ptr : nullptr;
        const int32_t *To = want_acc && reuse_ct ? ws.tpos.ptr : nullptr;
        int32_t *So = want_dist ? ws.srow.ptr : nullptr;
        uint8_t *codes = want_codes ? ws.codes.ptr : nullptr;       // sample-major value codes (ReliefF)
        launch_encode(ds, lean, all_ident, ws.tcol.ptr + c_lo, off, pc, (int64_t)Kb, ws.ldt, ws.ldc, Uo, Wo, Ao, Co, codes, So,
                      Ko, ws.u_lo, ws.u_hi, To, uk0, wr, st, launches);
    };
    if (!split) {
        launch(0, pt, ops, true, ws.have_codes);
    } else if (ops && (a0 % ENC_COLS) == 0 && (ws.p_toff.ptr[a0] & 31) == 0 &&
               (a1 == pt || ((a1 % ENC_COLS) == 0 && (ws.p_toff.ptr[a1] & 31) == 0))) {
        // the slice in ONE fused launch (distance and accumulation operands, as on one GPU), the other
        // columns distance-only: no column is staged twice
        launch(a0, a1, true, true, false);
        launch(0, a0, true, false, false);
        launch(a1, pt, true, false, false);
    } else {
        // (the distance launch addresses U / Wd by the GLOBAL one-hot offsets of toff, the slice launch
        // addresses At / krow by the slice-local ones)
        launch(0, pt, ops, false, ws.have_codes);
        launch(a0, a1, false, true, false);
    }
    // no synchronisation here: the pinned staging buffers live in the working set and are only
    // rewritten by the next build, which starts after fs_score's final stream synchronisation
    if (ws.dist_mode == kDistIncremental) build_removed(ds, ws, launches);
}

}  // namespace fs
