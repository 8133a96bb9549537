// mdr.cu -- multifactor dimensionality reduction (MDR): exhaustive one- and two-locus search of columns
// with at most 3 distinct values for the combination whose high-risk / low-risk cell labelling best
// separates a binary class, scored by cross-validated balanced accuracy.  The semantics are this
// project's own (DESIGN.md, "MDR"); oracle/mdr_oracle.py restates them in numpy.
//
// Data flow (all on the data set's stream):
//   encode   the reduced one-hot rows At [K, n] of the columns, shared with the joint-count path
//            (discrete_operand; a column with V <= 3 values owns V - 1 rows, a constant column none).
//   pack     At -> uint32 bit-planes [K, W] in SEGMENT order: segment s = 2 * fold + class holds the words
//            [seg.w[s], seg.w[s + 1]), padded with zero bits to whole words, so every word belongs to one
//            segment; plus the popcount of every row in every segment (marg [K, 2 cv]).  Reads K * n / 2
//            bytes.  Cached per (column list, folds) until the working set is rebuilt.
//   scan     16 x 16 position tiles of the upper triangle, one thread per pair: per word at most 2 x 2
//            AND + POPC of the pair's reduced rows (staged in shared memory), counted per segment in
//            registers (4 * 2 cv <= 80).  The full 3 x 3 table of every segment follows from the segment
//            marginals, as in joint_visit.  Every fold is evaluated in integers with one float64 division
//            per balanced accuracy.  Persistent blocks keep a block-local top list (mean test BA
//            descending, index ascending) and the per-fold best training BA.
//   merge    pairwise merges of the block lists (log2 of the grid launches) and one reduction of the
//            fold bests.  Every comparison is on (score, index), a total order, so the result does not
//            depend on which block saw which pair.
// fs_mdr_tables counts the per-segment tables of chosen combinations from the same planes.
//
// fs_interaction_scan (DESIGN.md section 11) is the same pack, scan and merge with a single fold, so the two
// segments are the two classes, and another evaluation policy: the KSA statistic of BOOST from the two
// class tables instead of balanced accuracies, and no fold bests.  The tables of the listed pairs follow
// from mdr_tables_kernel on the same planes.
#include <algorithm>
#include <climits>
#include <cmath>
#include <cstring>

#include "common.cuh"
#include "joint_math.cuh"

namespace fs {
namespace {

constexpr int kMdrMaxFolds = 10;
static_assert(2 * kMdrMaxFolds == kMdrMaxSegments, "MdrSeg holds 2 segments per fold");
constexpr int kMdrTile = 16;                        // positions per tile side: 16 x 16 pairs, one per thread
constexpr int kMdrThreads = kMdrTile * kMdrTile;
constexpr int kMdrChunk = 128;                      // words of a staged chunk
constexpr int kMdrLd = kMdrChunk + 1;               // odd row stride: the 16 B rows a warp reads sit in 16 banks
constexpr int kMdrPackRows = 16;                    // reduced rows per pack thread (its slot map is loaded once)

struct MdrCand {
    double score;                                   // mean test BA (top list) or training BA of a fold
    double train;                                   // mean training BA (top list)
    long long idx;                                  // combination index
};

__device__ __forceinline__ bool better(double s1, long long i1, double s2, long long i2) {
    return s1 > s2 || (s1 == s2 && i1 < i2);
}
__device__ __forceinline__ bool better(const MdrCand &a, const MdrCand &b) { return better(a.score, a.idx, b.score, b.idx); }

// number of entries of arr (sorted best first) better than x -- or, with or_equal, not worse than x
__device__ __forceinline__ int rank_in(const MdrCand *arr, int len, const MdrCand &x, bool or_equal) {
    int lo = 0, hi = len;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        const bool ahead = better(arr[mid], x) || (or_equal && arr[mid].score == x.score && arr[mid].idx == x.idx);
        if (ahead) lo = mid + 1;
        else hi = mid;
    }
    return lo;
}

// planes[k * W + w] bit b = 1 iff the sample in slot 32 w + b carries reduced row k (At nibble 0x2; low
// nibble = even sample).  slot[32 w + b]: internal row of that slot, -1 for padding.  marg[k * nseg + s] +=
// popcount of the word (integer atomics: the sum does not depend on their order).
__global__ void __launch_bounds__(128) mdr_pack_kernel(const int8_t *__restrict__ At, int64_t pitch, int64_t K,
                                                       const int32_t *__restrict__ slot, const uint8_t *__restrict__ wseg,
                                                       int64_t W, int nseg, uint32_t *__restrict__ planes,
                                                       int32_t *__restrict__ marg) {
    const int64_t w = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (w >= W) return;
    int32_t src[32];
    const int4 *sv = reinterpret_cast<const int4 *>(slot + 32 * w);
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int4 v = sv[q];
        src[4 * q] = v.x;
        src[4 * q + 1] = v.y;
        src[4 * q + 2] = v.z;
        src[4 * q + 3] = v.w;
    }
    const int seg = wseg[w];
    const uint8_t *base = reinterpret_cast<const uint8_t *>(At);
    const int64_t groups = (K + kMdrPackRows - 1) / kMdrPackRows;
    for (int64_t g = blockIdx.y; g < groups; g += gridDim.y) {
        const int64_t k1 = std::min<int64_t>(K, (g + 1) * kMdrPackRows);
        for (int64_t k = g * kMdrPackRows; k < k1; ++k) {
            const uint8_t *row = base + k * pitch;
            uint32_t m = 0;
#pragma unroll
            for (int b = 0; b < 32; ++b)
                if (src[b] >= 0) m |= (((unsigned)__ldg(row + (src[b] >> 1)) >> (4 * (src[b] & 1) + 1)) & 1u) << b;
            planes[k * W + w] = m;
            const int c = __popc(m);
            if (c) atomicAdd(marg + k * nseg + seg, c);
        }
    }
}

// Everything one scan block reads besides the planes.
struct MdrScanArgs {
    const uint32_t *planes;                         // [K, W]
    const int32_t *marg;                            // [K, nseg]
    const int32_t *start;                           // [n_kept + 1] first reduced row of every position
    int64_t W, n_kept, n_tiles, tiles_side;
    int n_top;
    double *all_train, *all_test;                   // [n_combos] or null: cand.train (MDR only), cand.score
    MdrCand *top_out;                               // [gridDim.x, n_top]
    MdrCand *fold_out;                              // [gridDim.x, n_folds] (MDR only)
};

// Full 3 x 3 table of one segment, cell va * 3 + vb, from the pair's reduced counts c[i][j] and the
// segment marginals m*: the reconstruction of joint_visit, written out over the compile-time 3 x 3 cells so
// that it stays in registers.  Rows a column does not own are zero planes, so their counts and marginals
// are 0 and the same expressions hold for V = 1, 2, 3.
__device__ __forceinline__ void seg_table(int la, int lb, int32_t ma0, int32_t ma1, int32_t mb0, int32_t mb1, uint32_t c00,
                                          uint32_t c01, uint32_t c10, uint32_t c11, int32_t ns, int32_t t[9]) {
    const int32_t c[2][2] = {{(int32_t)c00, (int32_t)c01}, {(int32_t)c10, (int32_t)c11}};
    const int32_t ma[2] = {ma0, ma1}, mb[2] = {mb0, mb1};
    const int32_t last = ns - (ma0 + ma1) - (mb0 + mb1) + (c[0][0] + c[0][1] + c[1][0] + c[1][1]);
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j) {
            int32_t v = 0;
            if (i < 2 && j < 2 && i < la && j < lb) v = c[i < 2 ? i : 0][j < 2 ? j : 0];
            else if (i < 2 && i < la && j == lb) v = ma[i < 2 ? i : 0] - c[i < 2 ? i : 0][0] - c[i < 2 ? i : 0][1];
            else if (j < 2 && i == la && j < lb) v = mb[j < 2 ? j : 0] - c[0][j < 2 ? j : 0] - c[1][j < 2 ? j : 0];
            else if (i == la && j == lb) v = last;
            t[i * 3 + j] = v;
        }
}

// Balanced accuracy of one split: (TP * N0 + TN * N1) / (2 N1 N0), exact integers, one division.
__device__ __forceinline__ double balanced(int64_t tp, int64_t tn, int32_t n1, int32_t n0) {
    return (double)(tp * n0 + tn * n1) / (double)(2 * (int64_t)n1 * n0);
}

// All folds of one combination from its per-segment reduced counts c[s][4] (pairs) and the marginals of
// its rows.  train[f] / test[f]: the fold's balanced accuracies; the means are summed in fold order.
template <int NSEG>
__device__ __forceinline__ void mdr_evaluate(int la, int lb, int ka, int kb, const int32_t *__restrict__ marg,
                                             const MdrSeg &seg, const uint32_t (&c)[NSEG][4], double (&train)[NSEG / 2],
                                             double &mean_train, double &mean_test) {
    constexpr int NF = NSEG / 2;
    auto m = [&](int k, int have, int s) -> int32_t { return have ? __ldg(marg + (int64_t)k * NSEG + s) : 0; };
    auto table = [&](int s, int32_t t[9]) {
        seg_table(la, lb, m(ka, la > 0, s), m(ka + 1, la > 1, s), m(kb, lb > 0, s), m(kb + 1, lb > 1, s), c[s][0], c[s][1],
                  c[s][2], c[s][3], seg.n[s], t);
    };
    int32_t all0[9], all1[9];
#pragma unroll
    for (int g = 0; g < 9; ++g) all0[g] = all1[g] = 0;
    int32_t n0 = 0, n1 = 0;
#pragma unroll
    for (int s = 0; s < NSEG; ++s) {
        int32_t t[9];
        table(s, t);
#pragma unroll
        for (int g = 0; g < 9; ++g) {
            if (s & 1) all1[g] += t[g];
            else all0[g] += t[g];
        }
        if (s & 1) n1 += seg.n[s];
        else n0 += seg.n[s];
    }
    double acc_train = 0.0, acc_test = 0.0;
#pragma unroll
    for (int f = 0; f < NF; ++f) {
        int32_t e0[9], e1[9];
        table(2 * f, e0);
        table(2 * f + 1, e1);
        const int32_t M0 = seg.n[2 * f], M1 = seg.n[2 * f + 1], N0 = n0 - M0, N1 = n1 - M1;
        int64_t TP = 0, TN = 0, tp = 0, tn = 0;
#pragma unroll
        for (int g = 0; g < 9; ++g) {
            const int32_t T0 = all0[g] - e0[g], T1 = all1[g] - e1[g];
            if ((int64_t)T1 * N0 > (int64_t)T0 * N1) {        // high risk; ties and empty cells are low risk
                TP += T1;
                tp += e1[g];
            } else {
                TN += T0;
                tn += e0[g];
            }
        }
        train[f] = balanced(TP, TN, N1, N0);
        acc_train += train[f];
        acc_test += balanced(tp, tn, M1, M0);
    }
    mean_train = acc_train / (double)NF;
    mean_test = acc_test / (double)NF;
}

// KSA statistic of one pair from its class tables t[k][i * 3 + j] and class sizes nk[k], in the operation
// order of DESIGN.md section 11 (cells in (i, j, k) order, products left to right).  The explicit
// round-to-nearest intrinsics keep the compiler from contracting the sum into FMAs, so the order holds.
__device__ __forceinline__ double ksa_statistic(const int32_t (&t)[2][9], const int32_t (&nk)[2]) {
    int32_t ni[3], nj[3], nik[3][2], njk[3][2];
#pragma unroll
    for (int i = 0; i < 3; ++i) {
        ni[i] = nj[i] = 0;
        nik[i][0] = nik[i][1] = njk[i][0] = njk[i][1] = 0;
    }
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j)
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const int32_t v = t[k][i * 3 + j];
                ni[i] += v;
                nj[j] += v;
                nik[i][k] += v;
                njk[j][k] += v;
            }
    double q[18];
    double eta = 0.0;
#pragma unroll
    for (int i = 0; i < 3; ++i)
#pragma unroll
        for (int j = 0; j < 3; ++j)
#pragma unroll
            for (int k = 0; k < 2; ++k) {
                const int32_t nij = t[0][i * 3 + j] + t[1][i * 3 + j];
                double v = 0.0;
                if (nij > 0 && nik[i][k] > 0 && njk[j][k] > 0)
                    v = __dmul_rn(__dmul_rn((double)nij, (double)nik[i][k]), (double)njk[j][k]) /
                        __dmul_rn(__dmul_rn((double)ni[i], (double)nj[j]), (double)nk[k]);
                q[(i * 3 + j) * 2 + k] = v;
                eta = __dadd_rn(eta, v);
            }
    const double N = (double)(nk[0] + nk[1]);
    double L = 0.0;
#pragma unroll
    for (int g = 0; g < 18; ++g) {
        const int32_t n = t[g & 1][g >> 1];
        if (n > 0) L = __dadd_rn(L, __dmul_rn((double)n, log(__dmul_rn((double)n, eta) / __dmul_rn(N, q[g]))));
    }
    return 2.0 * L;
}

// Evaluation policies of mdr_scan_kernel: eval turns a pair's (or column's) per-segment counts into the
// candidate's score (the top-list key) and train value, and the fold bests of the NF folds it reports in train.
template <int NSEG>
struct MdrEval {                                    // MDR: mean test / training balanced accuracy, fold bests
    static constexpr int NF = NSEG / 2;
    static __device__ __forceinline__ void eval(int la, int lb, int ka, int kb, const int32_t *__restrict__ marg,
                                                const MdrSeg &seg, const uint32_t (&c)[NSEG][4], double (&train)[NF],
                                                MdrCand &cand) {
        mdr_evaluate<NSEG>(la, lb, ka, kb, marg, seg, c, train, cand.train, cand.score);
    }
};

struct KsaEval {                                    // one fold, segments = classes: L_KSA, no fold bests
    static constexpr int NF = 0;
    static __device__ __forceinline__ void eval(int la, int lb, int ka, int kb, const int32_t *__restrict__ marg,
                                                const MdrSeg &seg, const uint32_t (&c)[2][4], double (&)[1],
                                                MdrCand &cand) {
        auto m = [&](int k, int have, int s) -> int32_t { return have ? __ldg(marg + (int64_t)k * 2 + s) : 0; };
        int32_t t[2][9];
#pragma unroll
        for (int s = 0; s < 2; ++s)
            seg_table(la, lb, m(ka, la > 0, s), m(ka + 1, la > 1, s), m(kb, lb > 0, s), m(kb + 1, lb > 1, s), c[s][0],
                      c[s][1], c[s][2], c[s][3], seg.n[s], t[s]);
        const int32_t nk[2] = {seg.n[0], seg.n[1]};
        cand.score = ksa_statistic(t, nk);
        cand.train = 0.0;
    }
};

// first linear tile of tile row i of the upper triangle (T tile rows): i * T - i (i - 1) / 2
__device__ __forceinline__ int64_t tri_off(int64_t i, int64_t T) { return i * T - i * (i - 1) / 2; }

// Dynamic shared memory: staged rows (pairs only) | top list | merge target | candidate buffer | sorted buffer.
__host__ __device__ inline size_t mdr_smem_bytes(bool pair, int n_top) {
    return (pair ? (size_t)4 * kMdrTile * kMdrLd * sizeof(uint32_t) : 0) +
           (2 * (size_t)n_top + 2 * kMdrThreads) * sizeof(MdrCand);
}

template <int NSEG, bool PAIR, class Eval>
__global__ void __launch_bounds__(kMdrThreads) mdr_scan_kernel(const MdrScanArgs args, const MdrSeg seg) {
    constexpr int NF = Eval::NF;
    constexpr int NFA = NF > 0 ? NF : 1;              // array extent: KsaEval keeps no fold bests
    extern __shared__ __align__(16) unsigned char smem[];
    uint32_t *stile = reinterpret_cast<uint32_t *>(smem);                 // [4 * kMdrTile rows][kMdrLd]: A rows, then B rows
    MdrCand *list = reinterpret_cast<MdrCand *>(smem + (PAIR ? (size_t)4 * kMdrTile * kMdrLd * sizeof(uint32_t) : 0));
    MdrCand *list2 = list + args.n_top;
    MdrCand *buf = list2 + args.n_top;
    MdrCand *sbuf = buf + kMdrThreads;
    __shared__ int s_rows[4 * kMdrTile];              // plane row of every staged row, -1: none
    __shared__ int s_cnt, s_nbuf;
    __shared__ double s_fb[kMdrThreads / 32][NFA];    // per warp: best training BA of every fold
    __shared__ long long s_fi[kMdrThreads / 32][NFA];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int tx = tid % kMdrTile, ty = tid / kMdrTile;
    if (tid == 0) {
        s_cnt = 0;
        s_nbuf = 0;
    }
    if (lane < NF) {
        s_fb[warp][lane] = -INFINITY;
        s_fi[warp][lane] = LLONG_MAX;
    }
    __syncthreads();
    const int64_t nk = args.n_kept;
    for (int64_t t = blockIdx.x; t < args.n_tiles; t += gridDim.x) {
        int64_t a, b = -1;
        if (PAIR) {
            const int64_t T = args.tiles_side;
            const double q = 2.0 * (double)T + 1.0;
            int64_t ti = (int64_t)floor((q - sqrt(q * q - 8.0 * (double)t)) * 0.5);
            ti = ti < 0 ? 0 : (ti > T - 1 ? T - 1 : ti);
            while (ti > 0 && tri_off(ti, T) > t) --ti;
            while (ti + 1 < T && tri_off(ti + 1, T) <= t) ++ti;
            const int64_t tj = ti + (t - tri_off(ti, T));
            a = ti * kMdrTile + ty;
            b = tj * kMdrTile + tx;
            if (tid < 4 * kMdrTile) {                   // staged row tid: side, position, reduced row
                const int side = tid >> 5, pos = (tid >> 1) & (kMdrTile - 1), r = tid & 1;
                const int64_t q0 = (side ? tj : ti) * kMdrTile + pos;
                int row = -1;
                if (q0 < nk && args.start[q0] + r < args.start[q0 + 1]) row = args.start[q0] + r;
                s_rows[tid] = row;
            }
        } else {
            a = t * kMdrThreads + tid;
        }
        const bool valid = PAIR ? (a < b && b < nk) : (a < nk);
        uint32_t c[NSEG][4];
#pragma unroll
        for (int s = 0; s < NSEG; ++s) c[s][0] = c[s][1] = c[s][2] = c[s][3] = 0;
        if (PAIR) {
            const uint32_t *pA = stile + (2 * ty) * kMdrLd;
            const uint32_t *pB = stile + (2 * kMdrTile + 2 * tx) * kMdrLd;
            for (int64_t w0 = 0; w0 < args.W; w0 += kMdrChunk) {
                const int nw = (int)std::min<int64_t>(kMdrChunk, args.W - w0);
                __syncthreads();                        // s_rows written / the previous chunk consumed
                {
                    // 4 threads per staged row, 16 B loads (W and w0 are multiples of 4)
                    const int row = tid >> 2, part = tid & 3;
                    const int kr = s_rows[row];
                    uint32_t *dst = stile + row * kMdrLd;
                    for (int w = 4 * part; w < nw; w += 16) {
                        uint4 v = make_uint4(0u, 0u, 0u, 0u);
                        if (kr >= 0) v = __ldg(reinterpret_cast<const uint4 *>(args.planes + (int64_t)kr * args.W + w0 + w));
                        dst[w] = v.x;
                        dst[w + 1] = v.y;
                        dst[w + 2] = v.z;
                        dst[w + 3] = v.w;
                    }
                }
                __syncthreads();
#pragma unroll
                for (int s = 0; s < NSEG; ++s) {
                    const int lo = (int)std::max<int64_t>(seg.w[s] - w0, 0), hi = (int)std::min<int64_t>(seg.w[s + 1] - w0, nw);
                    uint32_t c0 = 0, c1 = 0, c2 = 0, c3 = 0;
#pragma unroll 4
                    for (int w = lo; w < hi; ++w) {
                        const uint32_t a0 = pA[w], a1 = pA[kMdrLd + w], b0 = pB[w], b1 = pB[kMdrLd + w];
                        c0 += __popc(a0 & b0);
                        c1 += __popc(a0 & b1);
                        c2 += __popc(a1 & b0);
                        c3 += __popc(a1 & b1);
                    }
                    c[s][0] += c0;
                    c[s][1] += c1;
                    c[s][2] += c2;
                    c[s][3] += c3;
                }
            }
        }
        MdrCand cand{-INFINITY, 0.0, LLONG_MAX};
        double train[NFA];
#pragma unroll
        for (int f = 0; f < NF; ++f) train[f] = -INFINITY;
        if (valid) {
            const int ka = args.start[a], la = args.start[a + 1] - ka;
            const int kb = PAIR ? args.start[b] : 0, lb = PAIR ? args.start[b + 1] - kb : 0;
            Eval::eval(la, lb, ka, kb, args.marg, seg, c, train, cand);
            cand.idx = PAIR ? (long long)(a * nk - a * (a + 1) / 2 + (b - a - 1)) : (long long)a;
            if (args.all_test) {
                if (NF > 0) args.all_train[cand.idx] = cand.train;
                args.all_test[cand.idx] = cand.score;
            }
        }
        // per-fold best training BA: warp argmax, then the warp's slot (written by its lane 0 only)
#pragma unroll
        for (int f = 0; f < NF; ++f) {
            double v = train[f];
            long long i = valid ? cand.idx : LLONG_MAX;
#pragma unroll
            for (int o = 16; o >= 1; o >>= 1) {
                const double v2 = __shfl_xor_sync(0xffffffffu, v, o);
                const long long i2 = __shfl_xor_sync(0xffffffffu, i, o);
                if (better(v2, i2, v, i)) {
                    v = v2;
                    i = i2;
                }
            }
            if (lane == 0 && better(v, i, s_fb[warp][f], s_fi[warp][f])) {
                s_fb[warp][f] = v;
                s_fi[warp][f] = i;
            }
        }
        // top list: candidates that beat the current last entry go to the buffer, then one merge
        const int cnt = s_cnt;
        if (valid && (cnt < args.n_top || better(cand, list[args.n_top - 1]))) buf[atomicAdd(&s_nbuf, 1)] = cand;
        __syncthreads();
        const int nb = s_nbuf;
        if (nb > 0) {
            if (tid < nb) {
                const MdrCand x = buf[tid];
                int r = 0;
                for (int u = 0; u < nb; ++u) r += better(buf[u], x);
                sbuf[r] = x;                            // keys are distinct: a permutation
            }
            __syncthreads();
            for (int i = tid; i < cnt; i += kMdrThreads) {
                const int pos = i + rank_in(sbuf, nb, list[i], false);
                if (pos < args.n_top) list2[pos] = list[i];
            }
            for (int j = tid; j < nb; j += kMdrThreads) {
                const int pos = j + rank_in(list, cnt, sbuf[j], false);
                if (pos < args.n_top) list2[pos] = sbuf[j];
            }
            __syncthreads();
            const int ncnt = std::min(args.n_top, cnt + nb);
            for (int i = tid; i < ncnt; i += kMdrThreads) list[i] = list2[i];
            if (tid == 0) {
                s_cnt = ncnt;
                s_nbuf = 0;
            }
        }
        __syncthreads();
    }
    MdrCand *out = args.top_out + (int64_t)blockIdx.x * args.n_top;
    for (int i = tid; i < args.n_top; i += kMdrThreads) out[i] = i < s_cnt ? list[i] : MdrCand{-INFINITY, 0.0, LLONG_MAX};
    if (tid < NF) {
        double v = -INFINITY;
        long long i = LLONG_MAX;
        for (int q = 0; q < kMdrThreads / 32; ++q)
            if (better(s_fb[q][tid], s_fi[q][tid], v, i)) {
                v = s_fb[q][tid];
                i = s_fi[q][tid];
            }
        args.fold_out[(int64_t)blockIdx.x * NF + tid] = MdrCand{v, 0.0, i};
    }
}

// out list q = the best n_top of in lists 2q and 2q + 1 (each sorted best first, padded with sentinels).
// Stable merge: an entry of the first list goes before an equal entry of the second, so positions are a
// permutation even among the sentinels.
__global__ void __launch_bounds__(256) mdr_merge_kernel(const MdrCand *__restrict__ in, int64_t L, int n_top,
                                                        MdrCand *__restrict__ out) {
    const int64_t q = blockIdx.x;
    const MdrCand *A = in + 2 * q * n_top;
    MdrCand *o = out + q * n_top;
    if (2 * q + 1 >= L) {
        for (int i = threadIdx.x; i < n_top; i += blockDim.x) o[i] = A[i];
        return;
    }
    const MdrCand *B = A + n_top;
    for (int i = threadIdx.x; i < n_top; i += blockDim.x) {
        const int pa = i + rank_in(B, n_top, A[i], false);
        if (pa < n_top) o[pa] = A[i];
        const int pb = i + rank_in(A, n_top, B[i], true);
        if (pb < n_top) o[pb] = B[i];
    }
}

// fold_best[f] = index of the best training BA of fold f over the G block results
__global__ void mdr_fold_best_kernel(const MdrCand *__restrict__ fold_out, int64_t G, int nf, long long *__restrict__ fold_best) {
    const int f = threadIdx.x;
    if (f >= nf) return;
    double v = -INFINITY;
    long long i = LLONG_MAX;
    for (int64_t g = 0; g < G; ++g) {
        const MdrCand x = fold_out[g * nf + f];
        if (better(x.score, x.idx, v, i)) {
            v = x.score;
            i = x.idx;
        }
    }
    fold_best[f] = i;
}

// tables[(q * nseg + s) * 9 + va * 3 + vb] = samples of segment s in cell (va, vb) of combination q
// (order 1: vb = 0).  One thread per (combination, segment); the cells come from joint_visit.
__global__ void __launch_bounds__(128) mdr_tables_kernel(const uint32_t *__restrict__ planes, int64_t W,
                                                         const int32_t *__restrict__ marg, const int32_t *__restrict__ start,
                                                         MdrSeg seg, int nseg, const int64_t *__restrict__ combos, int order,
                                                         int64_t m, int64_t *__restrict__ tables) {
    const int64_t e = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= m * nseg) return;
    const int64_t q = e / nseg;
    const int s = (int)(e % nseg);
    const int64_t a = combos[q * order];
    const int ka = start[a], la = start[a + 1] - ka;
    int kb = 0, lb = 0;
    if (order == 2) {
        const int64_t b = combos[q * 2 + 1];
        kb = start[b];
        lb = start[b + 1] - kb;
    }
    int32_t ma[2] = {0, 0}, mb[2] = {0, 0};
    for (int i = 0; i < la; ++i) ma[i] = marg[(int64_t)(ka + i) * nseg + s];
    for (int j = 0; j < lb; ++j) mb[j] = marg[(int64_t)(kb + j) * nseg + s];
    int32_t cc[2][2] = {{0, 0}, {0, 0}};
    for (int i = 0; i < la; ++i)
        for (int j = 0; j < lb; ++j) {
            const uint32_t *ra = planes + (int64_t)(ka + i) * W, *rb = planes + (int64_t)(kb + j) * W;
            int32_t v = 0;
            for (int w = seg.w[s]; w < seg.w[s + 1]; ++w) v += __popc(ra[w] & rb[w]);
            cc[i][j] = v;
        }
    JointSums js;
    auto cnt = [&](int i, int j) { return cc[i][j]; };
    joint_sums(la, lb, ma, mb, cnt, js);
    int64_t *t = tables + e * 9;
    for (int g = 0; g < 9; ++g) t[g] = 0;
    joint_visit(la, lb, ma, mb, cnt, (int64_t)seg.n[s], js,
                [&](int i, int j, int64_t nij, int64_t, int64_t) { t[i * 3 + j] = nij; });
}

// Encode (the shared discrete operand) + pack of (feat_idx, fold); the planes are kept for the operand's
// generation and the folds.
// `what` names the caller in error messages.
void mdr_prepare(fs_dataset *ds, const int64_t *feat_idx, int64_t n_kept, const int32_t *fold, int n_folds, int *launches,
                 const char *what = "mdr") {
    FS_REQUIRE(ds->n_classes == 2, FS_ERR_INVALID, "%s: the data set must have 2 classes (has %d)", what, ds->n_classes);
    const int64_t n = ds->n;
    // balanced accuracies are ratios of integers below 2^53 (2 N1 N0 < 2^53); KSA products of two counts too
    FS_REQUIRE(n < (1LL << 26), FS_ERR_INVALID, "%s: n = %lld exceeds 2^26 samples", what, (long long)n);
    const DiscreteOperand &op = discrete_operand(ds, feat_idx, n_kept, 3, what, false, launches);
    const int nseg = 2 * n_folds;
    std::vector<int64_t> key(1 + n);
    key[0] = n_folds;
    std::copy(fold, fold + n, key.begin() + 1);
    if (ds->mdr_gen == op.generation && ds->mdr_key == key) return;
    ds->mdr_gen = 0;
    cudaStream_t st = ds->stream;

    // segments: s = 2 * fold + class, each padded to whole words; slots filled in internal row order
    std::vector<int64_t> seg_n(nseg, 0);
    for (int64_t r = 0; r < n; ++r) {
        const int32_t f = fold[ds->perm[r]];
        FS_REQUIRE(f >= 0 && f < n_folds, FS_ERR_INVALID, "%s: fold[%lld] = %d outside [0, %d)", what,
                   (long long)ds->perm[r], f, n_folds);
        ++seg_n[2 * f + ds->y_sorted[r]];
    }
    MdrSeg &seg = ds->mdr_seg;
    seg.w[0] = 0;
    for (int s = 0; s < nseg; ++s) {
        FS_REQUIRE(seg_n[s] > 0, FS_ERR_INVALID, "%s: fold %d has no sample of class %d", what, s / 2, s & 1);
        seg.n[s] = (int32_t)seg_n[s];
        seg.w[s + 1] = seg.w[s] + (int32_t)ceil_div(seg_n[s], 32);
    }
    const int64_t W = round_up(seg.w[nseg], 4);          // 16 B rows for the scan's staging loads
    for (int s = nseg + 1; s <= kMdrMaxSegments; ++s) seg.w[s] = seg.w[nseg];
    std::vector<int32_t> slot(32 * W, -1);
    std::vector<uint8_t> wseg(W, (uint8_t)(nseg - 1));
    std::vector<int64_t> fill(nseg, 0);
    for (int s = 0; s < nseg; ++s)
        for (int32_t w = seg.w[s]; w < seg.w[s + 1]; ++w) wseg[w] = (uint8_t)s;
    for (int64_t r = 0; r < n; ++r) {
        const int s = 2 * fold[ds->perm[r]] + ds->y_sorted[r];
        slot[32 * (int64_t)seg.w[s] + fill[s]++] = (int32_t)r;
    }

    const WorkSet &ws = ds->ws;
    const int64_t K = ws.K_used;
    ds->mdr_slot.reserve(32 * W);
    ds->mdr_wseg.reserve(W);
    ds->mdr_planes.reserve((size_t)std::max<int64_t>(K, 1) * W);
    ds->mdr_marg.reserve((size_t)std::max<int64_t>(K, 1) * nseg);
    // pageable sources: each copy is staged before the call returns
    FS_CUDA(cudaMemcpyAsync(ds->mdr_slot.ptr, slot.data(), slot.size() * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    FS_CUDA(cudaMemcpyAsync(ds->mdr_wseg.ptr, wseg.data(), W, cudaMemcpyHostToDevice, st));
    FS_CUDA(cudaMemsetAsync(ds->mdr_marg.ptr, 0, (size_t)std::max<int64_t>(K, 1) * nseg * sizeof(int32_t), st));
    if (K > 0) {
        const int64_t groups = ceil_div(K, kMdrPackRows);
        dim3 grid((unsigned)ceil_div(W, 128), (unsigned)std::min<int64_t>(groups, 65535));
        mdr_pack_kernel<<<grid, 128, 0, st>>>(ws.At.ptr, ws.ldt / 2, K, ds->mdr_slot.ptr, ds->mdr_wseg.ptr, W, nseg,
                                              ds->mdr_planes.ptr, ds->mdr_marg.ptr);
        FS_CUDA(cudaGetLastError());
        ++*launches;
    }
    FS_CUDA(cudaStreamSynchronize(st));
    ds->mdr_W = W;
    ds->mdr_nseg = nseg;
    ds->mdr_key = std::move(key);
    ds->mdr_gen = op.generation;
}

template <int NSEG, bool PAIR, class Eval>
int64_t launch_scan_t(const MdrScanArgs &args, const MdrSeg &seg, int sms, int64_t max_blocks, cudaStream_t st) {
    auto kern = mdr_scan_kernel<NSEG, PAIR, Eval>;
    const size_t smem = mdr_smem_bytes(PAIR, args.n_top);
    FS_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    int per_sm = 0;
    FS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kMdrThreads, smem));
    FS_REQUIRE(per_sm >= 1, FS_ERR_INVALID, "mdr: the scan kernel does not fit an SM with n_top = %d", args.n_top);
    const int64_t G = std::max<int64_t>(1, std::min<int64_t>((int64_t)per_sm * sms, std::min(args.n_tiles, max_blocks)));
    kern<<<(unsigned)G, kMdrThreads, smem, st>>>(args, seg);
    FS_CUDA(cudaGetLastError());
    return G;
}

template <int NSEG>
int64_t launch_scan_n(bool pair, const MdrScanArgs &args, const MdrSeg &seg, int sms, int64_t max_blocks, cudaStream_t st) {
    return pair ? launch_scan_t<NSEG, true, MdrEval<NSEG>>(args, seg, sms, max_blocks, st)
                : launch_scan_t<NSEG, false, MdrEval<NSEG>>(args, seg, sms, max_blocks, st);
}

// MDR scan of order 1 or 2 over nseg = 2 n_folds segments
int64_t launch_scan(int nseg, bool pair, const MdrScanArgs &args, const MdrSeg &seg, int sms, int64_t max_blocks,
                    cudaStream_t st) {
    switch (nseg) {
    case 4: return launch_scan_n<4>(pair, args, seg, sms, max_blocks, st);
    case 6: return launch_scan_n<6>(pair, args, seg, sms, max_blocks, st);
    case 8: return launch_scan_n<8>(pair, args, seg, sms, max_blocks, st);
    case 10: return launch_scan_n<10>(pair, args, seg, sms, max_blocks, st);
    case 12: return launch_scan_n<12>(pair, args, seg, sms, max_blocks, st);
    case 14: return launch_scan_n<14>(pair, args, seg, sms, max_blocks, st);
    case 16: return launch_scan_n<16>(pair, args, seg, sms, max_blocks, st);
    case 18: return launch_scan_n<18>(pair, args, seg, sms, max_blocks, st);
    default: return launch_scan_n<20>(pair, args, seg, sms, max_blocks, st);
    }
}

int64_t mdr_combos(int64_t n_kept, int order) { return order == 1 ? n_kept : n_kept * (n_kept - 1) / 2; }

void check_common(fs_dataset *ds, int64_t n_kept, int order, const int32_t *fold, int n_folds) {
    FS_REQUIRE(ds && fold, FS_ERR_INVALID, "mdr: null pointer");
    FS_REQUIRE(order == 1 || order == 2, FS_ERR_INVALID, "mdr: order must be 1 or 2 (got %d)", order);
    FS_REQUIRE(n_kept >= order, FS_ERR_INVALID, "mdr: %lld columns cannot form a combination of order %d",
               (long long)n_kept, order);
    FS_REQUIRE(n_folds >= 2 && n_folds <= kMdrMaxFolds, FS_ERR_INVALID, "mdr: n_folds = %d outside [2, %d]", n_folds,
               kMdrMaxFolds);
}

// Scan of the prepared planes and the merges of the block lists (plus, for MDR, the fold-best reduction):
// ksa selects the evaluation policy.  all (device, nullable): [2, n_combos] for MDR, [n_combos] for KSA.
// Returns the merged list (device, n_top entries) and sets *blocks to the scan's grid.
MdrCand *run_scan(fs_dataset *ds, int64_t n_kept, int order, int64_t n_top, bool ksa, double *all, PhaseTimer &tm,
                  int *launches, int64_t *blocks) {
    cudaStream_t st = ds->stream;
    const int nseg = ds->mdr_nseg, n_folds = ksa ? 0 : nseg / 2;
    tm.begin(&fs_stats::ms_dist_general);
    int sms = 0;
    FS_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ds->device));
    MdrScanArgs args{};
    args.planes = ds->mdr_planes.ptr;
    args.marg = ds->mdr_marg.ptr;
    args.start = ds->disc.start.ptr;
    args.W = ds->mdr_W;
    args.n_kept = n_kept;
    args.n_top = (int)n_top;
    if (order == 2) {
        args.tiles_side = ceil_div(n_kept, kMdrTile);
        args.n_tiles = args.tiles_side * (args.tiles_side + 1) / 2;
    } else {
        args.tiles_side = 0;
        args.n_tiles = ceil_div(n_kept, kMdrThreads);
    }
    if (all) {
        args.all_train = ksa ? nullptr : all;
        args.all_test = ksa ? all : all + mdr_combos(n_kept, order);
    }
    // at most as many blocks as the SMs hold at once (persistent), and never more than there are tiles
    const int64_t max_blocks = 16LL * sms;
    ds->mdr_top.reserve(2 * (size_t)max_blocks * n_top * sizeof(MdrCand));
    ds->mdr_fold.reserve((size_t)max_blocks * std::max(n_folds, 1) * sizeof(MdrCand));
    ds->mdr_best.reserve(kMdrMaxFolds);
    args.top_out = reinterpret_cast<MdrCand *>(ds->mdr_top.ptr);
    args.fold_out = reinterpret_cast<MdrCand *>(ds->mdr_fold.ptr);
    static_assert(sizeof(MdrCand) == 24, "MdrCand layout");
    const int64_t G = ksa ? launch_scan_t<2, true, KsaEval>(args, ds->mdr_seg, sms, max_blocks, st)
                          : launch_scan(nseg, order == 2, args, ds->mdr_seg, sms, max_blocks, st);
    ++*launches;
    tm.end();
    tm.begin(&fs_stats::ms_reduce);
    MdrCand *cur = args.top_out, *nxt = cur + max_blocks * n_top;
    for (int64_t L = G; L > 1; L = ceil_div(L, 2)) {
        mdr_merge_kernel<<<(unsigned)ceil_div(L, 2), 256, 0, st>>>(cur, L, (int)n_top, nxt);
        FS_CUDA(cudaGetLastError());
        ++*launches;
        std::swap(cur, nxt);
    }
    if (!ksa) {
        mdr_fold_best_kernel<<<1, 32, 0, st>>>(args.fold_out, G, n_folds, ds->mdr_best.ptr);
        FS_CUDA(cudaGetLastError());
        ++*launches;
    }
    tm.end();
    *blocks = G;
    return cur;
}

void scan_stats(fs_stats *stats, PhaseTimer &tm, int launches, int64_t G, const fs_dataset *ds, int64_t n_combos) {
    memset(stats, 0, sizeof(*stats));
    tm.finish(stats);
    stats->launches = launches;
    stats->n_chunks = (int32_t)G;
    stats->n_tensor_cols = ds->ws.pt;
    stats->onehot_k = ds->ws.K_used;
    stats->pairs_selected = n_combos;
}

// Positions (a, b) of the order-2 combination index idx over n positions: a from the quadratic, then exact
// integer fix-ups (the inverse of the scan's a * n - a (a + 1) / 2 + (b - a - 1)).
void decode_pair(int64_t idx, int64_t n, int64_t *a, int64_t *b) {
    auto off = [n](int64_t v) { return v * n - v * (v + 1) / 2; };
    const double q = 2.0 * (double)n - 1.0;
    int64_t v = (int64_t)std::floor((q - std::sqrt(std::max(q * q - 8.0 * (double)idx, 0.0))) * 0.5);
    v = std::min<int64_t>(std::max<int64_t>(v, 0), std::max<int64_t>(n - 2, 0));
    while (v > 0 && off(v) > idx) --v;
    while (v + 1 < n - 1 && off(v + 1) <= idx) ++v;
    *a = v;
    *b = idx - off(v) + v + 1;
}

}  // namespace
}  // namespace fs

using namespace fs;

extern "C" {

int fs_mdr_scan(fs_dataset *ds, const int64_t *feat_idx, int64_t n_kept, int32_t order, const int32_t *fold, int32_t n_folds,
                int64_t n_top, int64_t *top_idx, double *top_train, double *top_test, int64_t *fold_best,
                double *all_train, double *all_test, fs_stats *stats) {
    return api_call("fs_mdr_scan", [&] {
        if (ds && !feat_idx) n_kept = ds->p;
        check_common(ds, n_kept, order, fold, n_folds);
        FS_REQUIRE(top_idx && top_train && top_test && fold_best, FS_ERR_INVALID, "fs_mdr_scan: null output");
        FS_REQUIRE((all_train == nullptr) == (all_test == nullptr), FS_ERR_INVALID,
                   "fs_mdr_scan: all_train and all_test are both given or both null");
        const int64_t n_combos = mdr_combos(n_kept, order);
        FS_REQUIRE(n_top >= 1 && n_top <= std::min<int64_t>(FS_MDR_MAX_TOP, n_combos), FS_ERR_INVALID,
                   "fs_mdr_scan: n_top = %lld outside [1, min(%d, %lld combinations)]", (long long)n_top, FS_MDR_MAX_TOP,
                   (long long)n_combos);
        FS_CUDA(cudaSetDevice(ds->device));
        alloc_stream() = ds->stream;
        cudaStream_t st = ds->stream;
        int launches = 0;
        PhaseTimer tm(stats != nullptr, st);
        tm.begin(&fs_stats::ms_gather);
        mdr_prepare(ds, feat_idx, n_kept, fold, n_folds, &launches);
        tm.end();
        double *all = nullptr;
        if (all_train) {
            ds->mdr_all.reserve(2 * (size_t)n_combos);
            all = ds->mdr_all.ptr;
        }
        int64_t G = 0;
        const MdrCand *cur = run_scan(ds, n_kept, order, n_top, false, all, tm, &launches, &G);
        tm.stop();          // ms_total ends before the results are copied back
        std::vector<MdrCand> top(n_top);
        FS_CUDA(cudaMemcpyAsync(top.data(), cur, n_top * sizeof(MdrCand), cudaMemcpyDeviceToHost, st));
        FS_CUDA(cudaMemcpyAsync(fold_best, ds->mdr_best.ptr, n_folds * sizeof(long long), cudaMemcpyDeviceToHost, st));
        if (all_train) {
            FS_CUDA(cudaMemcpyAsync(all_train, all, n_combos * sizeof(double), cudaMemcpyDeviceToHost, st));
            FS_CUDA(cudaMemcpyAsync(all_test, all + n_combos, n_combos * sizeof(double), cudaMemcpyDeviceToHost, st));
        }
        FS_CUDA(cudaStreamSynchronize(st));
        for (int64_t i = 0; i < n_top; ++i) {
            top_idx[i] = top[i].idx;
            top_test[i] = top[i].score;
            top_train[i] = top[i].train;
        }
        if (stats) scan_stats(stats, tm, launches, G, ds, n_combos);
        return FS_OK;
    });
}

int fs_mdr_tables(fs_dataset *ds, const int64_t *feat_idx, int64_t n_kept, int32_t order, const int32_t *fold,
                  int32_t n_folds, const int64_t *combos, int64_t m, int64_t *tables_out) {
    return api_call("fs_mdr_tables", [&] {
        if (ds && !feat_idx) n_kept = ds->p;
        check_common(ds, n_kept, order, fold, n_folds);
        FS_REQUIRE(combos && tables_out && m >= 1, FS_ERR_INVALID, "fs_mdr_tables: invalid argument");
        for (int64_t q = 0; q < m; ++q) {
            const int64_t a = combos[q * order], b = order == 2 ? combos[q * 2 + 1] : -1;
            FS_REQUIRE(a >= 0 && a < n_kept && (order == 1 || (b >= 0 && b < n_kept && a != b)), FS_ERR_INVALID,
                       "fs_mdr_tables: combination %lld is not %d different positions below %lld", (long long)q, order,
                       (long long)n_kept);
        }
        FS_CUDA(cudaSetDevice(ds->device));
        alloc_stream() = ds->stream;
        cudaStream_t st = ds->stream;
        int launches = 0;
        mdr_prepare(ds, feat_idx, n_kept, fold, n_folds, &launches);
        const int nseg = ds->mdr_nseg;
        const size_t cells = (size_t)m * nseg * 9;
        ds->mdr_combos.reserve((size_t)m * order);
        ds->mdr_tables.reserve(cells);
        FS_CUDA(cudaMemcpyAsync(ds->mdr_combos.ptr, combos, (size_t)m * order * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        mdr_tables_kernel<<<(unsigned)ceil_div(m * nseg, 128), 128, 0, st>>>(ds->mdr_planes.ptr, ds->mdr_W, ds->mdr_marg.ptr,
                                                                             ds->disc.start.ptr, ds->mdr_seg, nseg,
                                                                             ds->mdr_combos.ptr, order, m, ds->mdr_tables.ptr);
        FS_CUDA(cudaGetLastError());
        FS_CUDA(cudaMemcpyAsync(tables_out, ds->mdr_tables.ptr, cells * sizeof(int64_t), cudaMemcpyDeviceToHost, st));
        FS_CUDA(cudaStreamSynchronize(st));
        return FS_OK;
    });
}

int fs_interaction_scan(fs_dataset *ds, const int64_t *feat_idx, int64_t n_kept, int64_t n_top, int64_t *top_idx,
                        double *top_ksa, int64_t *top_tables, double *all_ksa, fs_stats *stats) {
    return api_call("fs_interaction_scan", [&] {
        FS_REQUIRE(ds, FS_ERR_INVALID, "fs_interaction_scan: null data set");
        if (!feat_idx) n_kept = ds->p;
        FS_REQUIRE(top_idx && top_ksa && top_tables, FS_ERR_INVALID, "fs_interaction_scan: null output");
        FS_REQUIRE(n_kept >= 2, FS_ERR_INVALID, "fs_interaction_scan: %lld columns form no pair", (long long)n_kept);
        const int64_t n_pairs = mdr_combos(n_kept, 2);
        FS_REQUIRE(n_top >= 1 && n_top <= std::min<int64_t>(FS_MDR_MAX_TOP, n_pairs), FS_ERR_INVALID,
                   "fs_interaction_scan: n_top = %lld outside [1, min(%d, %lld pairs)]", (long long)n_top, FS_MDR_MAX_TOP,
                   (long long)n_pairs);
        FS_CUDA(cudaSetDevice(ds->device));
        alloc_stream() = ds->stream;
        cudaStream_t st = ds->stream;
        int launches = 0;
        PhaseTimer tm(stats != nullptr, st);
        tm.begin(&fs_stats::ms_gather);
        const std::vector<int32_t> fold(ds->n, 0);     // one fold: the segments are the two classes
        mdr_prepare(ds, feat_idx, n_kept, fold.data(), 1, &launches, "interaction");
        tm.end();
        double *all = nullptr;
        if (all_ksa) {
            ds->mdr_all.reserve((size_t)n_pairs);
            all = ds->mdr_all.ptr;
        }
        int64_t G = 0;
        const MdrCand *cur = run_scan(ds, n_kept, 2, n_top, true, all, tm, &launches, &G);
        tm.stop();          // ms_total ends before the results are copied back and the tables counted
        std::vector<MdrCand> top(n_top);
        FS_CUDA(cudaMemcpyAsync(top.data(), cur, n_top * sizeof(MdrCand), cudaMemcpyDeviceToHost, st));
        if (all_ksa) FS_CUDA(cudaMemcpyAsync(all_ksa, all, n_pairs * sizeof(double), cudaMemcpyDeviceToHost, st));
        FS_CUDA(cudaStreamSynchronize(st));
        std::vector<int64_t> pairs(2 * n_top);
        for (int64_t i = 0; i < n_top; ++i) {
            top_idx[i] = top[i].idx;
            top_ksa[i] = top[i].score;
            decode_pair(top[i].idx, n_kept, &pairs[2 * i], &pairs[2 * i + 1]);
        }
        ds->mdr_combos.reserve((size_t)n_top * 2);
        ds->mdr_tables.reserve((size_t)n_top * 2 * 9);
        FS_CUDA(cudaMemcpyAsync(ds->mdr_combos.ptr, pairs.data(), pairs.size() * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        mdr_tables_kernel<<<(unsigned)ceil_div(n_top * 2, 128), 128, 0, st>>>(ds->mdr_planes.ptr, ds->mdr_W, ds->mdr_marg.ptr,
                                                                              ds->disc.start.ptr, ds->mdr_seg, 2,
                                                                              ds->mdr_combos.ptr, 2, n_top, ds->mdr_tables.ptr);
        FS_CUDA(cudaGetLastError());
        ++launches;
        FS_CUDA(cudaMemcpyAsync(top_tables, ds->mdr_tables.ptr, (size_t)n_top * 2 * 9 * sizeof(int64_t),
                                cudaMemcpyDeviceToHost, st));
        FS_CUDA(cudaStreamSynchronize(st));
        if (stats) scan_stats(stats, tm, launches, G, ds, n_pairs);
        return FS_OK;
    });
}

}  // extern "C"
