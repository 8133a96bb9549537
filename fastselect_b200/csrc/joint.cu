// joint.cu -- joint-count path (SURVEY.md section 8(f)-4): pairwise contingency tables of discrete
// columns on the tensor cores, folded into mutual information or symmetrical uncertainty.
//
// Replaces _batch_mi_cpu / calculate_mi_matrices (mutual_information.py:49-63, :158-196; the reference
// leaves the p x p redundancy matrix to the CPU even with backend="gpu", :191-193) and CFS's
// _precompute_correlations_cpu / _precompute_correlations_gpu_kernel (CFS.py:81-104, :219-243: one
// thread per feature walking every sample of every other feature).
//
// Data flow (all on the data set's stream):
//   encode   the reduced one-hot rows At [K, n] of the columns -- the feature-major FP4 operand the
//            accumulation GEMM already uses (onehot.cu); a column with V values owns V - 1 rows.
//   marginals  popcount of every At row (HBM-bound, K * n / 2 bytes).
//   counts   C = At * At^T, contraction over the samples: the distance kernel of tc_dist.cu is
//            reused as it is (tcgen05 kind::mxf4, FP32 accumulators, exact below 2^24 samples) with
//            At as both operands and a zero s vector, so a band of C arrives NEGATED as int32 rows.
//            Only the upper triangle is needed: a band of rows [b0, b0 + R) is multiplied with the
//            rows b0 .. K only.  Tensor-pipe bound: 2 * K^2/2 * n operations for the whole matrix.
//   finish   one thread per column pair rebuilds the full V_a x V_b table from the reduced counts
//            and the marginals (joint_math.cuh) and writes the statistic to both triangles of the
//            p x p result.  Reads 4 * (V_a - 1)(V_b - 1) bytes per pair, writes 16.
// Bands bound the slab (FS_B200_JOINT_SLAB_MB, default 1024 MB) whatever K is.
// fs_joint_columns (bottom of the file) computes chosen rows of the same matrix from a CUDA-core count
// kernel instead of the GEMM, with the same encode, marginals and finishing arithmetic.
#include <algorithm>
#include <cstring>

#include "common.cuh"
#include "joint_math.cuh"

namespace fs {

namespace {

// marg[k] = number of samples carrying reduced row k: its 1.0 nibbles (0x2) in At.  One warp per row.
__global__ void __launch_bounds__(256) joint_marginals_kernel(const int8_t *__restrict__ At, int64_t pitch,
                                                              int64_t row_bytes, int64_t K, int32_t *__restrict__ marg) {
    const int64_t row = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5);
    const int lane = threadIdx.x & 31;
    if (row >= K) return;
    const uint8_t *r = reinterpret_cast<const uint8_t *>(At) + row * pitch;      // pitch: multiple of 64 bytes
    const int64_t vecs = row_bytes >> 4;
    int cnt = 0;
    for (int64_t w = lane; w < vecs; w += 32) {
        const uint4 q = reinterpret_cast<const uint4 *>(r)[w];
        cnt += __popc(q.x & 0x22222222u) + __popc(q.y & 0x22222222u) + __popc(q.z & 0x22222222u) + __popc(q.w & 0x22222222u);
    }
    for (int64_t b = (vecs << 4) + lane; b < row_bytes; b += 32) cnt += __popc((unsigned)r[b] & 0x22u);
#pragma unroll
    for (int o = 16; o >= 1; o >>= 1) cnt += __shfl_xor_sync(0xffffffffu, cnt, o);
    if (lane == 0) marg[row] = cnt;
}

}  // namespace

const DiscreteOperand &discrete_operand(fs_dataset *ds, const int64_t *feat_idx, int64_t n_kept, int max_values,
                                        const char *what, bool need_marg, int *launches) {
    FS_REQUIRE(ds->have_features, FS_ERR_STATE, "%s: call fs_dataset_set_features first", what);
    DiscreteOperand &op = ds->disc;
    const WorkSet &ws = ds->ws;
    std::vector<int64_t> key(1 + (feat_idx ? n_kept : 0));
    key[0] = feat_idx ? n_kept : -1;
    if (feat_idx) std::copy(feat_idx, feat_idx + n_kept, key.begin() + 1);
    // a list encoded for a laxer caller is checked again (and fails) below
    if (!(op.valid && ws.valid && ws.build_id == op.build_id && op.max_rows < max_values && op.key == key)) {
        // reduced rows of every position: V - 1 for a tensor-path column, none for a constant one
        std::vector<int32_t> start(n_kept + 1, 0);
        int max_rows = 0;
        for (int64_t c = 0; c < n_kept; ++c) {
            const int64_t f = feat_idx ? feat_idx[c] : c;
            FS_REQUIRE(f >= 0 && f < ds->p, FS_ERR_INVALID, "feat_idx[%lld]=%lld outside [0,%lld)", (long long)c,
                       (long long)f, (long long)ds->p);
            const unsigned ci = ds->col_info[f], path = ci & kColPathMask;
            const int rows = path == kColTensor ? (int)(ci >> 4) : 0;
            FS_REQUIRE((path == kColTensor && rows < max_values) || path == kColConst, FS_ERR_INVALID,
                       "%s: column %lld is not a discrete column with at most %d distinct values", what, (long long)f,
                       max_values);
            start[c + 1] = start[c] + rows;
            max_rows = std::max(max_rows, rows);
        }
        op.valid = false;
        build_lists(ds, feat_idx, n_kept, false, false);
        build_operands(ds, false, kDistNone, 0, ds->n, false, launches);
        FS_REQUIRE(ws.K_used == start[n_kept], FS_ERR_STATE, "%s: working set holds %lld reduced rows, expected %lld",
                   what, (long long)ws.K_used, (long long)start[n_kept]);
        op.start_h = std::move(start);
        op.start.reserve(n_kept + 1);
        FS_CUDA(cudaMemcpyAsync(op.start.ptr, op.start_h.data(), (n_kept + 1) * sizeof(int32_t), cudaMemcpyHostToDevice,
                                ds->stream));
        op.key = std::move(key);
        op.build_id = ws.build_id;
        op.max_rows = max_rows;
        op.have_marg = false;
        ++op.generation;
        op.valid = true;
    }
    if (need_marg && !op.have_marg) {
        const int64_t K = ws.K_used;
        op.marg.reserve(std::max<int64_t>(K, 1));
        if (K > 0) {
            joint_marginals_kernel<<<(unsigned)ceil_div(K, 8), 256, 0, ds->stream>>>(ws.At.ptr, ws.ldt / 2, (ds->n + 1) / 2,
                                                                                      K, op.marg.ptr);
            FS_CUDA(cudaGetLastError());
            ++*launches;
        }
        op.have_marg = true;
    }
    return op;
}

namespace {

// out[c, g] = out[g, c] = statistic of the columns at positions c in [c_lo, c_hi) and g in (c, n_kept).
// start[c] .. start[c + 1]: reduced rows of position c (an empty range for a constant column);
// D: the band's negated counts, its row 0 / column 0 being reduced row b0.
__global__ void __launch_bounds__(256) joint_finish_kernel(const int32_t *__restrict__ D, int64_t ldd, int64_t b0,
                                                           const int32_t *__restrict__ start, int64_t c_lo, int64_t c_hi,
                                                           int64_t n_kept, const int32_t *__restrict__ marg, int64_t n,
                                                           int kind, double log_base, double *__restrict__ out) {
    const int64_t g = c_lo + 1 + (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_kept) return;
    const int sg = start[g], lg = start[g + 1] - sg;
    for (int64_t c = c_lo + blockIdx.y; c < c_hi && c < g; c += gridDim.y) {
        const int sc = start[c], lc = start[c + 1] - sc;
        const double v = joint_pair_from_slab(D, ldd, sc - b0, sg - b0, lc, lg, marg + sc, marg + sg, n, kind, log_base);
        out[c * n_kept + g] = v;
        out[g * n_kept + c] = v;
    }
}

// Parity/debug view: full tables of the requested pairs whose smaller position lies in [c_lo, c_hi).
// tables[q * 256 + va * 16 + vb] with (a, b) in the caller's order.
__global__ void __launch_bounds__(128) joint_tables_kernel(const int32_t *__restrict__ D, int64_t ldd, int64_t b0,
                                                           const int32_t *__restrict__ start, int64_t c_lo, int64_t c_hi,
                                                           const int32_t *__restrict__ marg, int64_t n,
                                                           const int64_t *__restrict__ pairs, int64_t m,
                                                           int64_t *__restrict__ tables) {
    const int64_t q = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (q >= m) return;
    const int64_t a = pairs[2 * q], b = pairs[2 * q + 1];
    const int64_t c = a < b ? a : b, g = a < b ? b : a;
    if (c < c_lo || c >= c_hi) return;
    const int sc = start[c], lc = start[c + 1] - sc, sg = start[g], lg = start[g + 1] - sg;
    const int64_t ra = sc - b0, cb = sg - b0;
    auto cnt = [=](int i, int j) { return -D[(ra + i) * ldd + cb + j]; };
    JointSums s;
    joint_sums(lc, lg, marg + sc, marg + sg, cnt, s);
    int64_t *t = tables + q * 256;
    const bool swapped = a > b;
    joint_visit(lc, lg, marg + sc, marg + sg, cnt, n, s, [&](int i, int j, int64_t nij, int64_t, int64_t) {
        t[swapped ? j * 16 + i : i * 16 + j] = nij;
    });
}

// The GEMM bands shared by fs_joint_matrix (kind >= 0, d_out) and fs_joint_tables (d_pairs / d_tables).
void run_joint(fs_dataset *ds, int kind, double log_base, const int64_t *feat_idx, int64_t n_kept, int64_t pos_begin,
               int64_t pos_end, double *d_out, const int64_t *d_pairs, int64_t m, int64_t *d_tables, fs_stats *stats) {
    FS_REQUIRE(n_kept >= 1 && pos_begin >= 0 && pos_begin <= pos_end && pos_end <= n_kept, FS_ERR_INVALID,
               "joint counts: bad position range [%lld, %lld) of %lld columns", (long long)pos_begin, (long long)pos_end,
               (long long)n_kept);
    // FP32 accumulators hold the counts exactly below 2^24 samples
    FS_REQUIRE(ds->n < (1LL << 24), FS_ERR_INVALID, "joint counts: n = %lld exceeds the exact range (2^24)", (long long)ds->n);
    const int64_t n = ds->n;
    cudaStream_t st = ds->stream;
    int launches = 0;
    double ops = 0.0;
    PhaseTimer tm(stats != nullptr, st);
    tm.begin(&fs_stats::ms_gather);
    const DiscreteOperand &op = discrete_operand(ds, feat_idx, n_kept, FS_DISTINCT_CAP, "joint counts", true, &launches);
    const std::vector<int32_t> &start = op.start_h;
    const WorkSet &ws = ds->ws;
    const int64_t K = ws.K_used;
    const int64_t row_bytes = (n + 1) / 2, pitch = ws.ldt / 2;     // At: two samples per byte
    tm.end();

    // the reused distance kernel adds s_i + s_j: zeros here, for the band's rows (from 0) and columns
    const int64_t zero_len = round_up(std::max<int64_t>(K, 1), 256) + 256;
    ds->joint_zero.reserve(zero_len);
    FS_CUDA(cudaMemsetAsync(ds->joint_zero.ptr, 0, zero_len * sizeof(int32_t), st));
    const char *env = getenv("FS_B200_JOINT_SLAB_MB");
    const int64_t budget = std::max<int64_t>(1, env ? atoll(env) : 1024) << 20;
    const int64_t k_bytes = round_up(row_bytes, 128);              // contraction length walked by the kernel (TMA zero-fills)
    int64_t c_lo = pos_begin;
    int bands = 0;
    while (c_lo < pos_end) {
        ++bands;
        const int64_t b0 = start[c_lo], ncols = K - b0;
        int64_t c_hi = pos_end, R = 0, ldd = 128;
        if (ncols > 0) {
            ldd = round_up(ncols, 128);
            const int64_t max_rows = std::max<int64_t>(128, budget / (4 * ldd) / 128 * 128);
            c_hi = c_lo + 1;
            while (c_hi < pos_end && start[c_hi + 1] - b0 <= max_rows) ++c_hi;
            R = start[c_hi] - b0;
        }
        if (R > 0) {
            tm.begin(&fs_stats::ms_dist_tensor);
            ds->joint_slab.reserve((size_t)round_up(R, 128) * ldd);
            const int8_t *base = ws.At.ptr + (size_t)b0 * pitch;
            launch_tc_dist(base, base, row_bytes, pitch, k_bytes, ds->joint_zero.ptr, 0, R, ncols, ldd, false,
                           false, single_rank_peers(ds->joint_slab.ptr, ncols), st, &launches, &ops);
            tm.end();
        }
        tm.begin(&fs_stats::ms_reduce);
        if (d_out && c_lo + 1 < n_kept) {
            dim3 grid((unsigned)ceil_div(n_kept - c_lo - 1, 256), (unsigned)std::min<int64_t>(c_hi - c_lo, 4096));
            joint_finish_kernel<<<grid, 256, 0, st>>>(ds->joint_slab.ptr, ldd, b0, op.start.ptr, c_lo, c_hi, n_kept,
                                                      op.marg.ptr, n, kind, log_base, d_out);
            FS_CUDA(cudaGetLastError());
            ++launches;
        }
        if (d_tables && m > 0) {
            joint_tables_kernel<<<(unsigned)ceil_div(m, 128), 128, 0, st>>>(ds->joint_slab.ptr, ldd, b0, op.start.ptr,
                                                                            c_lo, c_hi, op.marg.ptr, n, d_pairs, m,
                                                                            d_tables);
            FS_CUDA(cudaGetLastError());
            ++launches;
        }
        tm.end();
        c_lo = c_hi;
    }
    FS_CUDA(cudaStreamSynchronize(st));
    if (stats) {
        memset(stats, 0, sizeof(*stats));
        tm.finish(stats);
        stats->launches = launches;
        stats->n_chunks = bands;
        stats->n_tensor_cols = ws.pt;
        stats->onehot_k = K;
        stats->ops_dist_tensor = ops;
    }
}

// ---------------------------------------------------------------------------------------------------
// Column path (fs_joint_columns): the statistic of a few positions against every position, for greedy
// searches that read one column of the p x p matrix per step.  Counts come from the CUDA cores instead of
// the GEMM: c(s, r) = #samples whose nibble is 0x2 in both selected reduced row s and At row r, one pass
// over At per launch of up to kColsMaxSel selected rows -- K * ceil(n / 2) bytes, HBM-bound for 0/1/2
// genotypes (two selected rows per position).  The finishing step is joint_statistic with the same
// operand order (smaller position first) and the same marginals as joint_finish_kernel, so a row of the
// result is bitwise the matching row of fs_joint_matrix.
constexpr int kColsMaxSel = 16;                     // selected reduced rows per count launch (>= 15: one position)
constexpr int kColsVecs = 4;                        // 16-byte At vectors per lane and sample chunk
constexpr int kColsChunkVecs = 32 * kColsVecs;      // sample chunk of one block: 128 vectors = 4096 samples

struct ColsSel {
    int32_t row[kColsMaxSel];                       // At rows of the selected reduced rows
};

// The 0x2 bit of every nibble of a 16-byte At vector (32 samples) -> one bit per sample.  The bit order is
// a fixed permutation of the samples, the same for every row, which is all the AND + POPC below needs.
__device__ __forceinline__ uint32_t fold_ones(const uint4 q) {
    return ((q.x >> 1) & 0x11111111u) | (q.y & 0x22222222u) | ((q.z << 1) & 0x44444444u) | ((q.w << 2) & 0x88888888u);
}

__device__ __forceinline__ uint32_t keep_bytes(uint32_t w, int64_t nb) {
    return nb >= 4 ? w : nb <= 0 ? 0u : w & ((1u << (8 * nb)) - 1u);
}

// counts[s * K + r] += c(s, r) over the samples of chunk blockIdx.y (counts zeroed by the caller; integer
// atomics, so the result does not depend on the order of the chunks).  The selected rows' masks of the chunk
// sit in shared memory with the bytes past row_bytes cleared: the pitch padding of At is never trusted, the
// AND removes it from the streamed rows.  One warp per At row: lane l reads vectors l, l + 32, ... of the
// chunk (512 contiguous bytes per instruction), and one warp reduction per selected row ends the row.
template <int S>
__global__ void __launch_bounds__(256) joint_cols_count_kernel(const int8_t *__restrict__ At, int64_t pitch,
                                                               int64_t row_bytes, int64_t K, ColsSel sel, int n_sel,
                                                               int32_t *__restrict__ counts) {
    __shared__ uint32_t sm[S][kColsChunkVecs];
    const uint8_t *base = reinterpret_cast<const uint8_t *>(At);
    const int64_t nvec = (row_bytes + 15) >> 4;
    const int64_t v0 = (int64_t)blockIdx.y * kColsChunkVecs;
    for (int t = threadIdx.x; t < S * kColsChunkVecs; t += blockDim.x) {
        const int s = t / kColsChunkVecs, w = t % kColsChunkVecs;
        const int64_t v = v0 + w;
        uint32_t m = 0;
        if (s < n_sel && v < nvec) {
            uint4 q = reinterpret_cast<const uint4 *>(base + (int64_t)sel.row[s] * pitch)[v];
            const int64_t nb = row_bytes - 16 * v;   // bytes of this vector inside the row (pitch: multiple of 64)
            q.x = keep_bytes(q.x, nb);
            q.y = keep_bytes(q.y, nb - 4);
            q.z = keep_bytes(q.z, nb - 8);
            q.w = keep_bytes(q.w, nb - 12);
            m = fold_ones(q);
        }
        sm[s][w] = m;
    }
    __syncthreads();
    const int lane = threadIdx.x & 31;
    for (int64_t r = (int64_t)blockIdx.x * 8 + (threadIdx.x >> 5); r < K; r += (int64_t)gridDim.x * 8) {
        const uint4 *row = reinterpret_cast<const uint4 *>(base + r * pitch);
        uint4 q[kColsVecs];
#pragma unroll
        for (int j = 0; j < kColsVecs; ++j) {
            const int64_t v = v0 + 32 * j + lane;
            q[j] = v < nvec ? __ldg(row + v) : make_uint4(0u, 0u, 0u, 0u);
        }
        uint32_t c[S];
#pragma unroll
        for (int s = 0; s < S; ++s) c[s] = 0;
#pragma unroll
        for (int j = 0; j < kColsVecs; ++j) {
            const uint32_t m = fold_ones(q[j]);
#pragma unroll
            for (int s = 0; s < S; ++s) c[s] += __popc(m & sm[s][32 * j + lane]);
        }
#pragma unroll
        for (int s = 0; s < S; ++s) {
            const uint32_t tot = __reduce_add_sync(0xffffffffu, c[s]);
            if (lane == s && s < n_sel && tot) atomicAdd(counts + s * K + r, (int32_t)tot);
        }
    }
}

// out[i * n_kept + g] = statistic(positions[i], g) for the positions [i0, i0 + gridDim.y) of one count launch;
// counts row off[i] + k holds reduced row k of positions[i] against every At row.
__global__ void __launch_bounds__(256) joint_cols_finish_kernel(const int32_t *__restrict__ counts, int64_t K,
                                                                const int32_t *__restrict__ start,
                                                                const int32_t *__restrict__ marg, int64_t n_kept,
                                                                const int64_t *__restrict__ positions,
                                                                const int32_t *__restrict__ off, int64_t i0, int64_t n,
                                                                int kind, double log_base, double *__restrict__ out) {
    const int64_t g = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (g >= n_kept) return;
    const int64_t i = i0 + blockIdx.y, c = positions[i];
    double v = 0.0;
    if (g != c) {
        const int sc = start[c], lc = start[c + 1] - sc, sg = start[g], lg = start[g + 1] - sg;
        const int32_t *C = counts + (int64_t)off[i] * K + sg;
        // the smaller position is the first operand, as in joint_finish_kernel (joint_visit walks the cells
        // in operand order, which fixes the float64 summation order)
        if (c < g)
            v = joint_statistic(kind, lc, lg, marg + sc, marg + sg, [=](int a, int b) { return C[a * K + b]; }, n, log_base);
        else
            v = joint_statistic(kind, lg, lc, marg + sg, marg + sc, [=](int a, int b) { return C[b * K + a]; }, n, log_base);
    }
    out[i * n_kept + g] = v;
}

template <int S>
void launch_cols_count(const int8_t *At, int64_t pitch, int64_t row_bytes, int64_t K, const ColsSel &sel, int n_sel,
                       int32_t *counts, int sms, cudaStream_t st) {
    const int64_t chunks = ceil_div(ceil_div(row_bytes, 16), kColsChunkVecs);
    // enough blocks for every SM several times over; each block walks many rows so that staging the
    // selected rows' chunk (an L2 hit) stays small next to the At bytes it streams
    const int64_t bx = std::max<int64_t>(1, std::min<int64_t>(ceil_div(K, 8), ceil_div((int64_t)sms * 16, chunks)));
    joint_cols_count_kernel<S><<<dim3((unsigned)bx, (unsigned)chunks), 256, 0, st>>>(At, pitch, row_bytes, K, sel, n_sel, counts);
}

void run_joint_columns(fs_dataset *ds, int kind, double log_base, const int64_t *feat_idx, int64_t n_kept,
                       const int64_t *positions, int64_t n_pos, double *d_out, fs_stats *stats) {
    const int64_t n = ds->n;
    const int64_t row_bytes = (n + 1) / 2;
    FS_REQUIRE(ceil_div(ceil_div(row_bytes, 16), kColsChunkVecs) <= 65535, FS_ERR_INVALID,
               "joint columns: n = %lld exceeds the sample range of the count kernel", (long long)n);
    cudaStream_t st = ds->stream;
    int launches = 0;
    PhaseTimer tm(stats != nullptr, st);
    tm.begin(&fs_stats::ms_gather);
    const DiscreteOperand &op = discrete_operand(ds, feat_idx, n_kept, FS_DISTINCT_CAP, "joint counts", true, &launches);
    tm.end();
    const std::vector<int32_t> &start = op.start_h;
    const WorkSet &ws = ds->ws;
    const int64_t K = ws.K_used, pitch = ws.ldt / 2;

    // launches: consecutive runs of positions with at most kColsMaxSel reduced rows together
    std::vector<int32_t> off(n_pos);
    std::vector<int64_t> cuts{0};
    for (int64_t i = 0, rows = 0; i < n_pos; ++i) {
        const int l = start[positions[i] + 1] - start[positions[i]];
        if (rows + l > kColsMaxSel) {
            cuts.push_back(i);
            rows = 0;
        }
        off[i] = (int32_t)rows;
        rows += l;
    }
    cuts.push_back(n_pos);
    ds->jc_pos.reserve(n_pos);
    ds->jc_off.reserve(n_pos);
    FS_CUDA(cudaMemcpyAsync(ds->jc_pos.ptr, positions, n_pos * sizeof(int64_t), cudaMemcpyHostToDevice, st));
    FS_CUDA(cudaMemcpyAsync(ds->jc_off.ptr, off.data(), n_pos * sizeof(int32_t), cudaMemcpyHostToDevice, st));
    ds->jc_counts.reserve((size_t)kColsMaxSel * std::max<int64_t>(K, 1));
    int sms = 0;
    FS_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, ds->device));
    for (size_t q = 0; q + 1 < cuts.size(); ++q) {
        const int64_t i0 = cuts[q], i1 = cuts[q + 1];
        ColsSel sel{};
        int n_sel = 0;
        for (int64_t i = i0; i < i1; ++i)
            for (int k = start[positions[i]]; k < start[positions[i] + 1]; ++k) sel.row[n_sel++] = k;
        if (n_sel > 0) {
            tm.begin(&fs_stats::ms_dist_general);
            FS_CUDA(cudaMemsetAsync(ds->jc_counts.ptr, 0, (size_t)n_sel * K * sizeof(int32_t), st));
            int32_t *cnt = ds->jc_counts.ptr;
            if (n_sel <= 1) launch_cols_count<1>(ws.At.ptr, pitch, row_bytes, K, sel, n_sel, cnt, sms, st);
            else if (n_sel <= 2) launch_cols_count<2>(ws.At.ptr, pitch, row_bytes, K, sel, n_sel, cnt, sms, st);
            else if (n_sel <= 4) launch_cols_count<4>(ws.At.ptr, pitch, row_bytes, K, sel, n_sel, cnt, sms, st);
            else if (n_sel <= 8) launch_cols_count<8>(ws.At.ptr, pitch, row_bytes, K, sel, n_sel, cnt, sms, st);
            else launch_cols_count<16>(ws.At.ptr, pitch, row_bytes, K, sel, n_sel, cnt, sms, st);
            FS_CUDA(cudaGetLastError());
            ++launches;
            tm.end();
        }
        tm.begin(&fs_stats::ms_reduce);
        dim3 grid((unsigned)ceil_div(n_kept, 256), (unsigned)(i1 - i0));
        joint_cols_finish_kernel<<<grid, 256, 0, st>>>(ds->jc_counts.ptr, K, op.start.ptr, op.marg.ptr, n_kept,
                                                       ds->jc_pos.ptr, ds->jc_off.ptr, i0, n, kind, log_base, d_out);
        FS_CUDA(cudaGetLastError());
        ++launches;
        tm.end();
    }
    // `positions`, `off` (pageable) were sources of asynchronous copies
    FS_CUDA(cudaStreamSynchronize(st));
    if (stats) {
        memset(stats, 0, sizeof(*stats));
        tm.finish(stats);
        stats->launches = launches;
        stats->n_chunks = (int32_t)(cuts.size() - 1);
        stats->n_tensor_cols = ws.pt;
        stats->onehot_k = K;
    }
}

}  // namespace
}  // namespace fs

using namespace fs;

extern "C" {

int fs_joint_matrix(fs_dataset *ds, int kind, double log_base, const int64_t *feat_idx, int64_t n_kept,
                    int64_t pos_begin, int64_t pos_end, double *out, int out_on_device, fs_stats *stats) {
    return api_call("fs_joint_matrix", [&] {
        FS_REQUIRE(ds && out, FS_ERR_INVALID, "fs_joint_matrix: null pointer");
        FS_REQUIRE(kind == FS_JOINT_MI || kind == FS_JOINT_SU, FS_ERR_INVALID, "fs_joint_matrix: unknown kind %d", kind);
        FS_REQUIRE(kind != FS_JOINT_MI || log_base > 0.0, FS_ERR_INVALID, "fs_joint_matrix: log_base must be positive");
        if (!feat_idx) n_kept = ds->p;
        FS_REQUIRE(n_kept >= 1, FS_ERR_INVALID, "fs_joint_matrix: no columns");
        FS_CUDA(cudaSetDevice(ds->device));
        alloc_stream() = ds->stream;
        double *d_out = out;
        const size_t cells = (size_t)n_kept * (size_t)n_kept;
        if (!out_on_device) {
            ds->joint_out.reserve(cells);
            d_out = ds->joint_out.ptr;
        }
        FS_CUDA(cudaMemsetAsync(d_out, 0, cells * sizeof(double), ds->stream));
        run_joint(ds, kind, log_base, feat_idx, n_kept, pos_begin, pos_end, d_out, nullptr, 0, nullptr, stats);
        if (!out_on_device) {
            FS_CUDA(cudaMemcpyAsync(out, d_out, cells * sizeof(double), cudaMemcpyDeviceToHost, ds->stream));
            FS_CUDA(cudaStreamSynchronize(ds->stream));
        }
        return FS_OK;
    });
}

int fs_joint_tables(fs_dataset *ds, const int64_t *feat_idx, int64_t n_kept, const int64_t *pairs, int64_t m,
                    int64_t *tables_out) {
    return api_call("fs_joint_tables", [&] {
        FS_REQUIRE(ds && pairs && tables_out && m >= 1, FS_ERR_INVALID, "fs_joint_tables: invalid argument");
        if (!feat_idx) n_kept = ds->p;
        for (int64_t q = 0; q < m; ++q)
            FS_REQUIRE(pairs[2 * q] >= 0 && pairs[2 * q] < n_kept && pairs[2 * q + 1] >= 0 && pairs[2 * q + 1] < n_kept &&
                           pairs[2 * q] != pairs[2 * q + 1],
                       FS_ERR_INVALID, "fs_joint_tables: pair %lld = (%lld, %lld) is not two different positions below %lld",
                       (long long)q, (long long)pairs[2 * q], (long long)pairs[2 * q + 1], (long long)n_kept);
        FS_CUDA(cudaSetDevice(ds->device));
        alloc_stream() = ds->stream;
        ds->joint_pairs.reserve(2 * m);
        ds->joint_tables.reserve(256 * m);
        FS_CUDA(cudaMemcpyAsync(ds->joint_pairs.ptr, pairs, 2 * m * sizeof(int64_t), cudaMemcpyHostToDevice, ds->stream));
        FS_CUDA(cudaMemsetAsync(ds->joint_tables.ptr, 0, 256 * m * sizeof(int64_t), ds->stream));
        run_joint(ds, -1, 1.0, feat_idx, n_kept, 0, n_kept, nullptr, ds->joint_pairs.ptr, m, ds->joint_tables.ptr, nullptr);
        FS_CUDA(cudaMemcpyAsync(tables_out, ds->joint_tables.ptr, 256 * m * sizeof(int64_t), cudaMemcpyDeviceToHost, ds->stream));
        FS_CUDA(cudaStreamSynchronize(ds->stream));
        return FS_OK;
    });
}

int fs_joint_columns(fs_dataset *ds, int kind, double log_base, const int64_t *feat_idx, int64_t n_kept,
                     const int64_t *positions, int64_t n_pos, double *out, int out_on_device, fs_stats *stats) {
    return api_call("fs_joint_columns", [&] {
        FS_REQUIRE(ds && out && positions, FS_ERR_INVALID, "fs_joint_columns: null pointer");
        FS_REQUIRE(kind == FS_JOINT_MI || kind == FS_JOINT_SU, FS_ERR_INVALID, "fs_joint_columns: unknown kind %d", kind);
        FS_REQUIRE(kind != FS_JOINT_MI || log_base > 0.0, FS_ERR_INVALID, "fs_joint_columns: log_base must be positive");
        if (!feat_idx) n_kept = ds->p;
        FS_REQUIRE(n_kept >= 1, FS_ERR_INVALID, "fs_joint_columns: no columns");
        FS_REQUIRE(n_pos >= 1, FS_ERR_INVALID, "fs_joint_columns: no positions");
        for (int64_t i = 0; i < n_pos; ++i)
            FS_REQUIRE(positions[i] >= 0 && positions[i] < n_kept, FS_ERR_INVALID,
                       "fs_joint_columns: position %lld = %lld outside [0, %lld)", (long long)i, (long long)positions[i],
                       (long long)n_kept);
        FS_CUDA(cudaSetDevice(ds->device));
        alloc_stream() = ds->stream;
        double *d_out = out;
        const size_t cells = (size_t)n_pos * (size_t)n_kept;
        if (!out_on_device) {
            ds->jc_out.reserve(cells);
            d_out = ds->jc_out.ptr;
        }
        run_joint_columns(ds, kind, log_base, feat_idx, n_kept, positions, n_pos, d_out, stats);
        if (!out_on_device) {
            FS_CUDA(cudaMemcpyAsync(out, d_out, cells * sizeof(double), cudaMemcpyDeviceToHost, ds->stream));
            FS_CUDA(cudaStreamSynchronize(ds->stream));
        }
        return FS_OK;
    });
}

}  // extern "C"
