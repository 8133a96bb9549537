// common.cuh -- shared declarations of libfastselect_b200 (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <chrono>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <exception>
#include <memory>
#include <string>
#include <vector>

#include "../../include/fastselect_b200.h"

namespace fs {

// ---------------------------------------------------------------------------
// errors: thread-local message + status codes (no exceptions cross the C ABI)
// ---------------------------------------------------------------------------
void set_error(const char *fmt, ...);
const char *get_error();

struct Fail {
    int code;
};

#define FS_CUDA(expr)                                                                       \
    do {                                                                                    \
        cudaError_t _e = (expr);                                                            \
        if (_e != cudaSuccess) {                                                            \
            fs::set_error("%s failed at %s:%d: %s", #expr, __FILE__, __LINE__,              \
                          cudaGetErrorString(_e));                                          \
            throw fs::Fail{_e == cudaErrorMemoryAllocation ? FS_ERR_OOM : FS_ERR_CUDA};     \
        }                                                                                   \
    } while (0)

#define FS_REQUIRE(cond, code, ...)          \
    do {                                     \
        if (!(cond)) {                       \
            fs::set_error(__VA_ARGS__);      \
            throw fs::Fail{code};            \
        }                                    \
    } while (0)

// Body of a C-ABI entry point: a Fail returns its code, any other exception (std::bad_alloc from a host
// container, ...) sets "<name>: <what>" and returns FS_ERR_OOM.  Nothing crosses the C ABI.
template <class F>
int api_call(const char *name, F &&body) noexcept {
    try {
        return body();
    } catch (const Fail &f) {
        return f.code;
    } catch (const std::exception &e) {
        set_error("%s: %s", name, e.what());
        return FS_ERR_OOM;
    }
}

// Stream used by DevBuf allocations of the current API call (set at every C-ABI entry).
cudaStream_t &alloc_stream();
void configure_pool(int device);

// Device buffer with RAII; never copies.  Memory comes from the device's stream-ordered
// pool (cudaMallocAsync) whose release threshold is raised so that freed blocks stay
// cached: a fit re-uses the previous fit's allocations instead of paying cudaMalloc /
// cudaFree for gigabyte-sized operands.
template <typename T>
struct DevBuf {
    T *ptr = nullptr;
    size_t count = 0;
    cudaStream_t st = nullptr;
    DevBuf() = default;
    DevBuf(const DevBuf &) = delete;
    DevBuf &operator=(const DevBuf &) = delete;
    ~DevBuf() { release(); }
    void release() {
        if (ptr) cudaFreeAsync(ptr, st);
        ptr = nullptr;
        count = 0;
    }
    void alloc(size_t n) {
        release();
        if (n == 0) return;
        st = alloc_stream();
        FS_CUDA(cudaMallocAsync(reinterpret_cast<void **>(&ptr), n * sizeof(T), st));
        count = n;
    }
    // grow-only (keeps the allocation when large enough)
    void reserve(size_t n) {
        if (n > count) alloc(n);
    }
};

// Pinned host staging buffer (grow-only): host->device copies of index arrays run at PCIe
// speed and are truly asynchronous.  Released blocks go to a process-wide free list instead of
// cudaFreeHost (page-locking costs milliseconds; every fit opens a new data set).
void *pinned_take(size_t bytes, size_t *got);
void pinned_give(void *ptr, size_t bytes);

template <typename T>
struct PinnedBuf {
    T *ptr = nullptr;
    size_t count = 0, bytes = 0;
    PinnedBuf() = default;
    PinnedBuf(const PinnedBuf &) = delete;
    PinnedBuf &operator=(const PinnedBuf &) = delete;
    ~PinnedBuf() {
        if (ptr) pinned_give(ptr, bytes);
    }
    void reserve(size_t n) {
        if (n <= count) return;
        if (ptr) pinned_give(ptr, bytes);
        ptr = nullptr;
        count = 0;
        ptr = static_cast<T *>(pinned_take(n * sizeof(T), &bytes));
        count = bytes / sizeof(T);
    }
};

// Device-time phases of one call (stats != nullptr only): begin(&fs_stats::ms_x) / end() record a span on the
// stream, and finish() adds every span into its field and sets ms_total from construction to stop() (or to
// finish() itself).  finish() adds: the caller zeroes *out first.
struct PhaseTimer {
    using Field = float fs_stats::*;
    struct Span { Field field; cudaEvent_t a, b; };
    bool on;
    cudaStream_t st;
    std::vector<Span> spans;
    cudaEvent_t t0 = nullptr, t1 = nullptr;
    bool stopped = false;
    PhaseTimer(bool enable, cudaStream_t s) : on(enable), st(s) {
        if (on) {
            cudaEventCreate(&t0);
            cudaEventCreate(&t1);
            cudaEventRecord(t0, st);
        }
    }
    void begin(Field f) {
        if (!on) return;
        Span s{f, nullptr, nullptr};
        cudaEventCreate(&s.a);
        cudaEventCreate(&s.b);
        cudaEventRecord(s.a, st);
        spans.push_back(s);
    }
    void end() {
        if (on) cudaEventRecord(spans.back().b, st);
    }
    void stop() {
        if (on && !stopped) cudaEventRecord(t1, st);
        stopped = true;
    }
    void finish(fs_stats *out) {
        if (!on) return;
        stop();
        cudaEventSynchronize(t1);
        for (auto &s : spans) {
            float t = 0.f;
            cudaEventElapsedTime(&t, s.a, s.b);
            out->*s.field += t;
        }
        cudaEventElapsedTime(&out->ms_total, t0, t1);
    }
    ~PhaseTimer() {
        for (auto &s : spans) {
            cudaEventDestroy(s.a);
            cudaEventDestroy(s.b);
        }
        if (t0) cudaEventDestroy(t0);
        if (t1) cudaEventDestroy(t1);
    }
};

// Host-side scope timer, printed to stderr when FS_B200_TRACE is set (debugging aid).
struct Trace {
    const char *name;
    std::chrono::steady_clock::time_point t0;
    bool on;
    explicit Trace(const char *nm) : name(nm), t0(std::chrono::steady_clock::now()), on(getenv("FS_B200_TRACE") != nullptr) {}
    ~Trace() {
        if (on)
            fprintf(stderr, "[fs trace] %-28s %8.3f ms\n", name,
                    std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count());
    }
};

static inline int64_t round_up(int64_t a, int64_t b) { return (a + b - 1) / b * b; }
static inline int64_t ceil_div(int64_t a, int64_t b) { return (a + b - 1) / b; }

// Feature chunk of the CUDA-core ("general") path: 128 bytes of one sample's
// features, i.e. 32 float32 or 16 float64 columns.  A chunk is either all
// continuous (type 0) or all "compare" columns (type 1: term = [a != b]).
constexpr int kChunkBytes = 128;
enum : uint8_t { kChunkContinuous = 0, kChunkCompare = 1 };

// Per-target-row result of the neighbour selection, consumed by the
// accumulation kernels.  coef[code] is the coefficient of a pair with
// neighbour code `code` (FS_MASK_*), already carrying the sign and the
// per-row 1/|H_i|, 1/|M_i| normalisation (MultiSURF.py:245-251).
struct RowInfo {
    double thresh;
    double coef[5];
    int32_t n_hit, n_miss, n_far_hit, n_far_miss;   // near hits, near misses, far hits, far misses
};

// Per-column path of the scoring pipeline (fs_dataset::col_info): bits 0-1 the path, bit 2
// "value is its own code", bits 4-7 V - 1 for tensor-path columns.
enum : unsigned { kColContinuous = 0, kColTensor = 1, kColCompare = 2, kColConst = 3, kColPathMask = 3, kColIdent = 4 };

// How the one-hot distance slab of a call is obtained: computed from scratch, updated by
// subtracting the contribution of the columns removed since the cached slab (TuRF iterations:
// d_ij -= sum over removed f of [x_if != x_jf], exact integers), or reused as it is.  kDistNone:
// the call computes no distances (the joint-count and MDR paths read only At).
enum DistMode : int { kDistNone = -1, kDistFull = 0, kDistIncremental = 1, kDistReuse = 2 };

// Who owns which target rows (one process per GPU) and where their distance slabs live; passed
// by value to the distance kernel.  A single rank is the trivial case {starts = {0, n}}.
constexpr int kMaxRanks = 16;
struct DistPeers {
    int32_t *slab[kMaxRanks];       // [world] distance slab of every rank (own: local; others: CUDA IPC mappings)
    int64_t starts[kMaxRanks + 1];  // [world + 1] first target row (internal order) of every rank's shard
    int32_t sb_base[kMaxRanks + 1]; // [world + 1] running count of 256-row super-blocks of the shards
    int32_t world, rank;
    int32_t coarse_shift;           // symmetric mode: log2 of the super-block group size (see tc_dist.cu)
};
// One rank whose slab holds all `cols` sample columns (the trivial case above), in symmetric mode with groups of 8
// super-blocks: one rasterisation band of 16 tiles
inline DistPeers single_rank_peers(int32_t *slab, int64_t cols) {
    DistPeers p{};
    p.world = 1;
    p.slab[0] = slab;
    p.starts[1] = cols;
    p.sb_base[1] = (int32_t)ceil_div(cols, 256);
    p.coarse_shift = 3;
    return p;
}

// ---------------------------------------------------------------------------
// multi-GPU group (comm.cu): every rank owns one exchange arena with the same layout
// ---------------------------------------------------------------------------
struct CommHeader {
    uint32_t flags[kMaxRanks];   // flags[q]: last barrier epoch rank q published here
    uint32_t error;              // != 0: a barrier gave up (1 + the rank that never arrived)
    uint32_t pad[15];
};
struct CommPeers {
    CommHeader *hdr[kMaxRanks];  // base of every rank's arena (own: local; others: peer / IPC mappings)
    int32_t world, rank;
};
// Byte offsets inside an arena (identical on every rank: computed from n, p and the world size only)
struct GroupLayout {
    size_t off_slab;      // int32 [max shard rows (padded to 128), ldn]  symmetric distance slab of the rank's target rows
    size_t off_mask_h;    // FP4 nibbles [ldn, ldn / 2]  signed hit masks of ALL target rows (every rank fills its rows everywhere)
    size_t off_mask_m;    //   "   miss masks
    size_t off_rinfo;     // RowInfo [ldn]
    size_t off_w;         // double [world, p]  per-rank contribution to the weight sums
    size_t off_x;         // raw X (optional; sharded upload)
    size_t total;
};
// a rank's shard may exceed n / world by this many rows (shard boundaries on super-blocks of 256 target rows)
constexpr int64_t kShardSlack = 256;
// Rows of padding behind each neighbour mask (score.cu, group_layout): the accumulation kernels' tensor-map box of a
// target tile may reach that many rows past the tile's first row (tc_accum.cu checks the bound)
constexpr int64_t kAccumMaskPadRows = 256;
GroupLayout group_layout(int64_t n, int64_t p, int64_t max_shard_rows, int world, size_t x_bytes);

// Working set of one fs_score call: the active columns split by path.
struct WorkSet {
    // general (CUDA-core) path
    int64_t pg = 0;        // active general columns
    int64_t ldg = 0;       // padded column count (multiple of the chunk)
    int elem = 4;          // sizeof(T): 4 (FS_ARITH_F32) or 8 (FS_ARITH_F64)
    DevBuf<char> xg;       // [n, ldg] of T, internal row order
    DevBuf<float> xg32;    // [n, ldg] float32 image of (x - column minimum): SURF's accumulation (float64 arithmetic, continuous columns only)
    bool have_xg32 = false;
    DevBuf<float> rg;      // [ldg] recip (0 in padding)
    DevBuf<uint8_t> ctype; // [ldg / chunk]
    DevBuf<int64_t> gcol;  // [pg] original column of each general column
    DevBuf<int64_t> gout;  // [pg] position in the caller's feat_idx list
    std::vector<int64_t> h_gcol, h_gout;
    std::vector<uint8_t> h_ctype;
    std::vector<float> h_rg;
    // the column lists are those of `key` under the typing lists_typing (see build_lists)
    std::vector<int64_t> key;
    bool lists_uploaded = false;
    uint64_t lists_typing = ~0ull, lists_version = 0;
    int64_t n_cont = 0, n_cmp = 0;
    // one-hot tensor-core path (filled by onehot.cu).  A column with V distinct values owns
    // V - 1 "reduced" one-hot rows (values 0..V-2); the last value is implied (see onehot.cu)
    int64_t pt = 0;                 // active tensor-path columns (V >= 2)
    int64_t K = 0;                  // K_used padded to 128
    int64_t K_used = 0;             // sum of (V_f - 1): reduced one-hot rows in use
    bool all_ident = false;         // every tensor column's value is its own code (one-byte input, values 0..V-1)
    bool all_v3 = false;            // every tensor column has exactly 3 values (2 reduced rows): with all_ident, 0/1/2 genotypes
    DevBuf<int64_t> tcol, tout;     // [pt]
    DevBuf<int32_t> toff;           // [pt+1] first reduced one-hot row of each column
    PinnedBuf<int64_t> p_tcol, p_tout;   // host copies of tcol / tout / toff (pinned staging)
    PinnedBuf<int32_t> p_toff, p_tpos;
    DevBuf<int32_t> tpos;           // [pt] codesT row of each active column when the resident codesT is reused
    DevBuf<int8_t> U;               // [n, K]    sample-major, U[i,(f,v)] = [code == v]            (target side of the distance GEMM)
    DevBuf<int8_t> Wd;              // [n, K]    sample-major, U + [code != last]                 (sample side of the distance GEMM)
    DevBuf<int8_t> At;              // [K, ldt]  feature-major reduced one-hot (sample index contiguous)
    DevBuf<uint8_t> codesT;         // [pt, ldt] feature-major value codes (accumulation epilogue)
    DevBuf<uint8_t> codes;          // [n, ldc]  sample-major value codes (ReliefF gather only)
    DevBuf<int32_t> srow;           // [n] number of tensor columns whose code is not the last one
    DevBuf<uint32_t> krow;          // [K] per reduced row: column | value << 24 | last << 28
    int64_t ldt = 0, ldc = 0;
    bool have_codes = false;
    bool have_dist_ops = false;     // U / Wd / srow of the active columns are built
    int64_t u_lo = 0, u_hi = 0;     // sample rows held by U (the target rows it was built for)
    // distance plan of this call (see DistMode) and, for an incremental update, the reduced
    // one-hot operands of the columns that left the active set since the cached slab was built
    int dist_mode = 0;
    std::vector<int64_t> removed;   // original column indices
    int64_t Kr = 0, Kr_used = 0;
    PinnedBuf<int64_t> p_rcol;
    PinnedBuf<int32_t> p_roff;
    DevBuf<int64_t> rcol;
    DevBuf<int32_t> roff;
    DevBuf<int8_t> Ur, Wdr;         // [n, Kr]
    DevBuf<int32_t> srow_r;         // [n]
    bool valid = false;             // the operands are those of the column lists
    uint64_t build_id = 0;          // bumped by every rebuild: state derived from At is stale when it changes
    // feature-sharded accumulation (multi-GPU group): At / codesT / krow hold only the tensor columns
    // [a0, a1) of the active list -- this rank's share -- with one-hot rows numbered from 0
    int64_t a0 = 0, a1 = 0;        // == [0, pt) on one GPU
    int64_t Ka = 0, Ka_used = 0;   // one-hot rows of the slice (padded / in use)
    DevBuf<int32_t> atoff;         // [a1 - a0 + 1] first reduced row of each slice column, from 0
    PinnedBuf<int32_t> p_atoff;
    bool acc_split = false;
};

// What the one-hot distance slab holds after the last call (kept for TuRF's incremental distance update):
// the buffer, the tensor-path columns it sums over and the target rows it covers
struct SlabCache {
    bool valid = false;
    const int32_t *buf = nullptr;
    std::vector<int64_t> cols;
    uint64_t version = ~0ull;       // WorkSet::lists_version cols were filled for
    int64_t r0 = -1, R = -1;
    void forget() { valid = false; }
    void record(const int32_t *b, const WorkSet &ws, int64_t r0_, int64_t R_) {
        buf = b;
        if (version != ws.lists_version || (int64_t)cols.size() != ws.pt) {
            cols.assign(ws.p_tcol.ptr, ws.p_tcol.ptr + ws.pt);
            version = ws.lists_version;
        }
        r0 = r0_;
        R = R_;
        valid = true;
    }
};

}  // namespace fs

namespace fs {
// Ranks that live in ONE process (host threads; fs_multi_*, emulated ranks in the tests) also meet on the
// host right before every device-side barrier is launched.  The GPUs are not drained -- their queues
// keep running -- but once every thread has ISSUED its work up to the barrier, no barrier kernel can
// spin on a peer whose host thread is still stuck in a CUDA call that implicitly synchronises the
// process (page-locked or device allocations: CUDA programming guide, "Implicit Synchronization").
// Ranks in separate processes (CUDA IPC) have no such coupling and never meet on the host.
struct HostBarrier;
bool host_barrier_wait(HostBarrier *hb, double timeout_s);

}  // namespace fs

namespace fs {
// The reduced one-hot operand At of a list of discrete columns (ws.At, built without the distance operands)
// with its per-position offsets: what the joint-count and MDR paths read.  Built by discrete_operand for the
// first call on a column list and kept while the working set is not rebuilt.
struct DiscreteOperand {
    bool valid = false;
    std::vector<int64_t> key;       // n_kept (-1: all columns), then feat_idx
    uint64_t build_id = 0;          // ws.build_id it was built for
    uint64_t generation = 0;        // bumped by every rebuild: state derived from the operand is stale when it changes
    int max_rows = 0;               // largest reduced-row count (V - 1) of a column of the list
    std::vector<int32_t> start_h;   // [n_kept + 1] first reduced row of every position (none for a constant column)
    DevBuf<int32_t> start;          // device copy of start_h
    bool have_marg = false;
    DevBuf<int32_t> marg;           // [K] marginal counts of the reduced rows, computed when first asked for
};

// Segments of the MDR bit-planes (mdr.cu): segment s = 2 * fold + class owns the words [w[s], w[s + 1]).
constexpr int kMdrMaxSegments = 20;
struct MdrSeg {
    int32_t w[kMdrMaxSegments + 1];     // first word of every segment; w[nseg] = words in use
    int32_t n[kMdrMaxSegments];         // samples of every segment
};
}  // namespace fs

struct fs_comm {
    int rank = 0, world = 1, device = 0;
    std::shared_ptr<fs::HostBarrier> host_barrier;
    void *arena = nullptr;
    size_t arena_bytes = 0;
    void *opened[fs::kMaxRanks] = {};     // IPC mappings this communicator opened
    fs::CommPeers peers{};
    uint32_t epoch = 0;
    unsigned long long timeout_ns = 0;
    bool connected = false;
};

struct fs_dataset {
    int device = 0;
    cudaStream_t stream = nullptr;
    int64_t n = 0, p = 0;
    int dtype = FS_F32;
    int n_classes = 0;
    // raw matrix on the device, original row order
    const void *x = nullptr;
    int64_t ldx = 0;
    fs::DevBuf<char> x_owned;
    // class-sorted internal order
    std::vector<int64_t> perm, inv_perm;     // perm[r] = original index of internal row r
    std::vector<int32_t> y_sorted;           // class of internal row r
    std::vector<int64_t> cls_start;          // [C+1] internal row range of each class
    fs::DevBuf<int64_t> d_perm, d_inv_perm;
    fs::DevBuf<int32_t> d_y;
    fs::DevBuf<int64_t> d_cls_start;
    // column scan
    fs::DevBuf<double> d_cmin, d_cmax, d_vals;  // d_vals: [p, FS_DISTINCT_CAP]
    fs::DevBuf<int32_t> d_cnt;
    std::vector<double> cmin, cmax;
    std::vector<int32_t> cnt;
    // typing
    bool have_features = false;
    uint64_t typing_epoch = 0;               // bumped whenever the typing (or the group's column shares) changes
    uint64_t ct_version = ~0ull;             // WorkSet::lists_version ct_pos was filled for
    int arith = FS_ARITH_F32;
    std::vector<uint8_t> is_discrete;
    std::vector<float> recip;
    std::vector<uint8_t> col_info;           // kCol* flags per column
    // resident codesT (ws.codesT): row of each original column in it (-1: none); see build_onehot
    std::vector<int32_t> ct_pos;
    bool ct_valid = false;
    // per-call scratch, kept between calls (TuRF re-scores the same data set)
    fs::WorkSet ws;
    fs::DevBuf<double> Dc;        // [R, ldn] continuous/general distance part
    fs::DevBuf<int32_t> Dd;       // [R, ldn] one-hot mismatch counts
    fs::SlabCache slab;           // what Dd or peer_slab holds after the last call
    // multi-GPU symmetric distances (fs_dataset_attach_comm): this rank's slab in its arena and the
    // peers' mapped slabs
    fs::DistPeers peers{};
    int32_t *peer_slab = nullptr;
    fs::DevBuf<int8_t> sel;       // [R, ldn] neighbour codes
    fs::DevBuf<fs::RowInfo> rinfo;
    fs::DevBuf<double> partial;   // accumulation partials
    fs::DevBuf<double> wsum;      // [n_kept]
    fs::DevBuf<int32_t> nbr_idx;  // ReliefF neighbour lists
    fs::DevBuf<double> nbr_w;
    fs::DevBuf<int32_t> nbr_cnt;
    fs::DevBuf<float> d_class_probs;
    fs::DevBuf<double> tpartial;  // tensor-path accumulation partials
    fs::DevBuf<int32_t> tile_desc; // target-tile descriptors of the accumulation kernel
    fs::DevBuf<int32_t> tile_consts; // per-(tile, phase, target) coefficient limbs and mask row sums
    fs::DevBuf<int8_t> maskH, maskM;
    // multi-GPU group (fs_dataset_attach_comm): arena layout of this data set, this rank's target rows
    fs_comm *comm = nullptr;
    bool x_in_arena = false;                 // fs_dataset_create_group: the raw matrix lives in the arena
    fs::GroupLayout glayout{};
    std::vector<int64_t> owner_bound;        // [world + 1] original-column boundaries of the ranks' accumulation shares
    // ReliefF reference tie order (select.cu): compacted list of tied rows, [R, n] (key, index) pairs
    fs::DevBuf<int32_t> tie_list;
    fs::DevBuf<uint2> tie_pairs;
    fs::DevBuf<unsigned long long> counters;
    // joint-count and MDR paths: the shared operand (joint.cu)
    fs::DiscreteOperand disc;
    fs::DevBuf<double> joint_out;       // [n_kept, n_kept]
    fs::DevBuf<int32_t> joint_zero;     // zeros: the s_i / s_j vector of the reused distance kernel
    fs::DevBuf<int32_t> joint_slab;     // [band rows, ldd] negated reduced joint counts of one band
    fs::DevBuf<int64_t> joint_pairs, joint_tables;
    // column path (fs_joint_columns)
    fs::DevBuf<int32_t> jc_counts;           // [selected rows of one launch, K] reduced joint counts
    fs::DevBuf<int64_t> jc_pos;              // [n_pos] requested positions
    fs::DevBuf<int32_t> jc_off;              // [n_pos] first count row of each position within its launch
    fs::DevBuf<double> jc_out;               // [n_pos, n_kept] (host output)
    // MDR (mdr.cu): bit-planes of the operand of generation mdr_gen (0: none) and the folds `mdr_key`
    uint64_t mdr_gen = 0;
    std::vector<int64_t> mdr_key;            // n_folds, fold
    fs::MdrSeg mdr_seg{};
    int64_t mdr_W = 0;                       // words of a plane row (multiple of 4)
    int mdr_nseg = 0;
    fs::DevBuf<int32_t> mdr_slot;            // [32 W] internal row of every bit slot, -1: padding
    fs::DevBuf<uint8_t> mdr_wseg;            // [W] segment of every word
    fs::DevBuf<uint32_t> mdr_planes;         // [K, W] bit-planes in segment order
    fs::DevBuf<int32_t> mdr_marg;            // [K, nseg] popcount of every plane row in every segment
    fs::DevBuf<double> mdr_all;              // [2, n_combos] mean training / test BA of every combination
    fs::DevBuf<char> mdr_top, mdr_fold;      // block-local top lists (two merge buffers) and fold bests
    fs::DevBuf<long long> mdr_best;          // [n_folds] merged fold bests
    fs::DevBuf<int64_t> mdr_combos, mdr_tables;
};

namespace fs {

// dataset.cu: the working set of the columns feat_idx (all p columns when null), in two halves.
// build_lists: the columns split by path, the accumulation slice of a multi-GPU group call that may shard the
// accumulation by one-hot columns (want_split; WorkSet::acc_split), uploaded; kept while the call's columns,
// flags and the typing stay.  Marks the operands stale when the lists change.
void build_lists(fs_dataset *ds, const int64_t *feat_idx, int64_t n_kept, bool want_split, bool group_call);
// build_operands: the general columns gathered and the one-hot operands (build_onehot) for the distance mode
// `dist_mode` of target rows [u_lo, u_hi), unless the operands built last serve; those being the full distance
// operands, an incremental update becomes a full computation.  Sets ws.dist_mode.
void build_operands(fs_dataset *ds, bool need_codes, int dist_mode, int64_t u_lo, int64_t u_hi, bool group_call,
                    int *launches);

// joint.cu: the operand of the discrete columns feat_idx (all p columns when null) of a data set whose features
// are set.  Every column must be constant or a tensor-path column with at most max_values distinct values
// (FS_ERR_INVALID "<what>: column ... is not a discrete column with at most <max_values> distinct values"); with
// need_marg the marginals are there too.
const DiscreteOperand &discrete_operand(fs_dataset *ds, const int64_t *feat_idx, int64_t n_kept, int max_values,
                                        const char *what, bool need_marg, int *launches);

// comm.cu
void comm_barrier(fs_comm *c, cudaStream_t st, int *launches);
void comm_check(fs_comm *c);
void comm_push(fs_comm *c, size_t off, size_t bytes, cudaStream_t st, int *launches);

// onehot.cu: the reduced one-hot operands of the working set's tensor-path columns (U, Wd, srow when
// ws.have_dist_ops -- Wd only of the rows this rank's distance kernel reads in a group call; At, krow, codesT
// or tpos; codes when ws.have_codes) and, for an incremental distance update, those of the removed columns
void build_onehot(fs_dataset *ds, WorkSet &ws, bool group_call, int *launches);

// tc_dist.cu: the one-hot mismatch counts of the target rows [r0, r0 + R) (internal order) against all samples,
// into the slab Dd [R, ldn] (or subtracted from it for an incremental update); with `exchange` (this rank computes
// its whole shard into its arena slab) symmetric and mirrored into the peers' slabs
void launch_dist_tensor(fs_dataset *ds, const WorkSet &ws, int64_t r0, int64_t R, int32_t *Dd, int64_t ldn, bool exchange,
                        cudaStream_t st, int *launches, double *ops);
// The distance GEMM itself: D[r, j] = srow[r0 + r] + srow[j] - sum_k a[r, k] b[j, k] (subtract: D[r, j] -= that)
// over the FP4 operands a (R rows) and b (n rows), row_bytes wide at a pitch of `pitch` bytes, contracted over K
// bytes (a multiple of 128; bytes past row_bytes are the tensor maps' zero fill)
void launch_tc_dist(const int8_t *a, const int8_t *b, int64_t row_bytes, int64_t pitch, int64_t K, const int32_t *srow,
                    int64_t r0, int64_t R, int64_t n, int64_t ldd, bool symmetric, bool subtract,
                    const DistPeers &peers, cudaStream_t st, int *launches, double *ops);

// tc_accum.cu: wsum[tout[c]] += the MultiSURF / SURF weight of every one-hot column c of the working set's
// accumulation slice over the target rows [row0, row0 + R), from the FP4 neighbour masks (rows of ldn / 2 bytes,
// kAccumMaskPadRows rows of padding behind them) and the row constants rinfo
void launch_accum_tensor(fs_dataset *ds, const WorkSet &ws, int64_t row0, int64_t R, const int8_t *mask_h,
                         const int8_t *mask_m, int64_t ldn, const RowInfo *rinfo, double *wsum, cudaStream_t st,
                         int *launches, double *ops);

// dist_general.cu: D[r, j] = sum over general columns of the per-feature term
// between target row r (rows of xa) and sample j (rows of xb).
void launch_dist_general(const WorkSet &ws, const void *xa, int64_t na, const void *xb, int64_t nb,
                         double *D, int64_t ldd, cudaStream_t st, int *launches);

// select.cu: neighbours of the target rows [r0, r0 + R)
void launch_select(fs_dataset *ds, int algo, int use_star, int32_t k, int64_t r0, int64_t R,
                   const double *Dc, const int32_t *Dd, int64_t ldn, int8_t *sel, int8_t *mask_h, int8_t *mask_m,
                   RowInfo *rinfo,
                   int32_t *nbr_idx, double *nbr_w, int32_t *nbr_cnt, int32_t nbr_cap,
                   const float *class_probs, cudaStream_t st, int *launches);

// accum_general.cu: the target rows are the rows [row0, row0 + R) of the general matrix
int64_t accum_general_partials(const WorkSet &ws, int64_t R);
void launch_accum_general(const WorkSet &ws, int64_t n, int64_t row0, const int8_t *sel, int64_t ldn,
                          const RowInfo *rinfo, int64_t R, double *partial, int64_t n_part,
                          cudaStream_t st, int *launches);
void launch_relieff_gather(const WorkSet &ws, int64_t n, int64_t row0, const int32_t *nbr_idx,
                           const double *nbr_w, const int32_t *nbr_cnt, int32_t nbr_cap, int64_t R,
                           double *partial, int64_t n_part, cudaStream_t st, int *launches);
// ReliefF on the one-hot columns: wsum[tout[c]] += the weight of every tensor-path column c from the value codes
// (ws.codes) of the target rows [row0, row0 + R) and of their neighbours; partial is scratch
void launch_relieff_codes(const WorkSet &ws, int64_t row0, const int32_t *nbr_idx, const double *nbr_w,
                          const int32_t *nbr_cnt, int32_t nbr_cap, int64_t R, DevBuf<double> &partial, double *wsum,
                          cudaStream_t st, int *launches);
// wsum[gout[c]] += sum_q partial[q, c]  (fixed order => bitwise reproducible)
void launch_reduce_partials(const WorkSet &ws, const double *partial, int64_t n_part, double *wsum,
                            cudaStream_t st, int *launches);

}  // namespace fs
