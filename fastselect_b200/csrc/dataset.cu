// dataset.cu -- device-resident data set: upload, per-column scan (min / max /
// distinct values), class-sorted row order, and the per-call working set of
// active columns.  Replaces cuda.to_device(x) and the host np.unique / range pass
// of the reference's fit (MultiSURF.py:409-425, SURF.py:347-365, ReliefF.py:366-391)
// and TuRF's X[:, active] copy (TuRF.py:110).
#include <algorithm>
#include <cstring>
#include <thread>
#include <condition_variable>
#include <functional>
#include <array>
#include <cstring>
#include <mutex>
#include <numeric>

#include "common.cuh"

namespace fs {

static thread_local char g_err[1024] = "";

void set_error(const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
const char *get_error() { return g_err; }

cudaStream_t &alloc_stream() {
    static thread_local cudaStream_t s = nullptr;
    return s;
}

// process-wide free list of page-locked staging blocks (see PinnedBuf)
namespace {
struct PinnedBlock { void *ptr; size_t bytes; };
std::mutex g_pinned_mu;
std::vector<PinnedBlock> g_pinned_free;
}  // namespace

void *pinned_take(size_t bytes, size_t *got) {
    {
        std::lock_guard<std::mutex> lk(g_pinned_mu);
        // smallest cached block that is large enough
        int best = -1;
        for (int i = 0; i < (int)g_pinned_free.size(); ++i)
            if (g_pinned_free[i].bytes >= bytes && (best < 0 || g_pinned_free[i].bytes < g_pinned_free[best].bytes)) best = i;
        if (best >= 0) {
            PinnedBlock b = g_pinned_free[best];
            g_pinned_free.erase(g_pinned_free.begin() + best);
            *got = b.bytes;
            return b.ptr;
        }
    }
    void *p = nullptr;
    bytes = (size_t)round_up((int64_t)bytes, 4096);
    FS_CUDA(cudaMallocHost(&p, bytes));
    *got = bytes;
    return p;
}

void pinned_give(void *ptr, size_t bytes) {
    std::lock_guard<std::mutex> lk(g_pinned_mu);
    if (g_pinned_free.size() >= 16) {           // bound the cache: drop the smallest block
        int small = 0;
        for (int i = 1; i < (int)g_pinned_free.size(); ++i)
            if (g_pinned_free[i].bytes < g_pinned_free[small].bytes) small = i;
        if (g_pinned_free[small].bytes < bytes) {
            cudaFreeHost(g_pinned_free[small].ptr);
            g_pinned_free[small] = PinnedBlock{ptr, bytes};
        } else {
            cudaFreeHost(ptr);
        }
        return;
    }
    g_pinned_free.push_back(PinnedBlock{ptr, bytes});
}

// ---------------------------------------------------------------------------
// A small process-wide pool of host threads (never torn down) for the staged upload of pageable matrices
// ---------------------------------------------------------------------------
namespace {
struct HostPool {
    std::mutex mu;
    std::condition_variable cv_work, cv_done;
    const std::function<void(int64_t, int64_t)> *fn = nullptr;
    int64_t next = 0, total = 0, per = 1;
    int active = 0;
    uint64_t generation = 0;
    int n_threads = 0;

    HostPool() {
        const unsigned hw = std::thread::hardware_concurrency();
        n_threads = (int)std::max(1u, std::min(8u, hw ? hw / 2 : 4u)) - 1;      // the caller works too
        for (int i = 0; i < n_threads; ++i) std::thread([this] { loop(); }).detach();
    }
    bool take(int64_t &a, int64_t &e) {
        if (next >= total) return false;
        a = next;
        e = std::min(total, next + per);
        next = e;
        return true;
    }
    void loop() {
        uint64_t seen = 0;
        std::unique_lock<std::mutex> lk(mu);
        for (;;) {
            cv_work.wait(lk, [&] { return generation != seen; });
            seen = generation;
            int64_t a, e;
            while (take(a, e)) {
                ++active;
                lk.unlock();
                (*fn)(a, e);
                lk.lock();
                --active;
            }
            if (active == 0) cv_done.notify_all();
        }
    }
    void run(int64_t n, int64_t chunk, const std::function<void(int64_t, int64_t)> &f) {
        std::unique_lock<std::mutex> lk(mu);
        fn = &f;
        next = 0;
        total = n;
        per = std::max<int64_t>(1, chunk);
        ++generation;
        cv_work.notify_all();
        int64_t a, e;
        while (take(a, e)) {
            ++active;
            lk.unlock();
            f(a, e);
            lk.lock();
            --active;
        }
        cv_done.wait(lk, [&] { return active == 0 && next >= total; });
        fn = nullptr;
    }
};
std::mutex g_pool_users;     // one staged upload at a time uses the pool
}  // namespace

void host_parallel_for(int64_t n, int64_t chunk, const std::function<void(int64_t, int64_t)> &f) {
    static HostPool *pool = new HostPool();      // leaked on purpose: its threads outlive static destruction
    std::lock_guard<std::mutex> users(g_pool_users);
    pool->run(n, chunk, f);
}

// keep freed blocks in the device's default memory pool (no trimming at synchronisation)
void configure_pool(int device) {
    static bool done[64] = {false};
    if (device < 0 || device >= 64 || done[device]) return;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, device) == cudaSuccess) {
        unsigned long long thresh = ~0ull;
        cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thresh);
    }
    cudaGetLastError();
    done[device] = true;
}

// ---------------------------------------------------------------------------
// column scan: one thread per column, rows streamed coalesced across columns.
// HBM-bound: reads n*p*sizeof(T) once.
// ---------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(128) column_scan_kernel(const T *__restrict__ x, int64_t row_begin, int64_t row_end,
                                                          int64_t p, int64_t ldx, double *__restrict__ cmin,
                                                          double *__restrict__ cmax, int32_t *__restrict__ cnt,
                                                          double *__restrict__ vals, int first, int last) {
    int64_t f = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (f >= p) return;
    // per-column state: carried through global memory between row chunks (the upload is chunked
    // so that the scan of one chunk runs under the copy of the next); values came from T, so the
    // round trip through double is exact
    T set[FS_DISTINCT_CAP] = {};
    int c = 0;
    bool over = false;
    T mn = x[row_begin * ldx + f], mx = mn;
    if (!first) {
        mn = (T)cmin[f];
        mx = (T)cmax[f];
        c = cnt[f];
        over = c > FS_DISTINCT_CAP;
        c = over ? FS_DISTINCT_CAP : c;
#pragma unroll
        for (int q = 0; q < FS_DISTINCT_CAP; ++q) set[q] = (T)vals[f * FS_DISTINCT_CAP + q];
    }
    for (int64_t i = row_begin; i < row_end; ++i) {
        T v = x[i * ldx + f];
        mn = v < mn ? v : mn;
        mx = v > mx ? v : mx;
        if (!over) {
            bool found = false;
#pragma unroll
            for (int q = 0; q < FS_DISTINCT_CAP; ++q) found |= (q < c) && (set[q] == v);
            if (!found) {
                if (c < FS_DISTINCT_CAP) {
#pragma unroll
                    for (int q = 0; q < FS_DISTINCT_CAP; ++q)
                        if (q == c) set[q] = v;
                    ++c;
                } else {
                    over = true;
                }
            }
        }
    }
    if (last) {
        // ascending value order (odd-even transposition on registers): for 0/1/2 genotypes the
        // value code is then the value itself, which the one-hot encoder exploits
#pragma unroll
        for (int pass = 0; pass < FS_DISTINCT_CAP; ++pass) {
#pragma unroll
            for (int q = pass & 1; q + 1 < FS_DISTINCT_CAP; q += 2) {
                const bool sw = (q + 1 < c) && (set[q + 1] < set[q]);
                const T lo = sw ? set[q + 1] : set[q], hi = sw ? set[q] : set[q + 1];
                set[q] = lo;
                set[q + 1] = hi;
            }
        }
    }
    cmin[f] = (double)mn;
    cmax[f] = (double)mx;
    cnt[f] = over ? FS_DISTINCT_CAP + 1 : c;
#pragma unroll
    for (int q = 0; q < FS_DISTINCT_CAP; ++q) vals[f * FS_DISTINCT_CAP + q] = q < c ? (double)set[q] : 0.0;
}

template <typename T>
static void run_scan(fs_dataset *ds, int64_t row_begin, int64_t row_end, bool first, bool last) {
    int64_t p = ds->p;
    dim3 grid((unsigned)ceil_div(p, 128));
    column_scan_kernel<T><<<grid, 128, 0, ds->stream>>>(static_cast<const T *>(ds->x), row_begin, row_end, p, ds->ldx,
                                                         ds->d_cmin.ptr, ds->d_cmax.ptr, ds->d_cnt.ptr,
                                                         ds->d_vals.ptr, first ? 1 : 0, last ? 1 : 0);
    FS_CUDA(cudaGetLastError());
}

static void scan_rows(fs_dataset *ds, int64_t row_begin, int64_t row_end, bool first, bool last) {
    switch (ds->dtype) {
        case FS_U8: run_scan<uint8_t>(ds, row_begin, row_end, first, last); break;
        case FS_I8: run_scan<int8_t>(ds, row_begin, row_end, first, last); break;
        case FS_F32: run_scan<float>(ds, row_begin, row_end, first, last); break;
        case FS_F64: run_scan<double>(ds, row_begin, row_end, first, last); break;
    }
}

static size_t dtype_size(int dtype) {
    switch (dtype) {
        case FS_U8:
        case FS_I8: return 1;
        case FS_F32: return 4;
        case FS_F64: return 8;
    }
    return 0;
}

// class-sorted row order + scan buffers (everything of create that does not need X)
static void prepare_create(fs_dataset *ds, const int32_t *y_enc) {
    const int64_t n = ds->n, p = ds->p;
    // stable class sort of the samples: hits of a target are one contiguous row
    // range, each miss class another (used by ReliefF's per-class selection).
    ds->perm.resize(n);
    std::iota(ds->perm.begin(), ds->perm.end(), (int64_t)0);
    std::stable_sort(ds->perm.begin(), ds->perm.end(),
                     [&](int64_t a, int64_t b) { return y_enc[a] < y_enc[b]; });
    ds->inv_perm.resize(n);
    ds->y_sorted.resize(n);
    ds->cls_start.assign(ds->n_classes + 1, 0);
    for (int64_t r = 0; r < n; ++r) {
        ds->inv_perm[ds->perm[r]] = r;
        ds->y_sorted[r] = y_enc[ds->perm[r]];
        ds->cls_start[ds->y_sorted[r] + 1]++;
    }
    for (int c = 0; c < ds->n_classes; ++c) ds->cls_start[c + 1] += ds->cls_start[c];
    ds->d_perm.alloc(n);
    ds->d_inv_perm.alloc(n);
    ds->d_y.alloc(n);
    ds->d_cls_start.alloc(ds->n_classes + 1);
    FS_CUDA(cudaMemcpyAsync(ds->d_perm.ptr, ds->perm.data(), n * sizeof(int64_t), cudaMemcpyHostToDevice, ds->stream));
    FS_CUDA(cudaMemcpyAsync(ds->d_inv_perm.ptr, ds->inv_perm.data(), n * sizeof(int64_t), cudaMemcpyHostToDevice, ds->stream));
    FS_CUDA(cudaMemcpyAsync(ds->d_y.ptr, ds->y_sorted.data(), n * sizeof(int32_t), cudaMemcpyHostToDevice, ds->stream));
    FS_CUDA(cudaMemcpyAsync(ds->d_cls_start.ptr, ds->cls_start.data(), (ds->n_classes + 1) * sizeof(int64_t),
                            cudaMemcpyHostToDevice, ds->stream));
    ds->d_cmin.alloc(p);
    ds->d_cmax.alloc(p);
    ds->d_cnt.alloc(p);
    ds->d_vals.alloc((size_t)p * FS_DISTINCT_CAP);
    ds->cmin.resize(p);
    ds->cmax.resize(p);
    ds->cnt.resize(p);
}

// column scan results back to the host
static void finish_create(fs_dataset *ds) {
    const int64_t p = ds->p;
    FS_CUDA(cudaMemcpyAsync(ds->cmin.data(), ds->d_cmin.ptr, p * sizeof(double), cudaMemcpyDeviceToHost, ds->stream));
    FS_CUDA(cudaMemcpyAsync(ds->cmax.data(), ds->d_cmax.ptr, p * sizeof(double), cudaMemcpyDeviceToHost, ds->stream));
    FS_CUDA(cudaMemcpyAsync(ds->cnt.data(), ds->d_cnt.ptr, p * sizeof(int32_t), cudaMemcpyDeviceToHost, ds->stream));
    FS_CUDA(cudaStreamSynchronize(ds->stream));
}

// Static ownership of the one-hot columns inside a multi-GPU group: rank r accumulates the tensor-path
// columns whose original index lies in [owner_bound[r], owner_bound[r + 1]) -- equal shares of the data
// set's tensor-path columns.  Fixed for the life of the typing, so that TuRF iterations keep finding
// their columns' value codes in the rank's resident codesT.
static void compute_owner_bounds(fs_dataset *ds) {
    ds->owner_bound.clear();
    if (!ds->comm || !ds->have_features) return;
    std::vector<int64_t> tc;
    for (int64_t f = 0; f < ds->p; ++f)
        if ((ds->col_info[f] & kColPathMask) == kColTensor) tc.push_back(f);
    const int world = ds->comm->world;
    const int64_t T = (int64_t)tc.size();
    ds->owner_bound.assign(world + 1, ds->p);
    ds->owner_bound[0] = 0;
    // shares of whole 64-column tiles of the encoder where the list is long enough
    for (int r = 1; r < world; ++r) {
        int64_t pos = T * r / world;
        if (T >= 64LL * 4 * world) pos = pos / 64 * 64;
        ds->owner_bound[r] = pos < T ? tc[pos] : ds->p;
    }
}

// Drop what was derived from the typing or the group: the working set's operands and the cached distance slab
// always, the resident codesT with `codes`, and with `retyped` the column lists (typing_epoch) and the ranks'
// accumulation shares
static void forget_derived(fs_dataset *ds, bool codes, bool retyped) {
    ds->ws.valid = false;
    ds->slab.forget();
    if (codes) ds->ct_valid = false;
    if (retyped) {
        ++ds->typing_epoch;
        compute_owner_bounds(ds);
    }
}

static int usable_devices() {
    int count = 0;
    if (cudaGetDeviceCount(&count) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    int ok = 0;
    for (int d = 0; d < count; ++d) {
        int major = 0;
        if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, d) == cudaSuccess && major == 10) ++ok;
    }
    return ok;
}

static fs_dataset *create_common(int dtype, int64_t n, int64_t p, int64_t ld, const int32_t *y_enc,
                                 int32_t n_classes, int32_t device, void *stream) {
    FS_REQUIRE(n >= 2 && p >= 1, FS_ERR_INVALID, "fs_dataset_create: need n >= 2 and p >= 1 (got n=%lld p=%lld)",
               (long long)n, (long long)p);
    FS_REQUIRE(n < (1LL << 31) - 256, FS_ERR_INVALID, "fs_dataset_create: n too large");
    FS_REQUIRE(dtype_size(dtype) != 0, FS_ERR_INVALID, "fs_dataset_create: unknown dtype %d", dtype);
    FS_REQUIRE(ld >= p, FS_ERR_INVALID, "fs_dataset_create: row stride %lld < p %lld", (long long)ld, (long long)p);
    FS_REQUIRE(y_enc != nullptr && n_classes >= 1, FS_ERR_INVALID, "fs_dataset_create: y_enc / n_classes missing");
    for (int64_t i = 0; i < n; ++i)
        FS_REQUIRE(y_enc[i] >= 0 && y_enc[i] < n_classes, FS_ERR_INVALID,
                   "fs_dataset_create: y_enc[%lld]=%d outside [0,%d)", (long long)i, y_enc[i], n_classes);
    FS_REQUIRE(usable_devices() > 0, FS_ERR_NO_DEVICE,
               "no usable NVIDIA sm_100 (B200) GPU: this library has no CPU fallback");
    int major = 0;
    FS_CUDA(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device));
    FS_REQUIRE(major == 10, FS_ERR_NO_DEVICE, "device %d is not sm_100 (compute capability major %d)", device, major);
    FS_CUDA(cudaSetDevice(device));
    configure_pool(device);
    alloc_stream() = static_cast<cudaStream_t>(stream);
    fs_dataset *ds = new fs_dataset();
    ds->device = device;
    ds->stream = static_cast<cudaStream_t>(stream);
    ds->n = n;
    ds->p = p;
    ds->dtype = dtype;
    ds->n_classes = n_classes;
    return ds;
}

// ---------------------------------------------------------------------------
// working set: gather the active general-path columns, internal row order
// ---------------------------------------------------------------------------
template <typename Tin, typename Tout>
__global__ void __launch_bounds__(256) gather_general_kernel(const Tin *__restrict__ x, int64_t ldx,
                                                             const int64_t *__restrict__ perm,
                                                             const int64_t *__restrict__ col, int64_t pg,
                                                             int64_t n, int64_t ldg, Tout *__restrict__ out) {
    int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    int64_t r = blockIdx.y;
    if (c >= ldg) return;
    for (; r < n; r += gridDim.y) {
        Tout v = (Tout)0;
        if (c < pg) {
            int64_t src = col[c];
            if (src >= 0) v = (Tout)x[perm[r] * ldx + src];
        }
        out[r * ldg + c] = v;
    }
}

// xg32[r, c] = (float)(xg[r, c] - min of the column): see launch_accum_general
__global__ void __launch_bounds__(256) narrow_general_kernel(const double *__restrict__ xg, const int64_t *__restrict__ col,
                                                             const double *__restrict__ cmin, int64_t n, int64_t ldg,
                                                             float *__restrict__ out) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= ldg) return;
    const int64_t src = col[c];
    const double m = src >= 0 ? cmin[src] : 0.0;
    for (int64_t r = blockIdx.y; r < n; r += gridDim.y) out[r * ldg + c] = (float)(xg[r * ldg + c] - m);
}

template <typename Tin>
static void run_gather(fs_dataset *ds, WorkSet &ws, int *launches) {
    dim3 grid((unsigned)ceil_div(ws.ldg, 256), (unsigned)std::min<int64_t>(ds->n, 4096));
    if (ws.elem == 4)
        gather_general_kernel<Tin, float><<<grid, 256, 0, ds->stream>>>(
            static_cast<const Tin *>(ds->x), ds->ldx, ds->d_perm.ptr, ws.gcol.ptr, ws.pg, ds->n, ws.ldg,
            reinterpret_cast<float *>(ws.xg.ptr));
    else
        gather_general_kernel<Tin, double><<<grid, 256, 0, ds->stream>>>(
            static_cast<const Tin *>(ds->x), ds->ldx, ds->d_perm.ptr, ws.gcol.ptr, ws.pg, ds->n, ws.ldg,
            reinterpret_cast<double *>(ws.xg.ptr));
    FS_CUDA(cudaGetLastError());
    ++*launches;
}

void build_lists(fs_dataset *ds, const int64_t *feat_idx, int64_t n_kept, bool want_split, bool group_call) {
    WorkSet &ws = ds->ws;
    Trace tr_all("build_lists");
    // key: flags + the explicit column list (none when every column is active)
    const bool all = feat_idx == nullptr;
    std::vector<int64_t> key(3 + (all ? 0 : n_kept));
    key[0] = (want_split ? 1 : 0) | (group_call ? 2 : 0);
    key[1] = ds->arith;
    key[2] = all ? -1 : n_kept;
    if (!all) memcpy(key.data() + 3, feat_idx, n_kept * sizeof(int64_t));
    // the lists depend only on the key and the typing (fs_dataset_set_features, and the group's column shares):
    // they are kept (host vectors, pinned staging and their device copies) until one of those changes, so that
    // re-scoring the same columns does not walk them on the host again
    if (ws.key == key && ws.lists_typing == ds->typing_epoch) return;
    ws.valid = false;
    ws.key.clear();                 // until the lists are complete (a bad column below throws)
    const int chunk = kChunkBytes / (ds->arith == FS_ARITH_F64 ? 8 : 4);
    ws.elem = ds->arith == FS_ARITH_F64 ? 8 : 4;
    // split the active columns: one-hot tensor path (discrete, 2 <= V <= FS_DISTINCT_CAP),
    // continuous, and wide discrete ("compare") columns.  The tensor-path lists are written
    // straight into the pinned staging buffers the encode kernel's inputs are copied from;
    // the per-column decisions were made once in fs_dataset_set_features (col_info).
    std::vector<int64_t> cont_col, cont_out, cmp_col, cmp_out;
    Trace *tr_loop = new Trace("  classify columns");
    ws.p_tcol.reserve(n_kept);
    ws.p_tout.reserve(n_kept);
    ws.p_toff.reserve(n_kept + 1);
    int64_t *tcol = ws.p_tcol.ptr, *tout = ws.p_tout.ptr;
    int32_t *toff = ws.p_toff.ptr;
    const uint8_t *info = ds->col_info.data();
    int64_t pt = 0, K = 0, first_const = -1, first_const_out = -1;
    unsigned ident = kColIdent;
    bool v3 = true;
    for (int64_t c = 0; c < n_kept; ++c) {
        const int64_t f = all ? c : feat_idx[c];
        FS_REQUIRE(f >= 0 && f < ds->p, FS_ERR_INVALID, "feat_idx[%lld]=%lld outside [0,%lld)", (long long)c,
                   (long long)f, (long long)ds->p);
        const unsigned ci = info[f];
        switch (ci & kColPathMask) {
            case kColTensor:
                tcol[pt] = f;
                tout[pt] = c;
                toff[pt] = (int32_t)K;
                K += ci >> 4;                      // V - 1 reduced one-hot rows
                ident &= ci;
                v3 = v3 && (ci >> 4) == 2;
                ++pt;
                break;
            case kColConst:
                // a constant column: every per-feature term is 0 (MultiSURF.py:184-185), so it
                // adds nothing to any distance and its weight stays 0 -- it takes no part
                if (first_const < 0) {
                    first_const = f;
                    first_const_out = c;
                }
                break;
            case kColCompare:
                cmp_col.push_back(f);
                cmp_out.push_back(c);
                break;
            default:
                cont_col.push_back(f);
                cont_out.push_back(c);
        }
    }
    delete tr_loop;
    FS_REQUIRE(K < (1LL << 31) - 128, FS_ERR_INVALID, "one-hot contraction length too large");
    toff[pt] = (int32_t)K;
    if (pt == 0 && cont_col.empty() && cmp_col.empty()) {
        // nothing but constant columns: keep one on the compare path so the pipeline has a
        // (zero) distance matrix to select on
        cmp_col.push_back(first_const);
        cmp_out.push_back(first_const_out);
    }
    ws.pt = pt;
    ws.K_used = K;
    // feature-sharded accumulation: this rank's share of the active one-hot columns is the run of the
    // (ascending) list that falls inside its static range of original columns (owner_bound)
    ws.a0 = 0;
    ws.a1 = pt;
    ws.acc_split = false;
    if (want_split && pt > 0 && ds->comm && (int)ds->owner_bound.size() == ds->comm->world + 1) {
        bool ascending = true;
        for (int64_t c = 1; c < pt && ascending; ++c) ascending = tcol[c] > tcol[c - 1];
        if (ascending) {
            const int rk = ds->comm->rank;
            ws.a0 = std::lower_bound(tcol, tcol + pt, ds->owner_bound[rk]) - tcol;
            ws.a1 = std::lower_bound(tcol, tcol + pt, ds->owner_bound[rk + 1]) - tcol;
            ws.acc_split = true;
        }
    }
    ws.all_ident = (ident & kColIdent) != 0;
    ws.all_v3 = v3 && pt > 0;
    ws.n_cont = (int64_t)cont_col.size();
    ws.n_cmp = (int64_t)cmp_col.size();

    // general path layout: [continuous | pad to chunk | compare | pad to chunk]
    ws.h_gcol.clear();
    ws.h_gout.clear();
    std::vector<uint8_t> &ctype = ws.h_ctype;
    std::vector<float> &rg = ws.h_rg;
    ctype.clear();
    rg.clear();
    auto append = [&](const std::vector<int64_t> &cols, const std::vector<int64_t> &outs, uint8_t type) {
        if (cols.empty()) return;
        for (size_t q = 0; q < cols.size(); ++q) {
            ws.h_gcol.push_back(cols[q]);
            ws.h_gout.push_back(outs[q]);
            rg.push_back(type == kChunkContinuous ? ds->recip[cols[q]] : 0.0f);
        }
        while (ws.h_gcol.size() % chunk) {
            ws.h_gcol.push_back(-1);
            ws.h_gout.push_back(-1);
            rg.push_back(0.0f);
        }
        ctype.resize(ws.h_gcol.size() / chunk, type);
    };
    append(cont_col, cont_out, kChunkContinuous);
    append(cmp_col, cmp_out, kChunkCompare);
    ws.pg = (int64_t)ws.h_gcol.size();
    ws.ldg = ws.pg;
    if (ws.pg > 0) {
        // (the staging vectors live in the working set: no synchronisation needed before they go out of scope)
        ws.rg.reserve(ws.ldg);
        ws.ctype.reserve(ctype.size());
        ws.gcol.reserve(ws.pg);
        ws.gout.reserve(ws.pg);
        FS_CUDA(cudaMemcpyAsync(ws.rg.ptr, rg.data(), rg.size() * sizeof(float), cudaMemcpyHostToDevice, ds->stream));
        FS_CUDA(cudaMemcpyAsync(ws.ctype.ptr, ctype.data(), ctype.size(), cudaMemcpyHostToDevice, ds->stream));
        FS_CUDA(cudaMemcpyAsync(ws.gcol.ptr, ws.h_gcol.data(), ws.pg * sizeof(int64_t), cudaMemcpyHostToDevice, ds->stream));
        FS_CUDA(cudaMemcpyAsync(ws.gout.ptr, ws.h_gout.data(), ws.pg * sizeof(int64_t), cudaMemcpyHostToDevice, ds->stream));
    }
    ws.key = std::move(key);
    ws.lists_typing = ds->typing_epoch;
    ++ws.lists_version;
    ws.lists_uploaded = false;
}

void build_operands(fs_dataset *ds, bool need_codes, int dist_mode, int64_t u_lo, int64_t u_hi, bool group_call,
                    int *launches) {
    WorkSet &ws = ds->ws;
    if (ws.valid && (ws.have_codes || !need_codes || ws.pt == 0) &&
        (dist_mode == kDistNone || dist_mode == kDistReuse || ws.pt == 0 ||
         (ws.have_dist_ops && ws.u_lo <= u_lo && u_hi <= ws.u_hi))) {
        ws.dist_mode = dist_mode == kDistIncremental ? kDistFull : dist_mode;
        return;
    }
    Trace tr_all("build_operands");
    ws.valid = false;
    ws.have_xg32 = false;
    if (ws.pg > 0) {
        ws.xg.reserve((size_t)ds->n * ws.ldg * ws.elem);
        switch (ds->dtype) {
            case FS_U8: run_gather<uint8_t>(ds, ws, launches); break;
            case FS_I8: run_gather<int8_t>(ds, ws, launches); break;
            case FS_F32: run_gather<float>(ds, ws, launches); break;
            case FS_F64: run_gather<double>(ds, ws, launches); break;
        }
        ws.have_xg32 = ws.elem == 8 && ws.n_cmp == 0;
        if (ws.have_xg32) {
            ws.xg32.reserve((size_t)ds->n * ws.ldg);
            dim3 grid((unsigned)ceil_div(ws.ldg, 256), (unsigned)std::min<int64_t>(ds->n, 4096));
            narrow_general_kernel<<<grid, 256, 0, ds->stream>>>(reinterpret_cast<const double *>(ws.xg.ptr), ws.gcol.ptr,
                                                                ds->d_cmin.ptr, ds->n, ws.ldg, ws.xg32.ptr);
            FS_CUDA(cudaGetLastError());
            ++*launches;
        }
    }
    ws.K = 0;
    ws.have_codes = need_codes;
    ws.dist_mode = dist_mode;
    ws.have_dist_ops = dist_mode == kDistFull;
    ws.u_lo = u_lo;
    ws.u_hi = u_hi;
    if (ws.pt > 0) {
        Trace tr("  build_onehot");
        build_onehot(ds, ws, group_call, launches);
    }
    ws.valid = true;
    ++ws.build_id;
}

}  // namespace fs

// ---------------------------------------------------------------------------
// C ABI
// ---------------------------------------------------------------------------
using namespace fs;

extern "C" {

int fs_device_count(void) { return usable_devices(); }
const char *fs_last_error(void) { return get_error(); }
int fs_abi_version(void) { return FS_ABI_VERSION; }

int fs_dataset_create(fs_dataset **out, const void *x, int dtype, int64_t n, int64_t p, int64_t row_stride_elems,
                      const int32_t *y_enc, int32_t n_classes, int32_t device, void *stream) {
    return api_call("fs_dataset_create", [&] {
        FS_REQUIRE(out && x, FS_ERR_INVALID, "fs_dataset_create: null pointer");
        std::unique_ptr<fs_dataset> owner(create_common(dtype, n, p, row_stride_elems, y_enc, n_classes, device, stream));
        fs_dataset *ds = owner.get();
        size_t es = dtype_size(dtype);
        ds->ldx = round_up(p, 16 / (int64_t)es > 0 ? 16 / (int64_t)es : 1);
        ds->x_owned.alloc((size_t)n * ds->ldx * es);
        ds->x = ds->x_owned.ptr;
        // upload in row chunks on a side stream; the scan of chunk i (data set's stream) runs
        // under the copy of chunk i + 1, so only the last chunk's scan is exposed
        const int64_t row_bytes = p * (int64_t)es;
        int64_t chunk_rows = std::max<int64_t>(1, (32LL << 20) / std::max<int64_t>(1, row_bytes));
        if (ceil_div(n, chunk_rows) > 64) chunk_rows = ceil_div(n, 64);
        const int n_chunks = (int)ceil_div(n, chunk_rows);
        cudaStream_t copy_stream = nullptr;
        std::vector<cudaEvent_t> done(n_chunks, nullptr);
        FS_CUDA(cudaStreamCreateWithFlags(&copy_stream, cudaStreamNonBlocking));
        try {
            // the copies must not start before the allocation (stream-ordered on ds->stream) exists
            cudaEvent_t ready;
            FS_CUDA(cudaEventCreateWithFlags(&ready, cudaEventDisableTiming));
            FS_CUDA(cudaEventRecord(ready, ds->stream));
            FS_CUDA(cudaStreamWaitEvent(copy_stream, ready, 0));
            cudaEventDestroy(ready);
            // A PAGEABLE source (an ordinary numpy array) would be staged by the driver, one thread, ~10 GB/s:
            // 45 ms for C3's 400 MB against 7 ms of PCIe time.  Instead several host threads copy every chunk into
            // one of a few page-locked blocks (the pool of PinnedBuf) while the previous chunk's DMA runs.
            cudaPointerAttributes attr{};
            const bool pageable = cudaPointerGetAttributes(&attr, x) != cudaSuccess || attr.type == cudaMemoryTypeUnregistered;
            (void)cudaGetLastError();            // an unregistered pointer may leave a sticky-free error behind
            const bool staged = pageable && (int64_t)n * row_bytes >= (8LL << 20) && !getenv("FS_B200_NO_STAGED_UPLOAD");
            if (!staged) {
                for (int c = 0; c < n_chunks; ++c) {
                    const int64_t r0 = c * chunk_rows, r1 = std::min<int64_t>(n, r0 + chunk_rows);
                    FS_CUDA(cudaMemcpy2DAsync(ds->x_owned.ptr + (size_t)r0 * ds->ldx * es, ds->ldx * es,
                                              static_cast<const char *>(x) + (size_t)r0 * row_stride_elems * es,
                                              row_stride_elems * es, p * es, r1 - r0, cudaMemcpyHostToDevice, copy_stream));
                    FS_CUDA(cudaEventCreateWithFlags(&done[c], cudaEventDisableTiming));
                    FS_CUDA(cudaEventRecord(done[c], copy_stream));
                }
                prepare_create(ds, y_enc);          // host work (class sort) overlaps the first copies
                for (int c = 0; c < n_chunks; ++c) {
                    const int64_t r0 = c * chunk_rows, r1 = std::min<int64_t>(n, r0 + chunk_rows);
                    FS_CUDA(cudaStreamWaitEvent(ds->stream, done[c], 0));
                    scan_rows(ds, r0, r1, c == 0, c == n_chunks - 1);
                }
            } else {
                // own chunking: 8 MB pieces through four page-locked blocks (small, so that the first call's
                // cudaMallocHost stays cheap), copied by the process-wide pool of host threads
                constexpr int kBlocks = 4;
                const int64_t srows = std::max<int64_t>(1, (8LL << 20) / std::max<int64_t>(1, row_bytes));
                const int64_t s_chunks = ceil_div(n, srows);
                PinnedBuf<char> stage[kBlocks];
                cudaEvent_t freed[kBlocks] = {nullptr, nullptr, nullptr, nullptr};
                for (int b = 0; b < kBlocks && b < s_chunks; ++b) stage[b].reserve((size_t)srows * (size_t)row_bytes);
                cudaEvent_t landed = nullptr;
                try {
                    prepare_create(ds, y_enc);
                    FS_CUDA(cudaEventCreateWithFlags(&landed, cudaEventDisableTiming));
                    for (int64_t c = 0; c < s_chunks; ++c) {
                        const int64_t r0 = c * srows, r1 = std::min<int64_t>(n, r0 + srows);
                        const int b = (int)(c % kBlocks);
                        if (freed[b]) FS_CUDA(cudaEventSynchronize(freed[b]));      // the block's previous DMA has finished
                        char *dst = stage[b].ptr;
                        const char *src = static_cast<const char *>(x) + (size_t)r0 * row_stride_elems * es;
                        const int64_t rows = r1 - r0;
                        // slices of ~512 KB: whole rows
                        const int64_t per = std::max<int64_t>(1, (512LL << 10) / std::max<int64_t>(1, row_bytes));
                        host_parallel_for(rows, per, [&](int64_t a, int64_t e) {
                            if ((int64_t)row_stride_elems == p)
                                memcpy(dst + (size_t)a * row_bytes, src + (size_t)a * row_bytes, (size_t)(e - a) * row_bytes);
                            else
                                for (int64_t r = a; r < e; ++r)
                                    memcpy(dst + (size_t)r * row_bytes, src + (size_t)r * row_stride_elems * es, (size_t)row_bytes);
                        });
                        FS_CUDA(cudaMemcpy2DAsync(ds->x_owned.ptr + (size_t)r0 * ds->ldx * es, ds->ldx * es, dst, (size_t)row_bytes,
                                                  p * es, rows, cudaMemcpyHostToDevice, copy_stream));
                        if (!freed[b]) FS_CUDA(cudaEventCreateWithFlags(&freed[b], cudaEventDisableTiming));
                        FS_CUDA(cudaEventRecord(freed[b], copy_stream));
                        FS_CUDA(cudaEventRecord(landed, copy_stream));
                        FS_CUDA(cudaStreamWaitEvent(ds->stream, landed, 0));
                        scan_rows(ds, r0, r1, c == 0, c == s_chunks - 1);
                    }
                    // the staging blocks go back to the pool when this scope ends: their DMAs must be over
                    FS_CUDA(cudaStreamSynchronize(copy_stream));
                } catch (...) {
                    cudaStreamSynchronize(copy_stream);
                    for (auto e : freed)
                        if (e) cudaEventDestroy(e);
                    if (landed) cudaEventDestroy(landed);
                    throw;
                }
                for (auto e : freed)
                    if (e) cudaEventDestroy(e);
                cudaEventDestroy(landed);
            }
            finish_create(ds);
        } catch (...) {
            cudaStreamSynchronize(copy_stream);
            for (auto e : done)
                if (e) cudaEventDestroy(e);
            cudaStreamDestroy(copy_stream);
            throw;
        }
        for (auto e : done)
            if (e) cudaEventDestroy(e);
        cudaStreamDestroy(copy_stream);
        *out = owner.release();
        return FS_OK;
    });
}

int fs_dataset_create_device(fs_dataset **out, const void *x_dev, int dtype, int64_t n, int64_t p,
                             int64_t row_stride_elems, const int32_t *y_enc, int32_t n_classes, int32_t device,
                             void *stream) {
    return api_call("fs_dataset_create_device", [&] {
        FS_REQUIRE(out && x_dev, FS_ERR_INVALID, "fs_dataset_create_device: null pointer");
        std::unique_ptr<fs_dataset> owner(create_common(dtype, n, p, row_stride_elems, y_enc, n_classes, device, stream));
        fs_dataset *ds = owner.get();
        ds->x = x_dev;
        ds->ldx = row_stride_elems;
        prepare_create(ds, y_enc);
        scan_rows(ds, 0, n, true, true);
        finish_create(ds);
        *out = owner.release();
        return FS_OK;
    });
}

int fs_dataset_column_stats(const fs_dataset *ds, double *col_min, double *col_max, int32_t *n_distinct) {
    if (!ds) {
        set_error("fs_dataset_column_stats: null data set");
        return FS_ERR_INVALID;
    }
    if (col_min) memcpy(col_min, ds->cmin.data(), ds->p * sizeof(double));
    if (col_max) memcpy(col_max, ds->cmax.data(), ds->p * sizeof(double));
    if (n_distinct) memcpy(n_distinct, ds->cnt.data(), ds->p * sizeof(int32_t));
    return FS_OK;
}

int fs_dataset_set_features(fs_dataset *ds, const uint8_t *is_discrete, const float *recip, int arith) {
    if (!ds || !is_discrete || !recip || (arith != FS_ARITH_F32 && arith != FS_ARITH_F64)) {
        set_error("fs_dataset_set_features: invalid argument");
        return FS_ERR_INVALID;
    }
    // the same typing again (a second fit-like pass over a resident data set): the per-column decisions,
    // the ownership bounds and the cached column lists stay; the GPU-side working set is still rebuilt
    const bool same = ds->have_features && ds->arith == arith && (int64_t)ds->is_discrete.size() == ds->p &&
                      memcmp(ds->is_discrete.data(), is_discrete, ds->p) == 0 &&
                      memcmp(ds->recip.data(), recip, ds->p * sizeof(float)) == 0;
    if (same) {
        forget_derived(ds, true, false);
        return FS_OK;
    }
    ds->is_discrete.assign(is_discrete, is_discrete + ds->p);
    ds->recip.assign(recip, recip + ds->p);
    ds->arith = arith;
    // per-column path of the scoring pipeline, decided once (build_lists reads one byte per column)
    ds->col_info.resize(ds->p);
    const bool byte_input = ds->dtype == FS_U8 || ds->dtype == FS_I8;
    for (int64_t f = 0; f < ds->p; ++f) {
        unsigned ci = kColContinuous;
        if (is_discrete[f]) {
            const int v = ds->cnt[f];
            if (v == 1) {
                ci = kColConst;
            } else if (v <= FS_DISTINCT_CAP) {
                ci = kColTensor | ((unsigned)(v - 1) << 4);
                // one-byte integer input whose V distinct values span exactly 0..V-1: the value is its own code
                if (byte_input && ds->cmin[f] == 0.0 && ds->cmax[f] == (double)(v - 1)) ci |= kColIdent;
            } else {
                ci = kColCompare;
            }
        }
        ds->col_info[f] = (uint8_t)ci;
    }
    ds->have_features = true;
    forget_derived(ds, true, true);
    return FS_OK;
}

int fs_dataset_row_order(const fs_dataset *ds, int64_t *perm_out) {
    if (!ds || !perm_out) {
        set_error("fs_dataset_row_order: invalid argument");
        return FS_ERR_INVALID;
    }
    memcpy(perm_out, ds->perm.data(), ds->n * sizeof(int64_t));
    return FS_OK;
}

int fs_dataset_attach_comm(fs_dataset *ds, fs_comm *comm, const int64_t *row_starts) {
    return api_call("fs_dataset_attach_comm", [&] {
        FS_REQUIRE(ds, FS_ERR_INVALID, "fs_dataset_attach_comm: null data set");
        if (comm == nullptr || comm->world <= 1) {         // detach: plain single-rank behaviour
            ds->comm = nullptr;
            ds->peer_slab = nullptr;
            forget_derived(ds, false, true);
            return FS_OK;
        }
        FS_REQUIRE(row_starts, FS_ERR_INVALID, "fs_dataset_attach_comm: row_starts missing");
        FS_REQUIRE(comm->connected, FS_ERR_STATE, "fs_dataset_attach_comm: the communicator is not connected");
        FS_REQUIRE(comm->device == ds->device, FS_ERR_INVALID, "fs_dataset_attach_comm: communicator on device %d, data set on %d",
                   comm->device, ds->device);
        const int world = comm->world, rank = comm->rank;
        FS_REQUIRE(row_starts[0] == 0 && row_starts[world] == ds->n, FS_ERR_INVALID,
                   "fs_dataset_attach_comm: row_starts must run from 0 to n");
        DistPeers pr{};
        pr.world = world;
        pr.rank = rank;
        int32_t sb = 0;
        int64_t max_shard = 0;
        for (int r = 0; r <= world; ++r) {
            if (r < world) {
                FS_REQUIRE(row_starts[r] < row_starts[r + 1] && (row_starts[r] & 3) == 0, FS_ERR_INVALID,
                           "fs_dataset_attach_comm: row_starts must be strictly ascending multiples of 4 (no empty shard)");
                max_shard = std::max<int64_t>(max_shard, row_starts[r + 1] - row_starts[r]);
            }
            pr.starts[r] = row_starts[r];
            pr.sb_base[r] = sb;
            if (r < world) sb += (int32_t)ceil_div(row_starts[r + 1] - row_starts[r], 256);
        }
        // the layout every rank computes from (n, p, world) alone; X lives in the arena only for data
        // sets created by fs_dataset_create_group (then ds->x already points there)
        const size_t es = dtype_size(ds->dtype);
        const bool x_in_arena = ds->x_in_arena;
        const GroupLayout L = group_layout(ds->n, ds->p, ceil_div(ds->n, world) + kShardSlack, world,
                                           x_in_arena ? (size_t)ds->n * ds->ldx * es : 0);
        FS_REQUIRE(max_shard <= ceil_div(ds->n, world) + kShardSlack, FS_ERR_INVALID,
                   "fs_dataset_attach_comm: shards must be balanced (largest %lld rows)", (long long)max_shard);
        FS_REQUIRE(L.total <= comm->arena_bytes, FS_ERR_INVALID,
                   "fs_dataset_attach_comm: arena of %llu bytes is smaller than the %llu this data set needs",
                   (unsigned long long)comm->arena_bytes, (unsigned long long)L.total);
        ds->glayout = L;
        for (int r = 0; r < world; ++r)
            pr.slab[r] = reinterpret_cast<int32_t *>(reinterpret_cast<char *>(comm->peers.hdr[r]) + L.off_slab);
        ds->peers = pr;
        ds->comm = comm;
        ds->peer_slab = pr.slab[rank];
        forget_derived(ds, false, true);          // the accumulation shares changed: cached column lists are stale
        return FS_OK;
    });
}

// Sharded upload: this rank copies rows [n * rank / world, n * (rank + 1) / world) of the host matrix into
// the X region of its arena, stores them into every peer's arena over NVLink, and after a device-side
// barrier every rank holds all of X having moved 1/world of it over PCIe.
int fs_dataset_create_group(fs_dataset **out, fs_comm *comm, const void *x, int dtype, int64_t n, int64_t p,
                            int64_t row_stride_elems, const int32_t *y_enc, int32_t n_classes, void *stream) {
    return api_call("fs_dataset_create_group", [&] {
        FS_REQUIRE(out && x && comm, FS_ERR_INVALID, "fs_dataset_create_group: null pointer");
        FS_REQUIRE(comm->connected, FS_ERR_STATE, "fs_dataset_create_group: the communicator is not connected");
        std::unique_ptr<fs_dataset> owner(create_common(dtype, n, p, row_stride_elems, y_enc, n_classes, comm->device, stream));
        fs_dataset *ds = owner.get();
        const size_t es = dtype_size(dtype);
        ds->ldx = round_up(p, 16 / (int64_t)es > 0 ? 16 / (int64_t)es : 1);
        const int world = comm->world, rank = comm->rank;
        const GroupLayout L = group_layout(n, p, ceil_div(n, world) + kShardSlack, world, (size_t)n * ds->ldx * es);
        FS_REQUIRE(L.total <= comm->arena_bytes, FS_ERR_INVALID,
                   "fs_dataset_create_group: arena of %llu bytes is smaller than the %llu this data set needs",
                   (unsigned long long)comm->arena_bytes, (unsigned long long)L.total);
        char *xa = static_cast<char *>(comm->arena) + L.off_x;
        ds->x = xa;
        ds->x_in_arena = true;
        const int64_t lo = n * rank / world, hi = n * (rank + 1) / world;
        cudaStream_t st = ds->stream;
        if (hi > lo)
            FS_CUDA(cudaMemcpy2DAsync(xa + (size_t)lo * ds->ldx * es, ds->ldx * es,
                                      static_cast<const char *>(x) + (size_t)lo * row_stride_elems * es,
                                      row_stride_elems * es, p * es, hi - lo, cudaMemcpyHostToDevice, st));
        prepare_create(ds, y_enc);          // host work (class sort) overlaps the copy
        int launches = 0;
        if (hi > lo && world > 1) comm_push(comm, L.off_x + (size_t)lo * ds->ldx * es, (size_t)(hi - lo) * ds->ldx * es, st, &launches);
        comm_barrier(comm, st, &launches);
        scan_rows(ds, 0, n, true, true);
        finish_create(ds);
        comm_check(comm);
        *out = owner.release();
        return FS_OK;
    });
}

int fs_dataset_destroy(fs_dataset *ds) {
    if (!ds) return FS_OK;
    cudaSetDevice(ds->device);
    cudaStreamSynchronize(ds->stream);
    alloc_stream() = ds->stream;
    delete ds;
    return FS_OK;
}

}  // extern "C"
