// multi.cu -- several GPUs from ONE process through the C ABI (fs_multi_*): one host thread per GPU,
// each driving its own rank of a multi-GPU group (comm.cu) whose arenas are mapped through peer
// access.  What `MultiSURF(backend='gpu').fit` uses when FASTSELECT_B200_GPUS > 1: no torchrun, no
// torch, no NCCL -- the exchanges are stores into the peers' arenas from the library's own kernels.
// The reference has no multi-GPU path (SURVEY.md 8e).
#include <algorithm>
#include <functional>
#include <map>
#include <mutex>
#include <string>
#include <thread>

#include "common.cuh"

struct fs_multi {
    int world = 0;
    std::vector<int> devices;
    std::vector<fs_comm *> comms;          // owned by the process-wide cache below, not by this object
    std::vector<fs_dataset *> sets;
    std::vector<cudaStream_t> streams;
    std::vector<int64_t> starts;           // [world + 1] shard starts (internal row order)
    std::vector<fs::DevBuf<double> *> outs;  // per-rank device result (ranks > 0)
    int64_t n = 0, p = 0;
};

namespace fs {
namespace {

// communicators (arenas, peer mappings) are kept for the life of the process, per device list:
// allocating gigabyte arenas and enabling peer access cost far more than a fit
std::mutex g_multi_mu;
std::map<std::string, std::vector<fs_comm *>> g_comm_cache;
std::map<std::string, std::vector<cudaStream_t>> g_stream_cache;

struct RankError {
    int code = FS_OK;
    std::string msg;
};

// run fn(rank) on one host thread per rank; the first failure (lowest rank) is re-raised on the caller
void run_ranks(int world, const std::function<int(int)> &fn) {
    std::vector<RankError> errs(world);
    std::vector<std::thread> th;
    th.reserve(world);
    for (int r = 0; r < world; ++r)
        th.emplace_back([&, r]() {
            const std::string name = "rank " + std::to_string(r);
            const int rc = api_call(name.c_str(), [&] { return fn(r); });
            errs[r].code = rc;
            if (rc != FS_OK) errs[r].msg = get_error();
        });
    for (auto &t : th) t.join();
    // a rank that failed leaves the others waiting at their next barrier until it times out: report the
    // root cause (the first error that is not a timeout) with every failing rank's message
    int first = -1;
    std::string all;
    for (int r = 0; r < world; ++r)
        if (errs[r].code != FS_OK) {
            if (first < 0 || (errs[first].code == FS_ERR_TIMEOUT && errs[r].code != FS_ERR_TIMEOUT)) first = r;
            all += (all.empty() ? "" : " | ") + std::string("rank ") + std::to_string(r) + ": " + errs[r].msg;
        }
    if (first >= 0) {
        set_error("%s", all.c_str());
        throw Fail{errs[first].code};
    }
}

std::string key_of(const std::vector<int> &devices) {
    std::string k;
    for (int d : devices) k += std::to_string(d) + ",";
    return k;
}

}  // namespace
}  // namespace fs

using namespace fs;

extern "C" {

int fs_multi_create(fs_multi **out, const void *x, int dtype, int64_t n, int64_t p, int64_t row_stride_elems,
                    const int32_t *y_enc, int32_t n_classes, const int32_t *devices, int32_t n_devices) {
    fs_multi *m = nullptr;
    const int rc = api_call("fs_multi_create", [&] {
        FS_REQUIRE(out && x && devices, FS_ERR_INVALID, "fs_multi_create: null pointer");
        FS_REQUIRE(n_devices >= 1 && n_devices <= kMaxRanks, FS_ERR_INVALID, "fs_multi_create: 1..%d devices", kMaxRanks);
        FS_REQUIRE(fs_device_count() > 0, FS_ERR_NO_DEVICE, "no usable NVIDIA sm_100 (B200) GPU: this library has no CPU fallback");
        // no empty shard: fewer ranks for very small data sets
        int world = n_devices;
        while (world > 1 && n / world < 8) --world;
        m = new fs_multi();
        m->world = world;
        m->n = n;
        m->p = p;
        m->devices.assign(devices, devices + world);
        for (int a = 0; a < world; ++a)
            for (int b = a + 1; b < world; ++b)
                FS_REQUIRE(m->devices[a] != m->devices[b], FS_ERR_INVALID, "fs_multi_create: device %d listed twice", m->devices[a]);
        m->sets.assign(world, nullptr);
        m->outs.assign(world, nullptr);
        const std::string key = key_of(m->devices);
        {
            std::lock_guard<std::mutex> lk(g_multi_mu);
            auto it = g_comm_cache.find(key);
            if (it != g_comm_cache.end()) {
                m->comms = it->second;
                m->streams = g_stream_cache[key];
            }
        }
        if (m->comms.empty()) {
            m->comms.assign(world, nullptr);
            m->streams.assign(world, nullptr);
            run_ranks(world, [&](int r) {
                FS_CUDA(cudaSetDevice(m->devices[r]));
                FS_CUDA(cudaStreamCreateWithFlags(&m->streams[r], cudaStreamNonBlocking));
                return fs_comm_create(&m->comms[r], r, world, m->devices[r]);
            });
            std::lock_guard<std::mutex> lk(g_multi_mu);
            g_comm_cache[key] = m->comms;
            g_stream_cache[key] = m->streams;
        }
        // arenas: grown when this data set needs more; any change means mapping the peers again
        const uint64_t need = fs_comm_required_bytes(n, p, dtype, world, 1);
        std::vector<int32_t> changed(world, 0);
        run_ranks(world, [&](int r) { return fs_comm_reserve(m->comms[r], need, nullptr, &changed[r]); });
        bool reconnect = false;
        for (int r = 0; r < world; ++r) reconnect = reconnect || changed[r] || !fs_comm_connected(m->comms[r]);
        if (reconnect) {
            std::vector<void *> ptrs(world);
            for (int r = 0; r < world; ++r) ptrs[r] = fs_comm_arena(m->comms[r]);
            run_ranks(world, [&](int r) { return fs_comm_connect(m->comms[r], nullptr, ptrs.data()); });
        }
        // (the join above is the host-level barrier fs_comm_connect asks for)
        run_ranks(world, [&](int r) {
            if (world == 1)
                return fs_dataset_create(&m->sets[r], x, dtype, n, p, row_stride_elems, y_enc, n_classes, m->devices[r], m->streams[r]);
            return fs_dataset_create_group(&m->sets[r], m->comms[r], x, dtype, n, p, row_stride_elems, y_enc, n_classes,
                                           m->streams[r]);
        });
        // balanced shards of the (class-sorted) target rows: whole super-blocks of 256 rows when every rank gets at
        // least four of them (the distance GEMM works in such blocks; see _shard.py::group_shard_starts), else
        // starts that are multiples of 4
        m->starts.assign(world + 1, n);
        const int64_t blocks = ceil_div(n, 256);
        for (int r = 0; r < world; ++r) {
            if (blocks >= 4 * (int64_t)world) {
                const int64_t base = blocks / world, extra = blocks % world;
                m->starts[r] = 256 * (r * base + std::max<int64_t>(0, r - (world - extra)));   // the last ranks take the odd blocks
            } else {
                const int64_t base = n / world, extra = n % world;
                m->starts[r] = (r * base + std::min<int64_t>(r, extra)) / 4 * 4;
            }
        }
        if (world > 1) run_ranks(world, [&](int r) { return fs_dataset_attach_comm(m->sets[r], m->comms[r], m->starts.data()); });
        *out = m;
        return FS_OK;
    });
    if (rc != FS_OK && m) {
        for (auto *ds : m->sets) fs_dataset_destroy(ds);
        delete m;
    }
    return rc;
}

int fs_multi_world(const fs_multi *m) { return m ? m->world : 0; }

int fs_multi_column_stats(const fs_multi *m, double *col_min, double *col_max, int32_t *n_distinct) {
    if (!m || m->sets.empty()) {
        set_error("fs_multi_column_stats: null handle");
        return FS_ERR_INVALID;
    }
    return fs_dataset_column_stats(m->sets[0], col_min, col_max, n_distinct);      // every rank scanned all of X
}

int fs_multi_set_features(fs_multi *m, const uint8_t *is_discrete, const float *recip, int arith) {
    if (!m) {
        set_error("fs_multi_set_features: null handle");
        return FS_ERR_INVALID;
    }
    for (auto *ds : m->sets) {
        const int rc = fs_dataset_set_features(ds, is_discrete, recip, arith);
        if (rc != FS_OK) return rc;
    }
    return FS_OK;
}

int fs_multi_score(fs_multi *m, int algo, int use_star, int32_t k, const float *class_probs, const int64_t *feat_idx,
                   int64_t n_kept, double *wsum_out, fs_stats *stats) {
    return api_call("fs_multi_score", [&] {
        FS_REQUIRE(m && wsum_out, FS_ERR_INVALID, "fs_multi_score: null pointer");
        if (!feat_idx) n_kept = m->p;
        const int world = m->world;
        run_ranks(world, [&](int r) {
            if (r == 0)
                return fs_score(m->sets[0], algo, use_star, k, class_probs, feat_idx, n_kept, m->starts[0], m->starts[1],
                                wsum_out, 0, stats);
            // the other ranks end up with the same complete vector on their device; it is not copied back
            FS_CUDA(cudaSetDevice(m->devices[r]));
            alloc_stream() = m->streams[r];
            if (!m->outs[r]) m->outs[r] = new DevBuf<double>();
            m->outs[r]->reserve((size_t)n_kept);
            return fs_score(m->sets[r], algo, use_star, k, class_probs, feat_idx, n_kept, m->starts[r], m->starts[r + 1],
                            m->outs[r]->ptr, 1, nullptr);
        });
        return FS_OK;
    });
}

int fs_multi_destroy(fs_multi *m) {
    if (!m) return FS_OK;
    for (int r = 0; r < m->world; ++r) {
        if (m->outs[r]) {
            cudaSetDevice(m->devices[r]);
            alloc_stream() = m->streams[r];
            delete m->outs[r];
        }
        fs_dataset_destroy(m->sets[r]);
    }
    delete m;       // communicators and streams stay in the process-wide cache
    return FS_OK;
}

}  // extern "C"
