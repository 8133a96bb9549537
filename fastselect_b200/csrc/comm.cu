// comm.cu -- the multi-GPU group of one scoring job: every rank's exchange arena (one plain
// cudaMalloc block per rank, mapped into the peers through CUDA IPC or, inside one process, through
// peer access), a device-side barrier over flags in those arenas, and the arena layout of a data set.
//
// The reference has no multi-GPU path (SURVEY.md 8e); its unit of parallelism is the target instance
// (MultiSURF.py:174).  Here the ranks exchange, all by stores into the peers' arenas over NVLink:
//   * the transposed tiles of the symmetric distance GEMM (tc_dist.cu),
//   * the neighbour masks / row constants of their target rows (so that every rank can contract ITS
//     share of the one-hot rows against the masks of ALL targets: feature-sharded accumulation),
//   * their slice of the weight vector (summed in rank order: bitwise identical on every rank),
//   * and, at upload time, their 1/G of the raw matrix.
// No host synchronisation separates the steps: a barrier is one tiny kernel per rank that publishes
// an epoch to every peer and spins until every peer's epoch arrived (bounded: FS_B200_BARRIER_TIMEOUT_S,
// default 20 s, then an error flag is raised instead of hanging the GPUs).
#include <algorithm>
#include <condition_variable>
#include <cstring>
#include <map>
#include <mutex>

#include "common.cuh"

namespace fs {

struct HostBarrier {
    std::mutex mu;
    std::condition_variable cv;
    int world = 0, waiting = 0;
    unsigned long long generation = 0;
};

// false on timeout (a rank never arrived)
bool host_barrier_wait(HostBarrier *hb, double timeout_s) {
    std::unique_lock<std::mutex> lk(hb->mu);
    const unsigned long long gen = hb->generation;
    if (++hb->waiting == hb->world) {
        hb->waiting = 0;
        ++hb->generation;
        hb->cv.notify_all();
        return true;
    }
    const bool ok = hb->cv.wait_for(lk, std::chrono::duration<double>(timeout_s), [&] { return hb->generation != gen; });
    if (!ok) --hb->waiting;
    return ok;
}

namespace {
constexpr size_t kAlign = 1024;
size_t align_up(size_t v) { return (v + kAlign - 1) / kAlign * kAlign; }

// host barriers of in-process groups, keyed by rank 0's arena
std::mutex g_hb_mu;
std::map<void *, std::weak_ptr<HostBarrier>> g_host_barriers;

std::mutex g_ipc_mu;
struct IpcEntry {
    char handle[64];
    void *ptr;
};
std::vector<IpcEntry> g_ipc_open;

void *ipc_open(const char *handle_bytes) {
    std::lock_guard<std::mutex> lk(g_ipc_mu);
    for (auto &e : g_ipc_open)
        if (memcmp(e.handle, handle_bytes, 64) == 0) return e.ptr;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle_bytes, sizeof(h));
    void *p = nullptr;
    FS_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    IpcEntry e;
    memcpy(e.handle, handle_bytes, 64);
    e.ptr = p;
    g_ipc_open.push_back(e);
    return p;
}
void ipc_close(void *ptr) {
    std::lock_guard<std::mutex> lk(g_ipc_mu);
    for (size_t i = 0; i < g_ipc_open.size(); ++i)
        if (g_ipc_open[i].ptr == ptr) {
            cudaIpcCloseMemHandle(ptr);
            g_ipc_open.erase(g_ipc_open.begin() + i);
            return;
        }
}
}  // namespace

GroupLayout group_layout(int64_t n, int64_t p, int64_t max_shard_rows, int world, size_t x_bytes) {
    GroupLayout L{};
    const int64_t ldn = round_up(n, 128);
    size_t o = align_up(sizeof(CommHeader));
    L.off_slab = o;
    o += align_up((size_t)round_up(std::max<int64_t>(max_shard_rows, 1), 128) * ldn * sizeof(int32_t));
    // padding behind each mask: the accumulation kernels' mask box may reach into it
    L.off_mask_h = o;
    o += align_up((size_t)(ldn + kAccumMaskPadRows) * (ldn / 2));
    L.off_mask_m = o;
    o += align_up((size_t)(ldn + kAccumMaskPadRows) * (ldn / 2));
    L.off_rinfo = o;
    o += align_up((size_t)ldn * sizeof(RowInfo));
    L.off_w = o;
    o += align_up((size_t)world * (size_t)p * sizeof(double));
    L.off_x = o;
    o += align_up(x_bytes);
    L.total = o;
    return L;
}

// One warp: lane q < world publishes `epoch` into flags[rank] of peer q's header, then waits until peer
// q's epoch arrived in this rank's own header.  Everything a rank stored into a peer's arena before
// its barrier kernel (earlier kernels of the same stream) is visible to that peer after the barrier.
__global__ void comm_barrier_kernel(CommPeers peers, uint32_t epoch, unsigned long long timeout_ns) {
    const int q = threadIdx.x;
    if (q >= peers.world) return;
    __threadfence_system();
    if (q != peers.rank) {
        volatile uint32_t *dst = &peers.hdr[q]->flags[peers.rank];
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(dst), "r"(epoch) : "memory");
    }
    // after a timeout the epochs are out of step anyway: later barriers of the call do not wait again
    if (q != peers.rank && peers.hdr[peers.rank]->error == 0) {
        const uint32_t *src = &peers.hdr[peers.rank]->flags[q];
        unsigned long long t0;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t0));
        for (;;) {
            uint32_t v;
            asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(src) : "memory");
            // epochs only grow; the comparison is wrap-safe
            if ((int32_t)(v - epoch) >= 0) break;
            unsigned long long t1;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
            if (t1 - t0 > timeout_ns) {
                peers.hdr[peers.rank]->error = 1u + (uint32_t)q;     // which peer never arrived
                break;
            }
            __nanosleep(200);
        }
    }
    __threadfence_system();
}

void comm_barrier(fs_comm *c, cudaStream_t st, int *launches) {
    if (c->world <= 1) return;
    if (c->host_barrier && !host_barrier_wait(c->host_barrier.get(), (double)c->timeout_ns * 1e-9)) {
        c->connected = false;
        FS_REQUIRE(false, FS_ERR_TIMEOUT, "multi-GPU barrier timed out on the host: a rank of this process never joined the call");
    }
    ++c->epoch;
    comm_barrier_kernel<<<1, 32, 0, st>>>(c->peers, c->epoch, c->timeout_ns);
    FS_CUDA(cudaGetLastError());
    if (launches) ++*launches;
    // ... and nobody issues anything further before every rank's barrier kernel is in its queue (a
    // synchronising call in between would order a late barrier kernel behind an early, spinning one)
    if (c->host_barrier && !host_barrier_wait(c->host_barrier.get(), (double)c->timeout_ns * 1e-9)) {
        c->connected = false;
        FS_REQUIRE(false, FS_ERR_TIMEOUT, "multi-GPU barrier timed out on the host: a rank of this process never joined the call");
    }
}

// Raises FS_ERR_TIMEOUT when a barrier of this call gave up (stream must be synchronised).
void comm_check(fs_comm *c) {
    if (c->world <= 1) return;
    uint32_t err = 0;
    FS_CUDA(cudaMemcpy(&err, &c->peers.hdr[c->rank]->error, sizeof(err), cudaMemcpyDeviceToHost));
    if (err != 0) {
        FS_CUDA(cudaMemset(&c->peers.hdr[c->rank]->error, 0, sizeof(err)));
        c->connected = false;      // epochs are out of step now: the group must be connected again
        FS_REQUIRE(false, FS_ERR_TIMEOUT, "multi-GPU barrier timed out waiting for rank %u (a rank failed or left the call)",
                   err - 1u);
    }
}

// dst[peer][off .. off + bytes) = own[off .. off + bytes) for every peer (16-byte aligned)
__global__ void __launch_bounds__(256) comm_push_kernel(CommPeers peers, size_t off, size_t bytes) {
    const size_t n16 = bytes / 16;
    const uint4 *src = reinterpret_cast<const uint4 *>(reinterpret_cast<const char *>(peers.hdr[peers.rank]) + off);
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n16; i += (size_t)gridDim.x * blockDim.x) {
        const uint4 v = src[i];
        for (int q = 0; q < peers.world; ++q)
            if (q != peers.rank) reinterpret_cast<uint4 *>(reinterpret_cast<char *>(peers.hdr[q]) + off)[i] = v;
    }
}

void comm_push(fs_comm *c, size_t off, size_t bytes, cudaStream_t st, int *launches) {
    if (c->world <= 1 || bytes == 0) return;
    FS_REQUIRE(off % 16 == 0 && bytes % 16 == 0, FS_ERR_INVALID, "comm_push: unaligned range");
    const size_t n16 = bytes / 16;
    const unsigned grid = (unsigned)std::min<size_t>(148 * 8, (n16 + 255) / 256);
    comm_push_kernel<<<grid, 256, 0, st>>>(c->peers, off, bytes);
    FS_CUDA(cudaGetLastError());
    if (launches) ++*launches;
}

}  // namespace fs

using namespace fs;

extern "C" {

int fs_comm_create(fs_comm **out, int32_t rank, int32_t world, int32_t device) {
    return api_call("fs_comm_create", [&] {
        FS_REQUIRE(out, FS_ERR_INVALID, "fs_comm_create: null pointer");
        FS_REQUIRE(world >= 1 && world <= kMaxRanks && rank >= 0 && rank < world, FS_ERR_INVALID,
                   "fs_comm_create: bad rank/world %d/%d (at most %d ranks)", rank, world, kMaxRanks);
        int major = 0;
        FS_REQUIRE(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device) == cudaSuccess && major == 10,
                   FS_ERR_NO_DEVICE, "fs_comm_create: device %d is not a usable sm_100 GPU", device);
        fs_comm *c = new fs_comm();
        c->rank = rank;
        c->world = world;
        c->device = device;
        c->timeout_ns = 20ull * 1000000000ull;
        if (const char *e = getenv("FS_B200_BARRIER_TIMEOUT_S")) c->timeout_ns = (unsigned long long)(atof(e) * 1e9);
        c->peers.rank = rank;
        c->peers.world = world;
        *out = c;
        return FS_OK;
    });
}

int fs_comm_reserve(fs_comm *c, uint64_t bytes, void *ipc_handle_out, int32_t *changed_out) {
    return api_call("fs_comm_reserve", [&] {
        FS_REQUIRE(c, FS_ERR_INVALID, "fs_comm_reserve: null communicator");
        FS_CUDA(cudaSetDevice(c->device));
        bool changed = false;
        if (c->arena == nullptr || c->arena_bytes < bytes) {
            if (c->arena) {
                FS_CUDA(cudaDeviceSynchronize());
                cudaFree(c->arena);
                c->arena = nullptr;
            }
            // plain cudaMalloc: stream-ordered pool memory cannot be exported through CUDA IPC
            const size_t want = (size_t)bytes + (size_t)bytes / 8;          // slack: growing data sets of similar size reuse it
            FS_CUDA(cudaMalloc(&c->arena, want));
            c->arena_bytes = want;
            c->connected = false;
            changed = true;
        }
        if (ipc_handle_out) {
            cudaIpcMemHandle_t h;
            FS_CUDA(cudaIpcGetMemHandle(&h, c->arena));
            static_assert(sizeof(h) == 64, "CUDA IPC handle size");
            memcpy(ipc_handle_out, &h, sizeof(h));
        }
        if (changed_out) *changed_out = changed ? 1 : 0;
        return FS_OK;
    });
}

void *fs_comm_arena(fs_comm *c) { return c ? c->arena : nullptr; }
uint64_t fs_comm_arena_bytes(fs_comm *c) { return c ? c->arena_bytes : 0; }
int fs_comm_connected(fs_comm *c) { return c && c->connected ? 1 : 0; }

int fs_comm_connect(fs_comm *c, const void *ipc_handles, void *const *raw_ptrs) {
    return api_call("fs_comm_connect", [&] {
        FS_REQUIRE(c && c->arena, FS_ERR_STATE, "fs_comm_connect: reserve the arena first");
        FS_REQUIRE(ipc_handles || raw_ptrs || c->world == 1, FS_ERR_INVALID, "fs_comm_connect: no handles");
        FS_CUDA(cudaSetDevice(c->device));
        for (int q = 0; q < c->world; ++q) {
            void *p = nullptr;
            if (q == c->rank) {
                p = c->arena;
            } else if (raw_ptrs) {
                p = raw_ptrs[q];
                // same process: the peer's allocation is reachable once peer access is on (a no-op on one device)
                cudaPointerAttributes at{};
                if (cudaPointerGetAttributes(&at, p) == cudaSuccess && at.device != c->device) {
                    cudaError_t e = cudaDeviceEnablePeerAccess(at.device, 0);
                    if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) FS_CUDA(e);
                    cudaGetLastError();
                }
            } else {
                void *old = c->opened[q];
                p = ipc_open(static_cast<const char *>(ipc_handles) + (size_t)q * 64);
                if (old && old != p) ipc_close(old);       // the peer re-allocated its arena
                c->opened[q] = p;
            }
            FS_REQUIRE(p != nullptr, FS_ERR_INVALID, "fs_comm_connect: rank %d has no arena", q);
            c->peers.hdr[q] = static_cast<CommHeader *>(p);
        }
        // ranks of one process (raw pointers) share a host barrier, found through rank 0's arena
        c->host_barrier.reset();
        if (raw_ptrs && c->world > 1) {
            std::lock_guard<std::mutex> lk(g_hb_mu);
            std::shared_ptr<HostBarrier> hb = g_host_barriers[raw_ptrs[0]].lock();
            if (!hb || hb->world != c->world) {
                hb = std::make_shared<HostBarrier>();
                hb->world = c->world;
                g_host_barriers[raw_ptrs[0]] = hb;
            }
            c->host_barrier = hb;
        }
        // epochs restart: every rank clears its own header, and the caller runs a host-level barrier
        // (all ranks connected) before the first collective call
        FS_CUDA(cudaMemset(c->arena, 0, sizeof(CommHeader)));
        FS_CUDA(cudaDeviceSynchronize());
        c->epoch = 0;
        c->connected = true;
        return FS_OK;
    });
}

int fs_comm_destroy(fs_comm *c) {
    if (!c) return FS_OK;
    cudaSetDevice(c->device);
    cudaDeviceSynchronize();
    for (int q = 0; q < kMaxRanks; ++q)
        if (c->opened[q]) ipc_close(c->opened[q]);
    if (c->arena) cudaFree(c->arena);
    delete c;
    return FS_OK;
}

uint64_t fs_comm_required_bytes(int64_t n, int64_t p, int32_t dtype, int32_t world, int32_t with_x) {
    if (n < 1 || p < 1 || world < 1) return 0;
    size_t es = dtype == FS_F32 ? 4 : dtype == FS_F64 ? 8 : 1;
    const int64_t ldx = round_up(p, 16 / (int64_t)es);
    const int64_t shard = ceil_div(n, world) + kShardSlack;
    return group_layout(n, p, shard, world, with_x ? (size_t)n * ldx * es : 0).total;
}

}  // extern "C"
