// score.cu -- the scoring pipeline behind fs_score / fs_debug_rows:
//   working set (active columns) -> distance slab for a chunk of target rows
//   -> neighbour selection -> weight accumulation -> fixed-order reduction.
// Replaces the reference host callers _multisurf_gpu_host_caller
// (MultiSURF.py:147-162), _surf_gpu_host_caller (SURF.py:117-128) and
// _relieff_gpu_host_caller (ReliefF.py:127-134), minus their final "/ n_samples".
#include <algorithm>
#include <chrono>
#include <cstring>

#include "common.cuh"

namespace fs {

struct DebugOut {
    double *dist = nullptr;    // [nt, n] original sample order
    double *thresh = nullptr;  // [nt]
    int8_t *mask = nullptr;    // [nt, n]
};

__global__ void count_selected_kernel(const RowInfo *rinfo, int64_t R, unsigned long long *out) {
    unsigned long long s = 0;
    for (int64_t r = blockIdx.x * blockDim.x + threadIdx.x; r < R; r += (int64_t)gridDim.x * blockDim.x)
        s += (unsigned long long)(rinfo[r].n_hit + rinfo[r].n_miss + rinfo[r].n_far_hit + rinfo[r].n_far_miss);
    atomicAdd(out, s);
}

// wsum[c] = sum over ranks q (in rank order: bitwise identical everywhere) of slots[q * stride + c]
__global__ void __launch_bounds__(256) sum_rank_slots_kernel(const double *__restrict__ slots, int world, int64_t stride,
                                                             int64_t n_kept, double *__restrict__ wsum) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= n_kept) return;
    double s = 0.0;
    for (int q = 0; q < world; ++q) s += slots[(int64_t)q * stride + c];
    wsum[c] = s;
}

// target rows per chunk of the distance slab; have_general / have_tensor: which slabs exist
static int64_t chunk_rows(bool have_general, bool have_tensor, int64_t ldn, int algo) {
    int64_t budget_mb = 6144;
    if (const char *e = getenv("FS_B200_CHUNK_MB")) budget_mb = std::max<int64_t>(16, atoll(e));
    int64_t per_row = ldn * ((have_general ? 8 : 0) + (have_tensor ? 4 : 0) + 1 + (have_tensor ? 2 : 0) + (algo == FS_RELIEFF ? 8 : 0));
    int64_t rows = budget_mb * (1LL << 20) / std::max<int64_t>(1, per_row);
    rows = std::max<int64_t>(128, rows / 128 * 128);
    return rows;
}

static void run_pipeline(fs_dataset *ds, int algo, int use_star, int32_t k, const float *class_probs,
                         const int64_t *feat_idx, int64_t n_kept, const std::vector<int64_t> &targets,
                         bool contiguous, double *d_wsum, DebugOut *dbg, fs_stats *stats) {
    FS_REQUIRE(ds->have_features, FS_ERR_STATE, "fs_score: call fs_dataset_set_features first");
    FS_REQUIRE(algo == FS_RELIEFF || algo == FS_SURF || algo == FS_MULTISURF, FS_ERR_INVALID, "unknown algo %d", algo);
    FS_REQUIRE(n_kept >= 1, FS_ERR_INVALID, "fs_score: n_kept must be >= 1");
    if (algo == FS_RELIEFF) {
        FS_REQUIRE(k >= 1 && k < ds->n, FS_ERR_INVALID, "ReliefF: k=%d must be in [1, n-1]", k);
        FS_REQUIRE(class_probs != nullptr, FS_ERR_INVALID, "ReliefF: class_probs missing");
    }
    FS_CUDA(cudaSetDevice(ds->device));
    cudaStream_t st = ds->stream;
    alloc_stream() = st;
    const int64_t n = ds->n;
    int launches = 0;
    double ops_dist = 0.0, ops_accum = 0.0;
    PhaseTimer timer(stats != nullptr, st);

    const int64_t ldn = round_up(n, 128);
    // Multi-GPU group call: this rank scores exactly its shard of the target rows, every rank does the
    // same with the same arguments, and the shard fits one chunk on every rank (the decision must be
    // identical everywhere: it is taken for the LARGEST shard with the most demanding slab set).  Then
    // distances are computed symmetrically across ranks, the accumulation may be sharded by one-hot
    // columns, and wsum_out receives the COMPLETE sums on every rank.
    fs_comm *comm = ds->comm;
    int64_t max_shard = 0;
    for (int q = 0; ds->peers_on && q < ds->peers.world; ++q)
        max_shard = std::max<int64_t>(max_shard, ds->peers.starts[q + 1] - ds->peers.starts[q]);
    const bool group_call = ds->peers_on && comm != nullptr && comm->world > 1 && contiguous && dbg == nullptr &&
                            targets[0] == ds->peers.starts[ds->peers.rank] &&
                            (int64_t)targets.size() == ds->peers.starts[ds->peers.rank + 1] - ds->peers.starts[ds->peers.rank] &&
                            round_up(max_shard, 128) <= chunk_rows(true, true, ldn, algo);
    if (group_call) FS_REQUIRE(comm->connected, FS_ERR_STATE, "fs_score: the multi-GPU group is not connected");
    const char *env_fs = getenv("FS_B200_FEATURE_SHARD");
    const bool want_split = group_call && algo != FS_RELIEFF && !(env_fs && env_fs[0] == '0');
    // the one-hot distance slab of a contiguous target range that fits one chunk is kept between
    // calls: TuRF's next iteration subtracts the removed columns instead of recomputing it
    // (with peers configured the decision is taken for the largest shard, so that all ranks agree)
    const int64_t cache_rows = std::max<int64_t>((int64_t)targets.size(), max_shard);
    const bool slab_cacheable = contiguous && dbg == nullptr && round_up(cache_rows, 128) <= chunk_rows(true, true, ldn, algo);
    if (!slab_cacheable) ds->dd_valid = false;
    timer.begin(&fs_stats::ms_gather);
    const auto prep0 = std::chrono::steady_clock::now();
    build_workset(ds, feat_idx, n_kept, algo == FS_RELIEFF, targets[0], (int64_t)targets.size(),
                  contiguous, slab_cacheable, want_split, group_call, true, &launches);
    const double ms_prep = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - prep0).count();
    timer.end();
    const WorkSet &ws = ds->ws;
    const bool fshard = group_call && ws.acc_split && ws.pt > 0;

    const int64_t Rmax = std::min<int64_t>(chunk_rows(ws.pg > 0, ws.pt > 0, ldn, algo), round_up((int64_t)targets.size(), 128));
    if (ws.pg > 0) ds->Dc.reserve((size_t)Rmax * ldn);
    // the one-hot distance slab: this rank's slab inside its exchange arena for a group call (the
    // peers store their mirrored tiles into it), else the data set's own buffer
    int32_t *Dd = nullptr;
    if (ws.pt > 0) {
        if (group_call) {
            Dd = ds->peer_slab;
        } else {
            ds->Dd.reserve((size_t)Rmax * ldn);
            Dd = ds->Dd.ptr;
        }
        if (ds->dd_buf != Dd) {
            // the cached slab lives in the other buffer: recompute in full (the working set may
            // have been built for an incremental update)
            if (ds->dd_valid && ws.dist_mode != kDistFull) {
                ds->dd_valid = false;
                ds->ws.valid = false;
                build_workset(ds, feat_idx, n_kept, algo == FS_RELIEFF, targets[0], (int64_t)targets.size(),
                              contiguous, slab_cacheable, want_split, group_call, true, &launches);
            }
            ds->dd_valid = false;
        }
    }
    ds->sel.reserve((size_t)Rmax * ldn);
    const bool use_masks = ws.pt > 0 && algo != FS_RELIEFF;
    // neighbour masks and row constants: inside a group call they live in the arena at the rows of this
    // rank's shard (with a sharded accumulation every rank then receives every other rank's rows)
    int8_t *mask_h = nullptr, *mask_m = nullptr;
    RowInfo *rinfo_buf = nullptr;
    char *arena = group_call ? static_cast<char *>(comm->arena) : nullptr;
    const int64_t shard0 = group_call ? targets[0] : 0;
    if (group_call) {
        mask_h = reinterpret_cast<int8_t *>(arena + ds->glayout.off_mask_h) + (size_t)shard0 * (ldn / 2);
        mask_m = reinterpret_cast<int8_t *>(arena + ds->glayout.off_mask_m) + (size_t)shard0 * (ldn / 2);
        rinfo_buf = reinterpret_cast<RowInfo *>(arena + ds->glayout.off_rinfo) + shard0;
    } else {
        if (use_masks) {
            // rows of ldn / 2 bytes, and the padding the accumulation kernels' mask box may reach into
            ds->maskH.reserve((size_t)(Rmax + kAccumMaskPadRows) * (ldn / 2));
            ds->maskM.reserve((size_t)(Rmax + kAccumMaskPadRows) * (ldn / 2));
            mask_h = ds->maskH.ptr;
            mask_m = ds->maskM.ptr;
        }
        ds->rinfo.reserve(Rmax);
        rinfo_buf = ds->rinfo.ptr;
    }
    // a group call accumulates into this rank's slot of the arena; the slots are summed at the end
    double *acc_out = d_wsum;
    if (group_call) {
        FS_REQUIRE(n_kept <= ds->p, FS_ERR_INVALID, "fs_score: more output columns than the data set has");
        acc_out = reinterpret_cast<double *>(arena + ds->glayout.off_w) + (size_t)comm->rank * ds->p;
    }
    ds->row_ids.reserve(Rmax);
    int32_t nbr_cap = 0;
    if (algo == FS_RELIEFF) {
        nbr_cap = (int32_t)std::min<int64_t>((int64_t)ds->n_classes * k, n);
        ds->nbr_idx.reserve((size_t)Rmax * nbr_cap);
        ds->nbr_w.reserve((size_t)Rmax * nbr_cap);
        ds->nbr_cnt.reserve(Rmax);
        ds->d_class_probs.reserve(ds->n_classes);
        FS_CUDA(cudaMemcpyAsync(ds->d_class_probs.ptr, class_probs, ds->n_classes * sizeof(float),
                                cudaMemcpyHostToDevice, st));
    }
    ds->counters.reserve(1);
    FS_CUDA(cudaMemsetAsync(ds->counters.ptr, 0, sizeof(unsigned long long), st));
    FS_CUDA(cudaMemsetAsync(acc_out, 0, n_kept * sizeof(double), st));

    int n_chunks = 0;
    for (int64_t t0 = 0; t0 < (int64_t)targets.size(); t0 += Rmax) {
        const int64_t R = std::min<int64_t>(Rmax, (int64_t)targets.size() - t0);
        const int64_t *h_ids = targets.data() + t0;
        ++n_chunks;
        FS_CUDA(cudaMemcpyAsync(ds->row_ids.ptr, h_ids, R * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        // target rows of the general matrix: a view for a contiguous range, a gathered copy otherwise
        const char *xa = nullptr;
        if (ws.pg > 0) {
            const size_t row_bytes = (size_t)ws.ldg * ws.elem;
            if (contiguous) {
                xa = ws.xg.ptr + (size_t)h_ids[0] * row_bytes;
            } else {
                ds->xa_gather.reserve((size_t)R * row_bytes);
                for (int64_t r = 0; r < R; ++r)
                    FS_CUDA(cudaMemcpyAsync(ds->xa_gather.ptr + (size_t)r * row_bytes,
                                            ws.xg.ptr + (size_t)h_ids[r] * row_bytes, row_bytes,
                                            cudaMemcpyDeviceToDevice, st));
                xa = ds->xa_gather.ptr;
            }
        }
        // ---- distances
        if (ws.pt > 0 && ws.dist_mode != kDistReuse) {
            ds->dd_valid = false;
            timer.begin(&fs_stats::ms_dist_tensor);
            launch_dist_tensor(ds, ws, h_ids[0], h_ids, ds->row_ids.ptr, contiguous, R, Dd, ldn, st, &launches, &ops_dist);
            timer.end();
            if (ds->last_dist_exchanged) {
                // tiles computed here were also stored into the peers' slabs and theirs into this one:
                // every rank must have finished its distance kernel before anyone selects (device-side
                // barrier over flags in the arenas: no host synchronisation inside the step)
                comm_barrier(comm, st, &launches);
            }
        }
        if (ws.pt > 0 && slab_cacheable) {
            ds->dd_buf = Dd;
            // Dd now holds the mismatch counts of exactly these columns for these target rows
            if (ds->dd_version != ws.lists_version || (int64_t)ds->dd_cols.size() != ws.pt) {
                ds->dd_cols.assign(ws.p_tcol.ptr, ws.p_tcol.ptr + ws.pt);
                ds->dd_version = ws.lists_version;
            }
            ds->dd_r0 = targets[0];
            ds->dd_R = (int64_t)targets.size();
            ds->dd_valid = true;
        }
        if (ws.pg > 0) {
            timer.begin(&fs_stats::ms_dist_general);
            launch_dist_general(ws, xa, R, ws.xg.ptr, n, ds->Dc.ptr, ldn, st, &launches);
            timer.end();
        }
        // ---- neighbour selection
        timer.begin(&fs_stats::ms_select);
        launch_select(ds, algo, use_star, k, ds->row_ids.ptr, R, ws.pg > 0 ? ds->Dc.ptr : nullptr,
                      ws.pt > 0 ? Dd : nullptr, ldn, ds->sel.ptr, use_masks ? mask_h : nullptr,
                      use_masks ? mask_m : nullptr, rinfo_buf, ds->nbr_idx.ptr,
                      ds->nbr_w.ptr, ds->nbr_cnt.ptr, nbr_cap, ds->d_class_probs.ptr, st, &launches);
        if (stats) {
            count_selected_kernel<<<32, 256, 0, st>>>(rinfo_buf, R, ds->counters.ptr);
            ++launches;
        }
        timer.end();
        // ---- accumulation
        if (ws.pt > 0 && fshard) {
            // sharded by one-hot columns: every rank sends the masks / constants of its target rows to all
            // peers, then contracts ITS columns against the masks of ALL n targets (the complete weight of
            // those columns, with the tiling of a single-GPU pass: bitwise the single-GPU result)
            timer.begin(&fs_stats::ms_accum_tensor);
            const size_t mrow = (size_t)(ldn / 2);
            comm_push(comm, ds->glayout.off_mask_h + (size_t)shard0 * mrow, (size_t)R * mrow, st, &launches);
            comm_push(comm, ds->glayout.off_mask_m + (size_t)shard0 * mrow, (size_t)R * mrow, st, &launches);
            comm_push(comm, ds->glayout.off_rinfo + (size_t)shard0 * sizeof(RowInfo), (size_t)R * sizeof(RowInfo), st, &launches);
            comm_barrier(comm, st, &launches);
            if ((int64_t)ds->all_ids_h.size() != n) {
                ds->all_ids_h.resize(n);
                for (int64_t r = 0; r < n; ++r) ds->all_ids_h[r] = r;
                ds->all_ids.alloc(n);
                FS_CUDA(cudaMemcpyAsync(ds->all_ids.ptr, ds->all_ids_h.data(), n * sizeof(int64_t), cudaMemcpyHostToDevice, st));
            }
            launch_accum_tensor(ds, ws, ds->all_ids.ptr, ds->all_ids_h.data(), true, n,
                                reinterpret_cast<const int8_t *>(arena + ds->glayout.off_mask_h),
                                reinterpret_cast<const int8_t *>(arena + ds->glayout.off_mask_m), ldn,
                                reinterpret_cast<const RowInfo *>(arena + ds->glayout.off_rinfo), acc_out, st, &launches,
                                &ops_accum);
            timer.end();
        } else if (ws.pt > 0) {
            timer.begin(&fs_stats::ms_accum_tensor);
            if (algo == FS_RELIEFF)
                launch_relieff_codes(ws, ds->row_ids.ptr, ds->nbr_idx.ptr, ds->nbr_w.ptr, ds->nbr_cnt.ptr, nbr_cap, R,
                                     ds->tpartial, acc_out, st, &launches);
            else
                launch_accum_tensor(ds, ws, ds->row_ids.ptr, h_ids, contiguous, R, mask_h, mask_m, ldn, rinfo_buf,
                                    acc_out, st, &launches, &ops_accum);
            timer.end();
        }
        if (ws.pg > 0) {
            const int64_t n_part = accum_general_partials(ws, R);
            ds->partial.reserve((size_t)n_part * ws.ldg);
            timer.begin(&fs_stats::ms_accum_general);
            if (algo == FS_RELIEFF)
                launch_relieff_gather(ws, n, xa, ds->nbr_idx.ptr, ds->nbr_w.ptr, ds->nbr_cnt.ptr, nbr_cap, R,
                                      ds->partial.ptr, n_part, st, &launches);
            else
                launch_accum_general(ws, n, xa, ds->sel.ptr, ldn, rinfo_buf, R, ds->partial.ptr, n_part, st,
                                     &launches);
            timer.end();
            timer.begin(&fs_stats::ms_reduce);
            launch_reduce_partials(ws, ds->partial.ptr, n_part, acc_out, st, &launches);
            timer.end();
        }
        // ---- parity/debug view of this chunk
        if (dbg) {
            std::vector<double> hd;
            std::vector<int32_t> hdd;
            std::vector<int8_t> hs((size_t)R * ldn);
            std::vector<RowInfo> hr(R);
            FS_CUDA(cudaStreamSynchronize(st));
            if (ws.pg > 0) {
                hd.resize((size_t)R * ldn);
                FS_CUDA(cudaMemcpy(hd.data(), ds->Dc.ptr, hd.size() * sizeof(double), cudaMemcpyDeviceToHost));
            }
            if (ws.pt > 0) {
                hdd.resize((size_t)R * ldn);
                FS_CUDA(cudaMemcpy(hdd.data(), Dd, hdd.size() * sizeof(int32_t), cudaMemcpyDeviceToHost));
            }
            FS_CUDA(cudaMemcpy(hs.data(), ds->sel.ptr, hs.size(), cudaMemcpyDeviceToHost));
            FS_CUDA(cudaMemcpy(hr.data(), rinfo_buf, R * sizeof(RowInfo), cudaMemcpyDeviceToHost));
            for (int64_t r = 0; r < R; ++r) {
                const int64_t t = t0 + r;
                if (dbg->thresh) dbg->thresh[t] = hr[r].thresh;
                for (int64_t j = 0; j < n; ++j) {
                    const int64_t orig = ds->perm[j];
                    if (dbg->dist) {
                        double d = 0.0;
                        if (ws.pg > 0) d += hd[(size_t)r * ldn + j];
                        if (ws.pt > 0) d += (double)hdd[(size_t)r * ldn + j];
                        if (algo != FS_MULTISURF) d = (double)(float)d;   // SURF.py:160, ReliefF.py:155
                        dbg->dist[(size_t)t * n + orig] = (j == h_ids[r]) ? 0.0 : d;
                    }
                    if (dbg->mask) dbg->mask[(size_t)t * n + orig] = hs[(size_t)r * ldn + j];
                }
            }
        }
    }
    if (group_call) {
        // every rank's contribution (its share of the one-hot columns in full, or partial sums over its
        // target rows) goes into its slot of every arena; the slots are added in rank order
        timer.begin(&fs_stats::ms_reduce);
        const size_t slot_bytes = (size_t)round_up(n_kept * (int64_t)sizeof(double), 16);
        comm_push(comm, ds->glayout.off_w + (size_t)comm->rank * ds->p * sizeof(double), slot_bytes, st, &launches);
        comm_barrier(comm, st, &launches);
        sum_rank_slots_kernel<<<(unsigned)ceil_div(n_kept, 256), 256, 0, st>>>(
            reinterpret_cast<const double *>(arena + ds->glayout.off_w), comm->world, ds->p, n_kept, d_wsum);
        FS_CUDA(cudaGetLastError());
        ++launches;
        // nobody may start the next call's memset of its slot before every rank has read all slots
        comm_barrier(comm, st, &launches);
        timer.end();
    }
    FS_CUDA(cudaStreamSynchronize(st));
    if (group_call) comm_check(comm);
    if (stats) {
        memset(stats, 0, sizeof(*stats));
        timer.finish(stats);
        unsigned long long sel_pairs = 0;
        FS_CUDA(cudaMemcpy(&sel_pairs, ds->counters.ptr, sizeof(sel_pairs), cudaMemcpyDeviceToHost));
        stats->launches = launches;
        stats->n_chunks = n_chunks;
        stats->n_tensor_cols = ws.pt;
        stats->n_general_cols = ws.n_cont + ws.n_cmp;
        stats->onehot_k = ws.K;
        stats->pairs_selected = (int64_t)sel_pairs;
        stats->ops_dist_tensor = ops_dist;
        stats->ops_accum_tensor = ops_accum;
        stats->ms_host_prep = ms_prep;
    }
}

}  // namespace fs

using namespace fs;

extern "C" {

int fs_score(fs_dataset *ds, int algo, int use_star, int32_t k, const float *class_probs,
             const int64_t *feat_idx, int64_t n_kept, int64_t row_begin, int64_t row_end, double *wsum_out,
             int out_on_device, fs_stats *stats) {
    return api_call("fs_score", [&] {
        FS_REQUIRE(ds && wsum_out, FS_ERR_INVALID, "fs_score: null pointer");
        if (!feat_idx) n_kept = ds->p;
        FS_REQUIRE(row_begin >= 0 && row_begin <= row_end && row_end <= ds->n, FS_ERR_INVALID,
                   "fs_score: bad row range [%lld, %lld) for n=%lld", (long long)row_begin, (long long)row_end,
                   (long long)ds->n);
        FS_CUDA(cudaSetDevice(ds->device));
        alloc_stream() = ds->stream;
        std::vector<int64_t> targets(row_end - row_begin);
        for (int64_t r = row_begin; r < row_end; ++r) targets[r - row_begin] = r;
        double *d_out = wsum_out;
        if (!out_on_device) {
            ds->wsum.reserve(n_kept);
            d_out = ds->wsum.ptr;
        }
        if (targets.empty()) {
            FS_CUDA(cudaMemsetAsync(d_out, 0, n_kept * sizeof(double), ds->stream));
            if (stats) memset(stats, 0, sizeof(*stats));
        } else {
            run_pipeline(ds, algo, use_star, k, class_probs, feat_idx, n_kept, targets, true, d_out, nullptr, stats);
        }
        if (!out_on_device) {
            FS_CUDA(cudaMemcpyAsync(wsum_out, d_out, n_kept * sizeof(double), cudaMemcpyDeviceToHost, ds->stream));
            FS_CUDA(cudaStreamSynchronize(ds->stream));
        }
        return FS_OK;
    });
}

int fs_debug_rows(fs_dataset *ds, int algo, int use_star, int32_t k, const float *class_probs,
                  const int64_t *feat_idx, int64_t n_kept, const int64_t *targets, int64_t nt, double *dist_out,
                  double *thresh_out, int8_t *mask_out, double *wsum_out) {
    return api_call("fs_debug_rows", [&] {
        FS_REQUIRE(ds && targets && nt >= 1, FS_ERR_INVALID, "fs_debug_rows: invalid argument");
        if (!feat_idx) n_kept = ds->p;
        FS_CUDA(cudaSetDevice(ds->device));
        alloc_stream() = ds->stream;
        std::vector<int64_t> ids(nt);
        for (int64_t t = 0; t < nt; ++t) {
            FS_REQUIRE(targets[t] >= 0 && targets[t] < ds->n, FS_ERR_INVALID, "fs_debug_rows: target %lld out of range",
                       (long long)targets[t]);
            ids[t] = ds->inv_perm[targets[t]];
        }
        ds->wsum.reserve(n_kept);
        DebugOut dbg{dist_out, thresh_out, mask_out};
        run_pipeline(ds, algo, use_star, k, class_probs, feat_idx, n_kept, ids, false, ds->wsum.ptr, &dbg, nullptr);
        if (wsum_out) FS_CUDA(cudaMemcpy(wsum_out, ds->wsum.ptr, n_kept * sizeof(double), cudaMemcpyDeviceToHost));
        return FS_OK;
    });
}

int fs_debug_slab(fs_dataset *ds, int64_t row_begin, int64_t nrows, int32_t *out, int64_t *info_out) {
    return api_call("fs_debug_slab", [&] {
        FS_REQUIRE(ds && out && nrows >= 1, FS_ERR_INVALID, "fs_debug_slab: invalid argument");
        FS_REQUIRE(ds->dd_valid && ds->dd_buf != nullptr, FS_ERR_STATE, "fs_debug_slab: no distance slab is cached");
        FS_REQUIRE(row_begin >= ds->dd_r0 && row_begin + nrows <= ds->dd_r0 + ds->dd_R, FS_ERR_STATE,
                   "fs_debug_slab: rows [%lld, %lld) outside the cached range [%lld, %lld)", (long long)row_begin,
                   (long long)(row_begin + nrows), (long long)ds->dd_r0, (long long)(ds->dd_r0 + ds->dd_R));
        FS_CUDA(cudaSetDevice(ds->device));
        FS_CUDA(cudaStreamSynchronize(ds->stream));
        const int64_t ldn = round_up(ds->n, 128);
        FS_CUDA(cudaMemcpy2D(out, ds->n * sizeof(int32_t), ds->dd_buf + (size_t)(row_begin - ds->dd_r0) * ldn,
                             ldn * sizeof(int32_t), ds->n * sizeof(int32_t), nrows, cudaMemcpyDeviceToHost));
        if (info_out) {
            info_out[0] = ds->dd_r0;
            info_out[1] = ds->dd_R;
            info_out[2] = (int64_t)ds->dd_cols.size();
        }
        return FS_OK;
    });
}

}  // extern "C"
