/*
 * fastselect_b200.h -- C ABI of libfastselect_b200.so
 *
 * B200-native (sm_100a) replacement for the Relief-family scoring hot path of
 * GavinLynch04/FastSelect: the n x n sample-pair distance computation, the
 * per-instance neighbour selection and the per-feature hit/miss weight
 * accumulation behind ReliefF, SURF, SURF*, MultiSURF, MultiSURF* (and TuRF,
 * which re-scores column subsets of one resident data set).
 *
 * Each entry point names the reference interface it replaces; citations are
 * file:line into the reference's src/fast_select/.
 *
 * Conventions: every function returns 0 on success and a negative fs_status on
 * failure; fs_last_error() returns a thread-local message for the last failure.
 * All output buffers are caller-allocated.  The library never keeps or frees
 * caller memory.  Calls on one fs_dataset must not overlap; different data sets
 * may be used from different threads.  There is NO CPU fallback: every compute
 * entry point fails with FS_ERR_NO_DEVICE when no sm_100 GPU is usable.
 */
#ifndef FASTSELECT_B200_H
#define FASTSELECT_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(__GNUC__)
#define FS_API __attribute__((visibility("default")))
#else
#define FS_API
#endif

#define FS_ABI_VERSION 9
/* distinct values tracked per column by fs_dataset_create; a column with more
 * distinct values reports FS_DISTINCT_CAP + 1 */
#define FS_DISTINCT_CAP 16

typedef struct fs_dataset fs_dataset; /* opaque; device-resident */

typedef enum { FS_RELIEFF = 0, FS_SURF = 1, FS_MULTISURF = 2 } fs_algo;
typedef enum { FS_U8 = 0, FS_I8 = 1, FS_F32 = 2, FS_F64 = 3 } fs_dtype;
/* arithmetic of the continuous per-feature term (SURVEY.md a1):
 *   FS_ARITH_F32: fl32(fl32(|a-b|) * r)  -- MultiSURF.py:184-188, ReliefF.py:151-154
 *   FS_ARITH_F64: |a-b| * (double)r       -- SURF.py:153-156 (X stays float64) */
typedef enum { FS_ARITH_F32 = 0, FS_ARITH_F64 = 1 } fs_arith;

typedef enum {
    FS_OK = 0,
    FS_ERR_INVALID = -1,    /* bad argument */
    FS_ERR_NO_DEVICE = -2,  /* no usable sm_100 GPU / driver */
    FS_ERR_CUDA = -3,       /* CUDA runtime error (message has the detail) */
    FS_ERR_OOM = -4,        /* device or host allocation failed */
    FS_ERR_STATE = -5,      /* call order violated (e.g. score before set_features) */
    FS_ERR_TIMEOUT = -6     /* a multi-GPU barrier gave up: a rank failed or left the collective call */
} fs_status;

/* neighbour codes in fs_debug_rows' mask_out (same values as the oracle's) */
enum { FS_MASK_NONE = 0, FS_MASK_NEAR_HIT = 1, FS_MASK_NEAR_MISS = 2, FS_MASK_FAR_MISS = 3, FS_MASK_FAR_HIT = 4 };

/* Per-call timings (CUDA events on the call's stream) and work counters. */
typedef struct fs_stats {
    float ms_total;          /* whole fs_score call on the device */
    float ms_gather;         /* column compaction / one-hot encode of the active columns */
    float ms_dist_tensor;    /* one-hot tcgen05 (FP4 kind::mxf4, exact) distance kernel(s) */
    float ms_dist_general;   /* CUDA-core distance kernel(s) (continuous / wide discrete) */
    float ms_select;         /* row statistics, thresholds / top-k, neighbour masks */
    float ms_accum_tensor;   /* mask x one-hot tcgen05 accumulation kernel(s) */
    float ms_accum_general;  /* CUDA-core accumulation / ReliefF gather kernel(s) */
    float ms_reduce;         /* final per-feature reduction */
    int32_t launches;        /* kernels launched by this call */
    int32_t n_chunks;        /* target-row chunks processed */
    int64_t n_tensor_cols;   /* active columns on the one-hot tensor-core path */
    int64_t n_general_cols;  /* active columns on the CUDA-core path */
    int64_t onehot_k;        /* contraction length of the one-hot operands (sum of V_f - 1, padded) */
    int64_t pairs_selected;  /* neighbour pairs with a non-zero coefficient */
    double ops_dist_tensor;  /* operations (2 per MAC) issued to the tensor pipe by the distance kernel(s) */
    double ops_accum_tensor; /* same, accumulation kernel(s) */
    double ms_host_prep;     /* host wall time spent preparing the working set (inside ms_gather) */
} fs_stats;

/* Number of usable sm_100 devices (0 when there is no driver/GPU).  Replaces
 * numba.cuda.is_available() in MultiSURF.py:393-406, SURF.py:338-343, ReliefF.py:382-385. */
FS_API int fs_device_count(void);
FS_API const char *fs_last_error(void);
FS_API int fs_abi_version(void);

/*
 * Upload X (host pointer, row-major, row stride in elements) to `device` and scan
 * every column once on the GPU: min, max and the set of distinct values (up to
 * FS_DISTINCT_CAP).  Replaces cuda.to_device(x) and the per-column np.unique /
 * range pass of fit (MultiSURF.py:409-425, SURF.py:347-365, ReliefF.py:366-391).
 * y_enc: class index 0..n_classes-1 per sample (labels are only compared for
 * equality: MultiSURF.py:216, SURF.py:175, ReliefF.py:166).
 * stream: a cudaStream_t (NULL = the legacy default stream); all later work on
 * this data set is issued on it.
 */
FS_API int fs_dataset_create(fs_dataset **out, const void *x, int dtype, int64_t n, int64_t p,
                      int64_t row_stride_elems, const int32_t *y_enc, int32_t n_classes,
                      int32_t device, void *stream);

/* Same, for a matrix that is already on `device` (row-major device pointer). */
FS_API int fs_dataset_create_device(fs_dataset **out, const void *x_dev, int dtype, int64_t n, int64_t p,
                             int64_t row_stride_elems, const int32_t *y_enc, int32_t n_classes,
                             int32_t device, void *stream);

/* Column scan results, each [p]: exact min / max as doubles, and the distinct-value
 * count (FS_DISTINCT_CAP + 1 means "more than FS_DISTINCT_CAP").  Any may be NULL. */
FS_API int fs_dataset_column_stats(const fs_dataset *ds, double *col_min, double *col_max,
                            int32_t *n_distinct);

/* Per-column typing chosen by the caller exactly as the reference's fit does:
 * is_discrete[p] (np.unique(col).size <= discrete_limit) and recip[p] = 1/range as
 * float32 (MultiSURF.py:409-420; SURF.py:347-355; ReliefF.py:366-380). */
FS_API int fs_dataset_set_features(fs_dataset *ds, const uint8_t *is_discrete, const float *recip, int arith);

FS_API int fs_dataset_destroy(fs_dataset *ds);

/*
 * Score the columns feat_idx[0..n_kept) (NULL = all p) for the target rows
 * [row_begin, row_end) of the data set's internal sample order (a fixed
 * permutation of the samples; any partition of [0, n) covers every sample once,
 * which is how target rows are sharded across GPUs).  Writes
 *     wsum_out[c] = sum over those targets i of W_i[feat_idx[c]]     (float64)
 * i.e. the reference host callers' result before the final "/ n_samples"
 * (_multisurf_gpu_host_caller MultiSURF.py:147-162, _surf_gpu_host_caller
 * SURF.py:117-128, _relieff_gpu_host_caller ReliefF.py:127-134).  A multi-GPU
 * caller sums the partial vectors (one allreduce) and divides by n.
 * k and class_probs[n_classes] are used by FS_RELIEFF only.
 * out_on_device != 0: wsum_out is a device pointer on the data set's device.
 */
FS_API int fs_score(fs_dataset *ds, int algo, int use_star, int32_t k, const float *class_probs,
             const int64_t *feat_idx, int64_t n_kept, int64_t row_begin, int64_t row_end,
             double *wsum_out, int out_on_device, fs_stats *stats);

/*
 * Parity/debug view of the same kernels for nt target samples given by ORIGINAL
 * sample index: the distance row (float64, original sample order, 0 at the target
 * itself), the neighbour threshold (MultiSURF: T_i; SURF: mean distance; ReliefF: 0)
 * and the neighbour code of every sample (FS_MASK_*).  Outputs are host pointers,
 * [nt*n], [nt], [nt*n]; any may be NULL.  wsum_out[n_kept] (host, may be NULL)
 * receives the sum of the targets' contributions, as fs_score does for a row range.
 */
FS_API int fs_debug_rows(fs_dataset *ds, int algo, int use_star, int32_t k, const float *class_probs,
                  const int64_t *feat_idx, int64_t n_kept, const int64_t *targets, int64_t nt,
                  double *dist_out, double *thresh_out, int8_t *mask_out, double *wsum_out);

/*
 * Multi-GPU group (the reference has no multi-GPU path, SURVEY.md 8e; its unit of parallelism is the
 * target instance, MultiSURF.py:174).  One rank per GPU -- one process per GPU (CUDA IPC) or one host
 * thread per GPU inside one process (peer access; see fs_multi_* below).  Every rank owns an exchange
 * ARENA (one cudaMalloc block) that the other ranks map; all exchanges are stores into the peers' arenas
 * over NVLink followed by a device-side barrier (flags in the arenas; no host synchronisation):
 *   - target rows are sharded across ranks; D is symmetric, so each rank computes half of the
 *     off-diagonal blocks of its row shard and stores every tile twice, the transposed copy straight
 *     into the owner's slab (from the GEMM epilogue);
 *   - MultiSURF / SURF: every rank sends the neighbour masks of its rows to all ranks and accumulates
 *     ITS SHARE OF THE ONE-HOT COLUMNS against the masks of all targets (so the one-hot encode of the
 *     accumulation operand is not replicated); ReliefF and continuous columns accumulate partial sums
 *     over the rank's rows;
 *   - the ranks' weight contributions are exchanged and added in rank order: fs_score then returns the
 *     COMPLETE sums, bitwise identical on every rank.
 *
 * fs_comm_create / fs_comm_reserve / fs_comm_connect: create this rank's communicator, make sure its
 *   arena holds `bytes` (fs_comm_required_bytes; *changed_out = 1 when it was (re)allocated -- then the
 *   64-byte IPC handle must be exchanged again), and map the peers: ipc_handles = world x 64 bytes, or
 *   raw_ptrs = the peers' arena pointers (ranks inside one process).  After fs_comm_connect the CALLER
 *   must run a host-level barrier over all ranks before the first collective call.
 * fs_dataset_create_group: like fs_dataset_create, but this rank uploads only rows
 *   [n * rank / world, n * (rank + 1) / world) of the host matrix (every rank passes the same x) and the
 *   shards are replicated over NVLink.  COLLECTIVE.
 * fs_dataset_attach_comm: row_starts[world + 1] = first internal row of every rank's shard (ascending
 *   multiples of 4, row_starts[world] = n, no empty shard, at most ceil(n / world) + 4 rows each).
 *   Afterwards fs_score(row_begin = row_starts[rank], row_end = row_starts[rank + 1]) is COLLECTIVE:
 *   every rank must call it with its own shard and otherwise identical arguments, and wsum_out
 *   receives the complete sums.  Other row ranges and fs_debug_rows stay local.  comm = NULL detaches.
 *   A barrier that waits longer than FS_B200_BARRIER_TIMEOUT_S (default 20 s) fails the call with
 *   FS_ERR_TIMEOUT instead of hanging; the group must then be connected again.
 */
typedef struct fs_comm fs_comm;
FS_API int fs_comm_create(fs_comm **out, int32_t rank, int32_t world, int32_t device);
FS_API uint64_t fs_comm_required_bytes(int64_t n, int64_t p, int32_t dtype, int32_t world, int32_t with_x);
FS_API int fs_comm_reserve(fs_comm *comm, uint64_t bytes, void *ipc_handle_out, int32_t *changed_out);
FS_API int fs_comm_connect(fs_comm *comm, const void *ipc_handles, void *const *raw_ptrs);
FS_API void *fs_comm_arena(fs_comm *comm);
FS_API uint64_t fs_comm_arena_bytes(fs_comm *comm);
FS_API int fs_comm_connected(fs_comm *comm);
FS_API int fs_comm_destroy(fs_comm *comm);
FS_API int fs_dataset_create_group(fs_dataset **out, fs_comm *comm, const void *x, int dtype, int64_t n, int64_t p,
                            int64_t row_stride_elems, const int32_t *y_enc, int32_t n_classes, void *stream);
FS_API int fs_dataset_attach_comm(fs_dataset *ds, fs_comm *comm, const int64_t *row_starts);

/*
 * Several GPUs from ONE process (no torchrun, no torch): one host thread per device drives one rank of a
 * multi-GPU group whose arenas are mapped through peer access.  Replaces, for a multi-GPU box, the same
 * host callers as fs_dataset_create + fs_score (MultiSURF.py:147-162, :409-432; SURF.py:117-128;
 * ReliefF.py:127-134).  devices[n_devices]: CUDA device ordinals (distinct, all sm_100, peer-accessible).
 * Every device uploads 1 / n_devices of X and the shards are replicated over NVLink; fs_multi_score
 * returns the complete weight sums (the value a single-GPU fs_score over all rows returns).
 * Communicators (arenas, peer mappings, streams) are cached per device list for the life of the process.
 */
typedef struct fs_multi fs_multi;
FS_API int fs_multi_create(fs_multi **out, const void *x, int dtype, int64_t n, int64_t p, int64_t row_stride_elems,
                    const int32_t *y_enc, int32_t n_classes, const int32_t *devices, int32_t n_devices);
FS_API int fs_multi_world(const fs_multi *m);        /* ranks in use (fewer than n_devices for tiny data sets) */
FS_API int fs_multi_column_stats(const fs_multi *m, double *col_min, double *col_max, int32_t *n_distinct);
FS_API int fs_multi_set_features(fs_multi *m, const uint8_t *is_discrete, const float *recip, int arith);
FS_API int fs_multi_score(fs_multi *m, int algo, int use_star, int32_t k, const float *class_probs,
                   const int64_t *feat_idx, int64_t n_kept, double *wsum_out, fs_stats *stats);
FS_API int fs_multi_destroy(fs_multi *m);

/*
 * Joint-count path (SURVEY.md section 8(f)-4): pairwise statistics of DISCRETE columns from their
 * contingency tables.  The tables of all column pairs are one GEMM over the samples between the
 * reduced one-hot rows of the columns (the operand the accumulation kernel already uses), run on
 * the tensor cores with exact integer results; a finishing kernel rebuilds every pair's full table
 * and folds it into the statistic.  Replaces _batch_mi_cpu / calculate_mi_matrices
 * (mutual_information.py:49-63, :158-196 -- the reference computes the redundancy matrix on the
 * CPU even with backend="gpu", :191-193) and _precompute_correlations_cpu / the one-thread-per-
 * feature GPU kernel of CFS (CFS.py:81-104, :219-243).
 *
 * Every column in feat_idx (NULL = all p) must have been marked discrete in
 * fs_dataset_set_features and hold at most FS_DISTINCT_CAP distinct values (FS_ERR_INVALID
 * otherwise); a class vector takes part as one more column of X.  Sample order and y_enc of the
 * data set are irrelevant here.
 *
 * fs_joint_matrix: out[a * n_kept + b] = statistic(feat_idx[a], feat_idx[b]) for the pairs with
 *   pos_begin <= min(a, b) < pos_end (both triangles are written; everything else, and the
 *   diagonal, is 0, as in mutual_information.py:53 / CFS.py:95), float64.  Ranks of a multi-GPU
 *   job take disjoint position ranges and sum their matrices.
 *   kind FS_JOINT_MI: sum p_xy ln(p_xy / (p_x p_y + 1e-12)) / log_base  (mutual_information.py:35-46)
 *   kind FS_JOINT_SU: 2 I(x; y) / (H(x) + H(y)) in bits                  (CFS.py:26-77; the reference
 *        keeps float32 intermediates there, this is the float64 value: |difference| < 1e-6)
 *   out_on_device != 0: out is a device pointer on the data set's device.
 *   The one-hot rows, their marginals and the position offsets of a column list are shared by
 *   fs_joint_matrix, fs_joint_tables, fs_joint_columns and fs_mdr_*: built by the first of these calls
 *   on a (column list, typing) and reused by the following ones until the data set's working set is
 *   rebuilt (fs_dataset_set_features, another column list, fs_score).
 * fs_joint_tables: the contingency tables themselves for m pairs of positions (pairs[2 * q],
 *   pairs[2 * q + 1]), exact integers: tables_out[q * 256 + va * 16 + vb] = #samples with the va-th
 *   smallest value of the first column and the vb-th smallest value of the second (host pointer).
 * fs_joint_columns: rows of the same matrix for n_pos chosen positions, without the p x p matrix:
 *   out[i * n_kept + g] = statistic(feat_idx[positions[i]], feat_idx[g]) for every g in [0, n_kept),
 *   0 at g == positions[i]; bitwise equal to row positions[i] of fs_joint_matrix.  Every position must
 *   lie in [0, n_kept); the other checks and error codes are those of fs_joint_matrix.  The counts come
 *   from one pass of the CUDA cores over the reduced one-hot rows per 16 selected reduced rows (one pass
 *   for a call of up to 8 genotype or one 16-state position), so a greedy search that needs k columns
 *   reads k passes, not p^2 statistics.  The one-hot rows, offsets and marginals are shared with
 *   fs_joint_matrix (see there).  In stats: ms_gather = their build (about 0 on a reuse), ms_dist_general = count kernels, ms_reduce = finish
 *   kernels, n_chunks = count launches.
 */
typedef enum { FS_JOINT_MI = 0, FS_JOINT_SU = 1 } fs_joint_kind;
FS_API int fs_joint_matrix(fs_dataset *ds, int kind, double log_base, const int64_t *feat_idx, int64_t n_kept,
                    int64_t pos_begin, int64_t pos_end, double *out, int out_on_device, fs_stats *stats);
FS_API int fs_joint_tables(fs_dataset *ds, const int64_t *feat_idx, int64_t n_kept, const int64_t *pairs, int64_t m,
                    int64_t *tables_out);
FS_API int fs_joint_columns(fs_dataset *ds, int kind, double log_base, const int64_t *feat_idx, int64_t n_kept,
                            const int64_t *positions, int64_t n_pos, double *out, int out_on_device, fs_stats *stats);

/*
 * MDR (multifactor dimensionality reduction; the semantics are this project's own, see DESIGN.md "MDR"):
 * exhaustive search over the combinations of order 1 or 2 of the positions of feat_idx (NULL = all p) for
 * the one whose high-risk cells best separate the two classes, scored by cross-validated balanced accuracy.
 * The data set's y_enc is the class (n_classes must be 2; class 1 is the case class).  fold[n] gives every
 * sample's cross-validation fold in [0, n_folds), in ORIGINAL sample order; 2 <= n_folds <= 10, and every
 * fold must hold samples of both classes.  Every scanned column must be discrete in fs_dataset_set_features
 * and hold at most 3 distinct values (FS_ERR_INVALID otherwise); a column's cell index is the rank of its
 * value among its sorted distinct values.  n < 2^26.
 *
 * Combination index: order 1, the position a; order 2, the lexicographic rank of (a, b), a < b:
 *   idx = a * n_kept - a * (a + 1) / 2 + (b - a - 1),   n_combos = n_kept * (n_kept - 1) / 2.
 * Per combination and fold f: training counts over the samples with fold != f, test counts over fold f;
 * a cell is high-risk iff T1 * N0 > T0 * N1 (int64; ties and empty cells are low-risk); balanced accuracy
 * = (TP * N0 + TN * N1) / (2 N1 N0) with one float64 division, the test one with the training labels; the
 * means over the folds are summed in fold order, then divided by n_folds.
 *
 * fs_mdr_scan: top_idx / top_train / top_test [n_top]: the n_top combinations with the highest mean test
 *   balanced accuracy (lower index first on ties), with their mean training / test values;
 *   1 <= n_top <= min(FS_MDR_MAX_TOP, n_combos).  fold_best[n_folds]: per fold, the combination with the
 *   highest training balanced accuracy (lower index first on ties).  all_train / all_test (nullable, both
 *   or neither, [n_combos] host arrays): the means of every combination.  The one-hot rows and offsets
 *   are shared with fs_joint_matrix (see there); the bit-planes of a (column list, fold vector) are built
 *   from them by the first call and reused by later calls until they are rebuilt.  In stats: ms_gather = encode + pack (about 0 on a reuse), ms_dist_general = scan kernel,
 *   ms_reduce = merges, n_chunks = scan blocks, pairs_selected = n_combos.
 * fs_mdr_tables: tables_out[((q * n_folds + f) * 2 + c) * 9 + va * 3 + vb], int64: samples of fold f and
 *   class c in cell (va, vb) of combination q = combos[q * order ..] (positions, any order; order 1: vb = 0).
 */
#define FS_MDR_MAX_TOP 2048
FS_API int fs_mdr_scan(fs_dataset *ds, const int64_t *feat_idx, int64_t n_kept, int32_t order, const int32_t *fold,
                       int32_t n_folds, int64_t n_top, int64_t *top_idx, double *top_train, double *top_test,
                       int64_t *fold_best, double *all_train, double *all_test, fs_stats *stats);
FS_API int fs_mdr_tables(fs_dataset *ds, const int64_t *feat_idx, int64_t n_kept, int32_t order, const int32_t *fold,
                         int32_t n_folds, const int64_t *combos, int64_t m, int64_t *tables_out);

/*
 * Two-locus interaction screen (the KSA stage of BOOST; the semantics are this project's own, see DESIGN.md
 * section 11): every pair (a, b), a < b, of the positions of feat_idx (NULL = all p) on the MDR planes of a
 * single fold, so the two segments are the two classes.  The data set's y_enc is the class (n_classes must
 * be 2); every scanned column must be discrete in fs_dataset_set_features and hold at most 3 distinct
 * values (FS_ERR_INVALID otherwise); a column's state is the rank of its value among its sorted distinct
 * values; n < 2^26.  Pair index: the order-2 index of fs_mdr_scan.
 *
 * Per pair, with n_ijk the samples of state i in a, state j in b and class k, and N = n:
 *   q_ijk = (n_ij * n_ik * n_jk) / (n_i * n_j * n_k), 0 when a numerator margin is 0;   eta = sum q_ijk;
 *   L_KSA = 2 * sum_{n_ijk > 0} n_ijk * log(n_ijk * eta / (N * q_ijk)),
 * all in float64, the sums in cell order (i, j, k).  L_KSA bounds the likelihood-ratio statistic of the
 * no-three-way-interaction model from above (G <= L_KSA).
 *
 * fs_interaction_scan: top_idx / top_ksa [n_top]: the n_top pairs with the highest L_KSA (lower index first
 *   on ties); 1 <= n_top <= min(FS_MDR_MAX_TOP, n_pairs), n_pairs = n_kept * (n_kept - 1) / 2.
 *   top_tables[(q * 2 + k) * 9 + i * 3 + j], int64 [n_top, 2, 9]: n_ijk of listed pair q, exact.  all_ksa
 *   (nullable, [n_pairs] host array): L_KSA of every pair.  The bit-planes are those of fs_mdr_scan with the
 *   fold vector of all zeros (built by the first call, reused by later ones).  In stats: ms_gather = encode +
 *   pack (about 0 on a reuse), ms_dist_general = scan kernel, ms_reduce = merges, n_chunks = scan blocks,
 *   pairs_selected = n_pairs; ms_total ends before the tables of the listed pairs are counted.
 */
FS_API int fs_interaction_scan(fs_dataset *ds, const int64_t *feat_idx, int64_t n_kept, int64_t n_top, int64_t *top_idx,
                               double *top_ksa, int64_t *top_tables, double *all_ksa, fs_stats *stats);

/*
 * Parity/debug view of the RESIDENT one-hot distance slab fs_score keeps between calls for TuRF's
 * incremental update (d_ij -= sum over removed columns, TuRF.py:99-113): the integer mismatch counts
 * of internal target rows [row_begin, row_begin + nrows) against all n samples (internal order), as
 * left by the last fs_score call.  out: host int32 [nrows * n].  FS_ERR_STATE when no slab is cached
 * or the rows are outside the cached range.  `info_out` (nullable, int64[3]) receives the first cached
 * row, the number of cached rows and the number of one-hot columns the slab sums over.
 */
FS_API int fs_debug_slab(fs_dataset *ds, int64_t row_begin, int64_t nrows, int32_t *out, int64_t *info_out);

/* Internal order: perm_out[r] = original index of internal row r ([n]). */
FS_API int fs_dataset_row_order(const fs_dataset *ds, int64_t *perm_out);

#ifdef __cplusplus
}
#endif
#endif /* FASTSELECT_B200_H */
