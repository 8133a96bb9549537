// select.cu -- per-target-row neighbour selection (one CTA per target row).
//
// Replaces, for each target i:
//   MultiSURF: mu_i, sigma_i, T_i = mu_i - sigma_i/2 and the near/far test d_ij < T_i
//              (MultiSURF.py:175-196, :216-243);
//   SURF:      the float32 mean distance and d_ij < mean (SURF.py:146-163, :175-190);
//   ReliefF:   k nearest hits and k nearest misses of every other class
//              (ReliefF.py:144-175) with per-neighbour weights (ReliefF.py:177-216).
// Output: one int8 neighbour code per pair (FS_MASK_*), a RowInfo per target with
// the per-code coefficients, and for ReliefF a compact neighbour list.
// HBM/L2-bound: each kernel streams its distance row twice (the row is L2-resident).
#include "common.cuh"

namespace fs {

__device__ __forceinline__ double load_d(const double *Dc, const int32_t *Dd, int64_t off) {
    double d = Dc ? Dc[off] : 0.0;
    if (Dd) d += (double)Dd[off];
    return d;
}

// deterministic block sum (fixed order): warp shuffles, then warp partials in order
template <typename T>
__device__ __forceinline__ T block_sum(T v, T *scratch /*[8]*/) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
    __syncthreads();
    if ((threadIdx.x & 31) == 0) scratch[threadIdx.x >> 5] = v;
    __syncthreads();
    T s = scratch[0];
#pragma unroll
    for (int w = 1; w < 8; ++w) s += scratch[w];
    return s;
}

template <int ALGO>
__global__ void __launch_bounds__(256) select_threshold_kernel(const double *__restrict__ Dc,
                                                               const int32_t *__restrict__ Dd, int64_t ldn,
                                                               int64_t n, int64_t r0,
                                                               const int32_t *__restrict__ y,
                                                               const int64_t *__restrict__ inv_perm, int use_star,
                                                               int8_t *__restrict__ sel,
                                                               int8_t *__restrict__ mask_h,
                                                               int8_t *__restrict__ mask_m,
                                                               RowInfo *__restrict__ rinfo) {
    __shared__ double sd[8];
    __shared__ int si[8];
    __shared__ double s_thresh;
    const int64_t r = blockIdx.x;
    const int64_t self = r0 + r;
    const int64_t base = r * ldn;
    const int tid = threadIdx.x;
    const double inv = 1.0 / (double)(n - 1);

    if (ALGO == FS_MULTISURF) {
        // pass 1: sum d, sum d^2 over j != i (MultiSURF.py:175-191)
        double s1 = 0.0, s2 = 0.0;
        for (int64_t j = tid; j < n; j += 256) {
            if (j == self) continue;
            double d = load_d(Dc, Dd, base + j);
            s1 += d;
            s2 = __fma_rn(d, d, s2);
        }
        s1 = block_sum(s1, sd);
        s2 = block_sum(s2, sd);
        if (tid == 0) {
            // MultiSURF.py:193-196 with the roundings of the reference's JIT'd code
            // (multiply by 1/(n-1); fused sum_d2*inv - mu*mu); see oracle/fs_oracle.c
            double mu = __dmul_rn(s1, inv);
            double var = __fma_rn(s2, inv, -__dmul_rn(mu, mu));
            var = var > 0.0 ? var : 0.0;
            s_thresh = __dsub_rn(mu, __dmul_rn(0.5, __dsqrt_rn(var)));
        }
    } else {
        // SURF.py:146-163: distances rounded to float32, d_ii = 0 included, np.sum in float32,
        // times 1/(n-1) in float64.  The float32 sum is taken in the order the reference's
        // JIT'd code uses on x86-64 (AVX2 width, observed with inspect_asm(); oracle
        // sum_mode 2, pinned to the reference): 32 interleaved partial sums over the leading
        // multiple of 32 folded 32->8->4->2->1, then a 4-wide loop seeded with that value,
        // then a scalar tail.  One warp does it (the chain per lane is n/32 adds).
        if (tid < 32) {
            const unsigned full = 0xffffffffu;
            // the sum runs over the samples in their ORIGINAL order (o -> internal row inv_perm[o])
            auto d32 = [&](int64_t o) -> float {
                const int64_t j = inv_perm[o];
                return j == self ? 0.0f : (float)load_d(Dc, Dd, base + j);
            };
            float s = 0.0f;
            int64_t done = 0;
            if (n >= 32) {
                const int64_t m = n & ~(int64_t)31;
                float p = 0.0f;
                for (int64_t t = 0; t < m; t += 32) p = __fadd_rn(p, d32(t + tid));
                // q[l] = (p[l] + p[l+8]) + (p[l+24] + p[l+16]), l < 8
                const float a = __fadd_rn(p, __shfl_down_sync(full, p, 8));
                const float q = __fadd_rn(a, __shfl_down_sync(full, a, 16));
                const float r4 = __fadd_rn(__shfl_down_sync(full, q, 4), q);      // r[l] = q[l+4] + q[l]
                const float u2 = __fadd_rn(__shfl_down_sync(full, r4, 2), r4);    // u[l] = r[l+2] + r[l]
                s = __fadd_rn(__shfl_down_sync(full, u2, 1), u2);                 // u[1] + u[0]
                s = __shfl_sync(full, s, 0);
                done = m;
            }
            if (n - done >= 4) {
                const int64_t m = done + ((n - done) & ~(int64_t)3);
                float v = tid == 0 ? s : 0.0f;
                if (tid < 4)
                    for (int64_t t = done; t < m; t += 4) v = __fadd_rn(v, d32(t + tid));
                const float u = __fadd_rn(__shfl_down_sync(full, v, 2), v);       // v[2]+v[0], v[3]+v[1]
                s = __fadd_rn(__shfl_down_sync(full, u, 1), u);                   // u1 + u0
                s = __shfl_sync(full, s, 0);
                done = m;
            }
            if (tid == 0) {
                for (int64_t t = done; t < n; ++t) s = __fadd_rn(s, d32(t));
                s_thresh = __dmul_rn((double)s, inv);
            }
        }
    }
    __syncthreads();
    const double thresh = s_thresh;
    const int32_t yi = y[self];
    int nh = 0, nm = 0, nfh = 0, nfm = 0;
    // two samples per thread and step: the signed masks of the tensor-core accumulation
    // (c_ij = -aH*mH + aM*mM, mH/mM in {-1, 0, 1}) are stored as e2m1 (FP4) nibbles, two samples per
    // byte, low nibble = even sample: +1 -> 0x2, -1 -> 0xA.  Row pitch ldn / 2 bytes.
    for (int64_t j0 = 2 * (int64_t)tid; j0 < n; j0 += 512) {
        uint32_t bh = 0, bm = 0;
#pragma unroll
        for (int h = 0; h < 2; ++h) {
            const int64_t j = j0 + h;
            if (j >= n) break;
            int code = FS_MASK_NONE;
            if (j != self) {
                double d = load_d(Dc, Dd, base + j);
                if (ALGO == FS_SURF) d = (double)(float)d;
                const bool hit = (y[j] == yi);
                if (d < thresh) {
                    code = hit ? FS_MASK_NEAR_HIT : FS_MASK_NEAR_MISS;
                } else if (use_star) {
                    if (!hit) code = FS_MASK_FAR_MISS;
                    else if (ALGO == FS_SURF) code = FS_MASK_FAR_HIT;
                }
            }
            sel[base + j] = (int8_t)code;
            bh |= (code == FS_MASK_NEAR_HIT ? 0x2u : code == FS_MASK_FAR_HIT ? 0xAu : 0u) << (4 * h);
            bm |= (code == FS_MASK_NEAR_MISS ? 0x2u : code == FS_MASK_FAR_MISS ? 0xAu : 0u) << (4 * h);
            nh += (code == FS_MASK_NEAR_HIT);
            nm += (code == FS_MASK_NEAR_MISS);
            nfm += (code == FS_MASK_FAR_MISS);
            nfh += (code == FS_MASK_FAR_HIT);
        }
        if (mask_h) {
            mask_h[(base >> 1) + (j0 >> 1)] = (int8_t)bh;
            mask_m[(base >> 1) + (j0 >> 1)] = (int8_t)bm;
        }
    }
    nh = block_sum(nh, si);
    nm = block_sum(nm, si);
    nfh = block_sum(nfh, si);
    nfm = block_sum(nfm, si);
    if (tid == 0) {
        RowInfo ri;
        ri.thresh = thresh;
        ri.n_hit = nh;
        ri.n_miss = nm;
        ri.n_far_hit = nfh;
        ri.n_far_miss = nfm;
        ri.coef[0] = 0.0;
        if (ALGO == FS_MULTISURF) {
            // MultiSURF.py:245-251: divide by the counts unless they are zero;
            // the far-miss term shares the near-miss normalisation
            const double sh = nh > 0 ? 1.0 / (double)nh : 1.0;
            const double sm = nm > 0 ? 1.0 / (double)nm : 1.0;
            ri.coef[FS_MASK_NEAR_HIT] = -sh;
            ri.coef[FS_MASK_NEAR_MISS] = sm;
            ri.coef[FS_MASK_FAR_MISS] = -sm;
            ri.coef[FS_MASK_FAR_HIT] = 0.0;
        } else {
            // SURF.py:191-193: near_miss - near_hit (+ far_hit - far_miss), no normalisation
            ri.coef[FS_MASK_NEAR_HIT] = -1.0;
            ri.coef[FS_MASK_NEAR_MISS] = 1.0;
            ri.coef[FS_MASK_FAR_MISS] = -1.0;
            ri.coef[FS_MASK_FAR_HIT] = 1.0;
        }
        rinfo[r] = ri;
    }
}

// exclusive rank of `flag` within the CTA (thread order) and the CTA total
__device__ __forceinline__ int block_rank(bool flag, int *warp_tot /*[8]*/, int &total) {
    const unsigned b = __ballot_sync(0xffffffffu, flag);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
    const int r = __popc(b & ((1u << lane) - 1u));
    __syncthreads();
    if (lane == 0) warp_tot[w] = __popc(b);
    __syncthreads();
    int off = 0, tot = 0;
#pragma unroll
    for (int q = 0; q < 8; ++q) {
        const int t = warp_tot[q];
        off += (q < w) ? t : 0;
        tot += t;
    }
    total = tot;
    return off + r;
}

__global__ void __launch_bounds__(256) relieff_select_kernel(
    const double *__restrict__ Dc, const int32_t *__restrict__ Dd, int64_t ldn, int64_t n,
    int64_t r0, const int32_t *__restrict__ y, const int64_t *__restrict__ cls_start,
    int n_classes, int k, const float *__restrict__ class_probs, int8_t *__restrict__ sel,
    RowInfo *__restrict__ rinfo, int32_t *__restrict__ nbr_idx, double *__restrict__ nbr_w,
    int32_t *__restrict__ nbr_cnt, int nbr_cap, int32_t *__restrict__ tie_list) {
    __shared__ int hist[256];
    __shared__ int warp_tot[8];
    __shared__ unsigned s_prefix;
    __shared__ int s_remaining;
    const int64_t r = blockIdx.x;
    const int64_t self = r0 + r;
    const int64_t base = r * ldn;
    const int tid = threadIdx.x;
    const int ci = y[self];

    for (int64_t j = tid; j < n; j += 256) sel[base + j] = FS_MASK_NONE;
    // ReliefF.py:177-179
    double denom = 1.0 - (double)class_probs[ci];
    if (denom == 0.0) denom = 1.0;

    auto key_of = [&](int64_t j) -> unsigned {
        // ReliefF.py:144-155: float32 distances, inf on the diagonal (the target itself
        // stays a candidate of its own class and is taken last)
        return j == self ? 0x7f800000u : __float_as_uint((float)load_d(Dc, Dd, base + j));
    };

    int slot_base = 0, n_hit = 0, n_miss = 0;
    bool ambiguous = false;     // some class has more candidates tied at the k-th distance than slots
    for (int c = 0; c < n_classes; ++c) {
        const int64_t s0 = cls_start[c], s1 = cls_start[c + 1];
        const int64_t len = s1 - s0;
        const int kk = (int)(len < (int64_t)k ? len : (int64_t)k);
        if (kk == 0) continue;
        // ReliefF.py:181-216: -1/h_found per hit; P(c)/(1-P(c_i))/k per miss of class c
        const double w = (c == ci) ? -1.0 / (double)kk : ((double)class_probs[c] / denom) / (double)k;
        const int8_t code = (c == ci) ? FS_MASK_NEAR_HIT : FS_MASK_NEAR_MISS;
        unsigned kth = 0xffffffffu;
        int need_eq = 0;
        if (kk < len) {
            // radix select of the kk-th smallest key, 8 bits per pass, MSB first
            __syncthreads();
            if (tid == 0) { s_prefix = 0u; s_remaining = kk; }
            unsigned mask = 0u;
            for (int shift = 24; shift >= 0; shift -= 8) {
                hist[tid] = 0;
                __syncthreads();
                const unsigned prefix = s_prefix;
                for (int64_t j = s0 + tid; j < s1; j += 256) {
                    const unsigned key = key_of(j);
                    // warp-aggregated histogram update: distances of one row share their leading
                    // bytes, so most lanes hit the same bin (one shared atomic per distinct bin)
                    const unsigned bin = (key & mask) == prefix ? (key >> shift) & 255u : 0xffffffffu;
                    const unsigned peers = __match_any_sync(__activemask(), bin);
                    if (bin != 0xffffffffu && (tid & 31) == __ffs(peers) - 1) atomicAdd(&hist[bin], __popc(peers));
                }
                __syncthreads();
                if (tid == 0) {
                    int rem = s_remaining, cum = 0, b = 0;
                    for (; b < 256; ++b) {
                        if (cum + hist[b] >= rem) break;
                        cum += hist[b];
                    }
                    s_remaining = rem - cum;
                    s_prefix = prefix | ((unsigned)b << shift);
                }
                mask |= 255u << shift;
                __syncthreads();
            }
            kth = s_prefix;
            need_eq = s_remaining;
        }
        // ordered pass: ties at the k-th distance are taken in sample order
        int eq_taken = 0, slot = slot_base;
        for (int64_t b0 = s0; b0 < s1; b0 += 256) {
            const int64_t j = b0 + tid;
            const bool valid = j < s1;
            bool take = valid;
            if (kk < len) {
                const unsigned key = valid ? key_of(j) : 0xffffffffu;
                const bool eq = valid && key == kth;
                int tot_eq;
                const int rk = block_rank(eq, warp_tot, tot_eq);
                take = valid && (key < kth || (eq && eq_taken + rk < need_eq));
                eq_taken += tot_eq;
                if (b0 + 256 >= s1 && eq_taken > need_eq) ambiguous = true;
            }
            int tot_take;
            const int rk2 = block_rank(take, warp_tot, tot_take);
            if (take) {
                const int sidx = slot + rk2;
                sel[base + j] = code;
                if (sidx < nbr_cap) {
                    nbr_idx[r * nbr_cap + sidx] = (int32_t)j;
                    nbr_w[r * nbr_cap + sidx] = w;
                }
            }
            slot += tot_take;
        }
        if (c == ci) n_hit += slot - slot_base; else n_miss += slot - slot_base;
        slot_base = slot;
    }
    if (tid == 0) {
        // compacted list of the rows that need the reference's tie order: [0] = count
        if (tie_list && ambiguous) tie_list[1 + atomicAdd(&tie_list[0], 1)] = (int32_t)r;
        nbr_cnt[r] = slot_base < nbr_cap ? slot_base : nbr_cap;
        RowInfo ri;
        ri.thresh = 0.0;
        for (int q = 0; q < 5; ++q) ri.coef[q] = 0.0;
        ri.n_hit = n_hit;
        ri.n_miss = n_miss;
        ri.n_far_hit = 0;
        ri.n_far_miss = 0;
        rinfo[r] = ri;
    }
}


// ---------------------------------------------------------------------------
// ReliefF tie order of the reference.  When several candidates are tied at the k-th
// distance (discrete data), which of them the reference takes is decided by the order
// numba's np.argsort leaves them in (ReliefF.py:157; numba/misc/quicksort.py: median-of-
// three partition with an explicit stack, insertion sort below 15 elements).  For each row
// of relieff_select_kernel's compacted tie list, one CTA stages the float32 distance row in
// ORIGINAL sample order, one thread replays that quicksort on it -- the algorithm is
// sequential -- then scans the order exactly as ReliefF.py:164-175 does and rewrites the
// row's neighbour codes and list.  Untied rows (all rows of continuous data) are not listed.
// ---------------------------------------------------------------------------
// A row's (key, index) pairs and its per-class neighbour counters (n * 8 + n_classes * 4 bytes) are
// staged in shared memory up to this size (n <= 25 599 with 2 classes), in a global scratch of one row
// per CTA beyond it.
constexpr size_t kTieSmemBytes = 200 * 1024;
// uint2 slots of one row of the global scratch: n pairs, then the counters (padded to a whole pair)
__host__ __device__ __forceinline__ int64_t tie_row_pairs(int64_t n, int n_classes) { return n + (n_classes + 1) / 2; }
// The CTA's threads only stage the row.  With global scratch a one-warp CTA lets an SM run 32
// sorts at once instead of 8 (B200, n = 30 000, 2 048 tied rows: 55 ms against 92 ms).
constexpr int kTieThreadsSmem = 256, kTieThreadsGlobal = 32;

// numba's quicksort on (key, index) pairs: the reference permutes an index array R and
// compares A[R[i]]; moving the pairs themselves performs exactly the same swaps.  Keys are
// non-negative float32 distances (and +inf), whose order is that of their bit patterns; only
// the key half is compared, so equal distances stay ties.  Inlined, so that pairs in shared
// memory are accessed as such.
__device__ __forceinline__ uint32_t pkey(const uint2 *P, int64_t i) { return P[i].x; }
__device__ __forceinline__ void pswap(uint2 *P, int64_t a, int64_t b) {
    const uint2 t = P[a]; P[a] = P[b]; P[b] = t;
}
__device__ __forceinline__ void numba_argsort_pairs(uint2 *P, int64_t n) {
    if (n < 2) return;
    int32_t stack_lo[100], stack_hi[100];
    int sp = 1;
    stack_lo[0] = 0; stack_hi[0] = (int32_t)(n - 1);
    while (sp > 0) {
        --sp;
        int64_t low = stack_lo[sp], high = stack_hi[sp];
        while (high - low >= 15) {
            // partition around the median of {low, mid, high}
            const int64_t mid = (low + high) >> 1;
            if (pkey(P, mid) < pkey(P, low)) pswap(P, low, mid);
            if (pkey(P, high) < pkey(P, mid)) pswap(P, high, mid);
            if (pkey(P, mid) < pkey(P, low)) pswap(P, low, mid);
            const uint32_t pivot = pkey(P, mid);
            pswap(P, high, mid);
            int64_t i = low, j = high - 1;
            for (;;) {
                while (i < high && pkey(P, i) < pivot) ++i;
                while (j >= low && pivot < pkey(P, j)) --j;
                if (i >= j) break;
                pswap(P, i, j);
                ++i; --j;
            }
            pswap(P, i, high);
            if (high - i > i - low) {
                if (high > i) { stack_lo[sp] = (int32_t)(i + 1); stack_hi[sp] = (int32_t)high; ++sp; }
                high = i - 1;
            } else {
                if (i > low) { stack_lo[sp] = (int32_t)low; stack_hi[sp] = (int32_t)(i - 1); ++sp; }
                low = i + 1;
            }
        }
        // insertion sort of [low, high]
        for (int64_t i = low + 1; i <= high; ++i) {
            const uint2 kv = P[i];
            int64_t j = i;
            while (j > low && kv.x < P[j - 1].x) { P[j] = P[j - 1]; --j; }
            P[j] = kv;
        }
    }
}

// kShared: the pairs and counters live in dynamic shared memory (shared-memory latency instead of a
// global access per comparison); otherwise in `scratch`, tie_row_pairs(n, n_classes) pairs per CTA.
// A template parameter rather than a pointer chosen at run time, so that the shared instantiation
// keeps shared loads/stores.
template <bool kShared>
__global__ void __launch_bounds__(kShared ? kTieThreadsSmem : kTieThreadsGlobal) relieff_ties_kernel(
    const double *__restrict__ Dc, const int32_t *__restrict__ Dd, int64_t ldn, int64_t n,
    int64_t r0, const int32_t *__restrict__ y, const int64_t *__restrict__ inv_perm,
    int n_classes, int k, const float *__restrict__ class_probs, const int32_t *__restrict__ tie_list,
    uint2 *scratch, int8_t *__restrict__ sel, int32_t *__restrict__ nbr_idx, double *__restrict__ nbr_w,
    int32_t *__restrict__ nbr_cnt, int nbr_cap) {
    extern __shared__ __align__(16) unsigned char ties_smem[];
    if ((int)blockIdx.x >= tie_list[0]) return;
    uint2 *P = kShared ? reinterpret_cast<uint2 *>(ties_smem) : scratch + (int64_t)blockIdx.x * tie_row_pairs(n, n_classes);
    int32_t *found = reinterpret_cast<int32_t *>(P + n);      // neighbours taken per class
    const int64_t r = tie_list[1 + blockIdx.x];
    const int64_t self = r0 + r;
    const int64_t base = r * ldn;
    for (int64_t o = threadIdx.x; o < n; o += blockDim.x) {
        const int64_t j = inv_perm[o];
        const float d = j == self ? __int_as_float(0x7f800000) : (float)load_d(Dc, Dd, base + j);   // ReliefF.py:146-155
        P[o] = make_uint2(__float_as_uint(d), (uint32_t)o);
    }
    for (int64_t j = threadIdx.x; j < n; j += blockDim.x) sel[base + j] = FS_MASK_NONE;
    for (int c = threadIdx.x; c < n_classes; c += blockDim.x) found[c] = 0;
    __syncthreads();
    if (threadIdx.x != 0) return;
    numba_argsort_pairs(P, n);
    const int ci = y[self];
    double denom = 1.0 - (double)class_probs[ci];
    if (denom == 0.0) denom = 1.0;
    // ReliefF.py:164-175 (the scan never ends early in the reference: the target's own class
    // cannot reach k misses; stopping once every class is served selects the same samples)
    int slot = 0, filled = 0;
    for (int64_t q = 0; q < n && filled < n_classes; ++q) {
        const int64_t j = inv_perm[P[q].y];
        const int c = y[j];
        if (found[c] >= k) continue;
        if (++found[c] == k) ++filled;
        sel[base + j] = c == ci ? FS_MASK_NEAR_HIT : FS_MASK_NEAR_MISS;
        if (slot < nbr_cap) {
            nbr_idx[r * nbr_cap + slot] = (int32_t)j;
            nbr_w[r * nbr_cap + slot] = c == ci ? -1.0 : ((double)class_probs[c] / denom) / (double)k;
        }
        ++slot;
    }
    // hits are normalised by the number found (ReliefF.py:211-212)
    const double wh = found[ci] > 0 ? -1.0 / (double)found[ci] : 0.0;
    const int m = slot < nbr_cap ? slot : nbr_cap;
    for (int e = 0; e < m; ++e)
        if (nbr_w[r * nbr_cap + e] == -1.0) nbr_w[r * nbr_cap + e] = wh;
    nbr_cnt[r] = m;
}

void launch_select(fs_dataset *ds, int algo, int use_star, int32_t k, int64_t r0, int64_t R,
                   const double *Dc, const int32_t *Dd, int64_t ldn, int8_t *sel, int8_t *mask_h, int8_t *mask_m,
                   RowInfo *rinfo, int32_t *nbr_idx, double *nbr_w, int32_t *nbr_cnt, int32_t nbr_cap, const float *class_probs,
                   cudaStream_t st, int *launches) {
    if (R == 0) return;
    dim3 grid((unsigned)R);
    if (algo == FS_MULTISURF)
        select_threshold_kernel<FS_MULTISURF><<<grid, 256, 0, st>>>(Dc, Dd, ldn, ds->n, r0, ds->d_y.ptr,
                                                                    ds->d_inv_perm.ptr, use_star, sel, mask_h, mask_m,
                                                                    rinfo);
    else if (algo == FS_SURF)
        select_threshold_kernel<FS_SURF><<<grid, 256, 0, st>>>(Dc, Dd, ldn, ds->n, r0, ds->d_y.ptr,
                                                               ds->d_inv_perm.ptr, use_star, sel, mask_h, mask_m, rinfo);
    else {
        // reference tie order unless FS_B200_RELIEFF_TIES=index (ties then go by sample index)
        const char *env = getenv("FS_B200_RELIEFF_TIES");
        const bool emulate = !(env && env[0] == 'i');
        if (emulate) {
            ds->tie_list.reserve(R + 1);
            FS_CUDA(cudaMemsetAsync(ds->tie_list.ptr, 0, sizeof(int32_t), st));
        }
        relieff_select_kernel<<<grid, 256, 0, st>>>(Dc, Dd, ldn, ds->n, r0, ds->d_y.ptr, ds->d_cls_start.ptr,
                                                    ds->n_classes, k, class_probs, sel, rinfo, nbr_idx, nbr_w,
                                                    nbr_cnt, nbr_cap, emulate ? ds->tie_list.ptr : nullptr);
        if (emulate) {
            FS_CUDA(cudaGetLastError());
            ++*launches;
            // one CTA per row of the compacted list (CTAs beyond the list's length exit at once; no
            // host round trip for the count)
            const size_t row_bytes = (size_t)ds->n * sizeof(uint2) + (size_t)ds->n_classes * sizeof(int32_t);
            const bool smem = row_bytes <= kTieSmemBytes;
            auto kernel = smem ? relieff_ties_kernel<true> : relieff_ties_kernel<false>;
            if (smem)
                FS_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)row_bytes));
            else
                ds->tie_pairs.reserve((size_t)R * tie_row_pairs(ds->n, ds->n_classes));
            kernel<<<grid, smem ? kTieThreadsSmem : kTieThreadsGlobal, smem ? row_bytes : 0, st>>>(
                Dc, Dd, ldn, ds->n, r0, ds->d_y.ptr, ds->d_inv_perm.ptr, ds->n_classes, k, class_probs,
                ds->tie_list.ptr, smem ? nullptr : ds->tie_pairs.ptr, sel, nbr_idx, nbr_w, nbr_cnt, nbr_cap);
        }
    }
    FS_CUDA(cudaGetLastError());
    ++*launches;
}

}  // namespace fs
