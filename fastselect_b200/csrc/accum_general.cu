// accum_general.cu -- CUDA-core per-feature weight accumulation for continuous
// (and wide discrete) columns, the ReliefF neighbour gathers (general columns, and
// the value codes of the one-hot columns), and the final reduction of the partial
// weight vectors.
//
// Replaces the hit/miss accumulation loops and normalisation of the reference
// kernels (MultiSURF.py:198-251, SURF.py:165-195, ReliefF.py:181-216) in the
// matrix form  wsum[f] = sum_i sum_j c_ij * term_f(i, j),  where c_ij is the
// coefficient of the pair's neighbour code for target i (RowInfo::coef: sign and
// 1/|H_i|, 1/|M_i| folded in).
//
// accum_general_kernel: one thread per feature column (coalesced 128-byte row
// segments per warp), 16 target rows held in registers, the samples j streamed
// once per 16 targets; the 16 x 128 coefficient tile of each j-tile is decoded
// from the int8 codes into shared memory.  float32 products are accumulated in
// float32 over one 128-sample tile and then folded into a float64 accumulator, so
// the result is accurate to ~1e-7 relative while the inner loop is 2 FP32
// instructions per (pair, feature) on float32 data (the column's 1/range is applied once
// to the column total).  Partials are written per (row chunk, feature)
// and reduced in a fixed order: results are bitwise reproducible.
#include <algorithm>

#include "common.cuh"

namespace fs {

constexpr int kAccThreads = 128;  // features per CTA
constexpr int kAccRows = 16;      // target rows per register block
constexpr int kAccJT = 128;       // samples per coefficient tile

__device__ __forceinline__ float term_cont32(float a, float b, float r) {
    return __fmul_rn(fabsf(__fsub_rn(a, b)), r);
}
// SURF.py:153-158: float64 product, stored as float32
__device__ __forceinline__ float term_cont32(double a, double b, float r) {
    return (float)__dmul_rn(fabs(__dsub_rn(a, b)), (double)r);
}

// Inner-loop term of the accumulation.  float32 data: |a - b| only (FSUB, then one FFMA with
// the |.| operand modifier) -- the column's 1/range is a common factor of every term of the
// column and is applied once to the column's total, so the loop is 2 FP32 instructions per
// (pair, feature) instead of 3.  The reference rounds |a-b|*r per term in float32 and adds in
// float32 (MultiSURF.py:184-243); either way the sum carries float32 accumulation-order noise
// of ~1e-7 relative, far inside the 1e-5 tolerance.  float64 data (SURF): the reference's
// float64 product, rounded to float32 (SURF.py:153-158).
__device__ __forceinline__ float absdiff32(float a, float b, float) { return fabsf(__fsub_rn(a, b)); }
__device__ __forceinline__ float absdiff32(double a, double b, float r) { return term_cont32(a, b, r); }
template <typename T>
__device__ __forceinline__ double column_scale(float r) { return sizeof(T) == 4 ? (double)r : 1.0; }

// One 128-sample tile of the accumulation for this thread's column: sample values are fetched
// kAhead rows ahead of their use, the 16 coefficients of a sample come as four 16-byte broadcast
// loads from shared memory.  FULL: the tile has all kAccJT samples (no bounds checks).
template <typename T, bool FULL, bool CMP>
__device__ __forceinline__ void accumulate_tile(const T *__restrict__ xp, int64_t ld, int nj,
                                                const float (*__restrict__ coef)[kAccRows],
                                                const T (&xi)[kAccRows], float r, float (&acc)[kAccRows]) {
    constexpr int kAhead = 8;
    const int jend = FULL ? kAccJT : nj;
#pragma unroll 1
    for (int jb = 0; jb < jend; jb += kAhead, xp += (int64_t)kAhead * ld) {
        T xj[kAhead];
#pragma unroll
        for (int u = 0; u < kAhead; ++u) xj[u] = (FULL || jb + u < nj) ? xp[(int64_t)u * ld] : xp[0];
#pragma unroll
        for (int u = 0; u < kAhead; ++u) {
            // samples beyond nj have coefficient 0 in the tile: no check needed, the term vanishes
            const float4 *cp = reinterpret_cast<const float4 *>(coef[jb + u]);
            float c[kAccRows];
#pragma unroll
            for (int q = 0; q < kAccRows / 4; ++q) {
                const float4 v = cp[q];
                c[4 * q] = v.x; c[4 * q + 1] = v.y; c[4 * q + 2] = v.z; c[4 * q + 3] = v.w;
            }
            if (CMP) {
#pragma unroll
                for (int a = 0; a < kAccRows; ++a) acc[a] += (xi[a] != xj[u]) ? c[a] : 0.0f;
            } else {
#pragma unroll
                for (int a = 0; a < kAccRows; ++a) acc[a] = fmaf(c[a], absdiff32(xi[a], xj[u], r), acc[a]);
            }
        }
    }
}

template <typename T>
__global__ void __launch_bounds__(kAccThreads)
accum_general_kernel(const T *__restrict__ xg, int64_t n, int64_t ld, const float *__restrict__ recip,
                     const uint8_t *__restrict__ ctype, const T *__restrict__ xa, const int8_t *__restrict__ sel,
                     int64_t ldn, const RowInfo *__restrict__ rinfo, int64_t R, int64_t rows_per_cta,
                     double *__restrict__ partial, int FT) {
    // FT: columns per 128-byte chunk of the matrix the chunk types were laid out for (32 float32 / 16 float64)
    __shared__ __align__(16) float scoef[2][kAccJT][kAccRows];
    __shared__ float stab[kAccRows][5];

    const int tid = threadIdx.x;
    const int64_t f = (int64_t)blockIdx.y * kAccThreads + tid;   // blockIdx.x = row chunk (fastest)
    const bool live = f < ld;
    const int64_t fc = live ? f : ld - 1;
    const float r = recip[fc];
    const bool cmp = ctype[fc / FT] == kChunkCompare;
    const int64_t r_begin = (int64_t)blockIdx.x * rows_per_cta;
    const int64_t r_end = r_begin + rows_per_cta < R ? r_begin + rows_per_cta : R;

    double total = 0.0;
    for (int64_t rb = r_begin; rb < r_end; rb += kAccRows) {
        const int nr = (int)(r_end - rb < kAccRows ? r_end - rb : kAccRows);
        T xi[kAccRows];
#pragma unroll
        for (int a = 0; a < kAccRows; ++a) xi[a] = xa[(rb + (a < nr ? a : nr - 1)) * ld + fc];
        __syncthreads();
        if (tid < kAccRows * 5) {
            const int a = tid / 5, q = tid % 5;
            stab[a][q] = a < nr ? (float)rinfo[rb + a].coef[q] : 0.0f;
        }
        // neighbour codes of a sample tile: thread = (target row a, 16 consecutive samples), one
        // 16-byte load.  The codes of tile t + 1 are fetched while tile t is being accumulated and
        // the decoded coefficient tiles are double-buffered, so the global-load latency of the
        // codes is hidden and one barrier per tile suffices.
        const int ca = tid >> 3, cchunk = tid & 7;
        uint4 code = make_uint4(0u, 0u, 0u, 0u);
        auto fetch_codes = [&](int64_t j0) {
            if (ca < nr) code = *reinterpret_cast<const uint4 *>(sel + (rb + ca) * ldn + j0 + 16 * cchunk);
        };
        __syncthreads();                       // stab
        fetch_codes(0);
        int buf = 0;
        for (int64_t j0 = 0; j0 < n; j0 += kAccJT, buf ^= 1) {
            const int nj = (int)(n - j0 < kAccJT ? n - j0 : kAccJT);
            // decode 16 coefficients of this thread's row (codes beyond the last sample are padding)
            {
                const uint32_t cw[4] = {code.x, code.y, code.z, code.w};
#pragma unroll
                for (int q = 0; q < 16; ++q) {
                    const int jj = 16 * cchunk + q;
                    uint32_t cd = (cw[q >> 2] >> (8 * (q & 3))) & 0xffu;
                    cd = cd > 4u ? 0u : cd;             // padding bytes beyond sample n are not codes
                    scoef[buf][jj][ca] = (ca < nr && jj < nj) ? stab[ca][cd] : 0.0f;
                }
            }
            __syncthreads();
            if (j0 + kAccJT < n) fetch_codes(j0 + kAccJT);
            float acc[kAccRows];
#pragma unroll
            for (int a = 0; a < kAccRows; ++a) acc[a] = 0.0f;
            // the chunk type is uniform per warp (float32: 32 columns per chunk), so this branch does
            // not diverge; full tiles run without any per-sample bounds check
            const T *xp = xg + j0 * ld + fc;
            if (nj == kAccJT) {
                if (cmp) accumulate_tile<T, true, true>(xp, ld, nj, scoef[buf], xi, r, acc);
                else accumulate_tile<T, true, false>(xp, ld, nj, scoef[buf], xi, r, acc);
            } else {
                if (cmp) accumulate_tile<T, false, true>(xp, ld, nj, scoef[buf], xi, r, acc);
                else accumulate_tile<T, false, false>(xp, ld, nj, scoef[buf], xi, r, acc);
            }
#pragma unroll
            for (int a = 0; a < kAccRows; ++a) total += (double)acc[a];
        }
    }
    if (live) partial[(int64_t)blockIdx.x * ld + f] = cmp ? total : total * column_scale<T>(r);
}

// ReliefF: per target row at most C*k neighbours; one thread per feature gathers
// the neighbour rows (coalesced) -- HBM/L2-bound: n*k*C*p*sizeof(T) bytes.
template <typename T>
__global__ void __launch_bounds__(kAccThreads)
relieff_gather_kernel(const T *__restrict__ xg, int64_t ld, const float *__restrict__ recip,
                      const uint8_t *__restrict__ ctype, const T *__restrict__ xa,
                      const int32_t *__restrict__ nbr_idx, const double *__restrict__ nbr_w,
                      const int32_t *__restrict__ nbr_cnt, int nbr_cap, int64_t R, int64_t rows_per_cta,
                      double *__restrict__ partial) {
    constexpr int FT = kChunkBytes / sizeof(T);
    __shared__ int32_t sidx[256];
    __shared__ double sw[256];
    const int tid = threadIdx.x;
    const int64_t f = (int64_t)blockIdx.y * kAccThreads + tid;
    const bool live = f < ld;
    const int64_t fc = live ? f : ld - 1;
    const float r = recip[fc];
    const bool cmp = ctype[fc / FT] == kChunkCompare;
    const int64_t r_begin = (int64_t)blockIdx.x * rows_per_cta;
    const int64_t r_end = r_begin + rows_per_cta < R ? r_begin + rows_per_cta : R;
    double total = 0.0;
    for (int64_t row = r_begin; row < r_end; ++row) {
        const T xi = xa[row * ld + fc];
        const int cnt = nbr_cnt[row];
        for (int s0 = 0; s0 < cnt; s0 += 256) {
            const int m = cnt - s0 < 256 ? cnt - s0 : 256;
            __syncthreads();
            for (int e = tid; e < m; e += kAccThreads) {
                sidx[e] = nbr_idx[row * nbr_cap + s0 + e];
                sw[e] = nbr_w[row * nbr_cap + s0 + e];
            }
            __syncthreads();
#pragma unroll 4
            for (int e = 0; e < m; ++e) {
                const T xj = xg[(int64_t)sidx[e] * ld + fc];
                // ReliefF.py:151-154: float32 term, accumulated in float64
                double t;
                if (cmp) t = (xi != xj) ? 1.0 : 0.0;
                else if (sizeof(T) == 4) t = (double)__fmul_rn(fabsf(__fsub_rn((float)xi, (float)xj)), r);
                else t = __dmul_rn(fabs(__dsub_rn((double)xi, (double)xj)), (double)r);
                total = __fma_rn(sw[e], t, total);
            }
        }
    }
    if (live) partial[(int64_t)blockIdx.x * ld + f] = total;
}

// Rows per CTA.  CTAs that share a 128-column strip of X (same blockIdx.y) are launched
// back to back (blockIdx.x fastest), so with ~128 row chunks per strip only ~8 strips are
// in flight on the chip at a time and each strip (n x 512 B) stays L2-resident while its
// CTAs sweep it once per 16 target rows.
static int64_t rows_per_cta_for(int64_t R, int64_t ld) {
    (void)ld;
    const int64_t want_chunks = 128;
    return std::max<int64_t>(kAccRows, round_up(ceil_div(R, want_chunks), kAccRows));
}

int64_t accum_general_partials(const WorkSet &ws, int64_t R) {
    if (ws.pg == 0 || R == 0) return 0;
    return ceil_div(R, rows_per_cta_for(R, ws.ldg));
}

void launch_accum_general(const WorkSet &ws, int64_t n, int64_t row0, const int8_t *sel, int64_t ldn,
                          const RowInfo *rinfo, int64_t R, double *partial, int64_t n_part, cudaStream_t st,
                          int *launches) {
    if (ws.pg == 0 || R == 0) return;
    const int64_t rows = rows_per_cta_for(R, ws.ldg);
    dim3 grid((unsigned)n_part, (unsigned)ceil_div(ws.ldg, kAccThreads));
    const size_t a_off = (size_t)row0 * ws.ldg;        // the target rows: a view of the matrix
    // float64 arithmetic (SURF) with only continuous columns: the reference STORES each term as float32
    // (diffs_from_i, SURF.py:143-158) and adds float32 sums, so the accumulation runs on the float32 image
    // of the offset-free columns (x - column minimum: |x'| <= range, so the image keeps 2^-24 of the RANGE,
    // not of |x|) with the float32 kernel -- FP32 pipe instead of three FP64 operations per (pair, feature).
    // float64 data with compare columns stays on the float64 kernel.
    if (ws.elem == 8 && ws.have_xg32) {
        accum_general_kernel<float><<<grid, kAccThreads, 0, st>>>(
            ws.xg32.ptr, n, ws.ldg, ws.rg.ptr, ws.ctype.ptr, ws.xg32.ptr + a_off, sel, ldn, rinfo, R, rows,
            partial, kChunkBytes / 8);
    } else if (ws.elem == 4) {
        const float *xg = reinterpret_cast<const float *>(ws.xg.ptr);
        accum_general_kernel<float><<<grid, kAccThreads, 0, st>>>(
            xg, n, ws.ldg, ws.rg.ptr, ws.ctype.ptr, xg + a_off, sel, ldn, rinfo, R, rows, partial, kChunkBytes / 4);
    } else {
        const double *xg = reinterpret_cast<const double *>(ws.xg.ptr);
        accum_general_kernel<double><<<grid, kAccThreads, 0, st>>>(
            xg, n, ws.ldg, ws.rg.ptr, ws.ctype.ptr, xg + a_off, sel, ldn, rinfo, R, rows, partial, kChunkBytes / 8);
    }
    FS_CUDA(cudaGetLastError());
    ++*launches;
}

void launch_relieff_gather(const WorkSet &ws, int64_t n, int64_t row0, const int32_t *nbr_idx,
                           const double *nbr_w, const int32_t *nbr_cnt, int32_t nbr_cap, int64_t R,
                           double *partial, int64_t n_part, cudaStream_t st, int *launches) {
    (void)n;
    if (ws.pg == 0 || R == 0) return;
    const int64_t rows = rows_per_cta_for(R, ws.ldg);
    dim3 grid((unsigned)n_part, (unsigned)ceil_div(ws.ldg, kAccThreads));
    const size_t a_off = (size_t)row0 * ws.ldg;        // the target rows: a view of the matrix
    if (ws.elem == 4) {
        const float *xg = reinterpret_cast<const float *>(ws.xg.ptr);
        relieff_gather_kernel<float><<<grid, kAccThreads, 0, st>>>(xg, ws.ldg, ws.rg.ptr, ws.ctype.ptr, xg + a_off, nbr_idx,
                                                                   nbr_w, nbr_cnt, nbr_cap, R, rows, partial);
    } else {
        const double *xg = reinterpret_cast<const double *>(ws.xg.ptr);
        relieff_gather_kernel<double><<<grid, kAccThreads, 0, st>>>(xg, ws.ldg, ws.rg.ptr, ws.ctype.ptr, xg + a_off, nbr_idx,
                                                                    nbr_w, nbr_cnt, nbr_cap, R, rows, partial);
    }
    FS_CUDA(cudaGetLastError());
    ++*launches;
}

// ReliefF on the one-hot columns: sparse neighbour lists, value codes compared directly
// (ReliefF.py:181-216; at most C*k neighbours per target) -- HBM/L2-bound gather.
__global__ void __launch_bounds__(128) relieff_codes_gather_kernel(
    const uint8_t *__restrict__ codes, int64_t ldc, int64_t pt, int64_t row0,
    const int32_t *__restrict__ nbr_idx, const double *__restrict__ nbr_w, const int32_t *__restrict__ nbr_cnt,
    int nbr_cap, int64_t R, int64_t rows_per_cta, double *__restrict__ partial) {
    __shared__ int32_t sidx[256];
    __shared__ double sw[256];
    const int tid = threadIdx.x;
    const int64_t c = (int64_t)blockIdx.y * 128 + tid;
    const bool live = c < pt;
    const int64_t cc = live ? c : pt - 1;
    const int64_t r_begin = (int64_t)blockIdx.x * rows_per_cta;
    const int64_t r_end = r_begin + rows_per_cta < R ? r_begin + rows_per_cta : R;
    double total = 0.0;
    for (int64_t row = r_begin; row < r_end; ++row) {
        const uint8_t ci = codes[(row0 + row) * ldc + cc];
        const int cnt = nbr_cnt[row];
        for (int s0 = 0; s0 < cnt; s0 += 256) {
            const int m = cnt - s0 < 256 ? cnt - s0 : 256;
            __syncthreads();
            for (int e = tid; e < m; e += 128) {
                sidx[e] = nbr_idx[row * nbr_cap + s0 + e];
                sw[e] = nbr_w[row * nbr_cap + s0 + e];
            }
            __syncthreads();
#pragma unroll 4
            for (int e = 0; e < m; ++e) {
                const uint8_t cj = codes[(int64_t)sidx[e] * ldc + cc];
                total += (ci != cj) ? sw[e] : 0.0;
            }
        }
    }
    if (live) partial[(int64_t)blockIdx.x * pt + c] = total;
}

__global__ void __launch_bounds__(256) reduce_code_partials_kernel(const double *__restrict__ partial, int64_t n_part,
                                                                   int64_t pt, const int64_t *__restrict__ tout,
                                                                   double *__restrict__ wsum) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= pt) return;
    double s = 0.0;
    for (int64_t q = 0; q < n_part; ++q) s += partial[q * pt + c];
    wsum[tout[c]] += s;
}

// Grid: 128-column strips x chunks of target rows, about 8 CTAs per SM of a B200 (148 SMs) in all.
void launch_relieff_codes(const WorkSet &ws, int64_t row0, const int32_t *nbr_idx, const double *nbr_w,
                          const int32_t *nbr_cnt, int32_t nbr_cap, int64_t R, DevBuf<double> &partial, double *wsum,
                          cudaStream_t st, int *launches) {
    const int64_t ctiles = ceil_div(ws.pt, 128);
    const int64_t want = std::max<int64_t>(1, ceil_div(148 * 8, ctiles));
    const int64_t rows = std::max<int64_t>(1, ceil_div(R, want));
    const int64_t n_part = ceil_div(R, rows);
    partial.reserve((size_t)n_part * ws.pt);
    dim3 grid((unsigned)n_part, (unsigned)ctiles);
    relieff_codes_gather_kernel<<<grid, 128, 0, st>>>(ws.codes.ptr, ws.ldc, ws.pt, row0, nbr_idx, nbr_w, nbr_cnt, nbr_cap, R,
                                                      rows, partial.ptr);
    FS_CUDA(cudaGetLastError());
    reduce_code_partials_kernel<<<(unsigned)ceil_div(ws.pt, 256), 256, 0, st>>>(partial.ptr, n_part, ws.pt, ws.tout.ptr, wsum);
    FS_CUDA(cudaGetLastError());
    *launches += 2;
}

__global__ void __launch_bounds__(256) reduce_partials_kernel(const double *__restrict__ partial, int64_t n_part,
                                                              int64_t ld, const int64_t *__restrict__ gout,
                                                              int64_t pg, double *__restrict__ wsum) {
    const int64_t c = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (c >= pg) return;
    const int64_t o = gout[c];
    if (o < 0) return;
    double s = 0.0;
    for (int64_t q = 0; q < n_part; ++q) s += partial[q * ld + c];
    wsum[o] += s;
}

void launch_reduce_partials(const WorkSet &ws, const double *partial, int64_t n_part, double *wsum,
                            cudaStream_t st, int *launches) {
    if (ws.pg == 0 || n_part == 0) return;
    reduce_partials_kernel<<<(unsigned)ceil_div(ws.pg, 256), 256, 0, st>>>(partial, n_part, ws.ldg, ws.gout.ptr,
                                                                          ws.pg, wsum);
    FS_CUDA(cudaGetLastError());
    ++*launches;
}

}  // namespace fs
