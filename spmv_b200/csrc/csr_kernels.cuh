// csr_kernels.cuh -- kernels that work directly on the CSR arrays:
//   csr_reforder_kernel   Method_Serial    (bit-identical summation order to the reference)
//   csr_vector_kernel     Method_Parallel  (sub-warp per row, batched scalar stream loads through L1)
//   row_block_kernel      Method_Balanced  (one warp per nnz-balanced row block of the csrSplitter)
//   band_*_kernel         band-major ("virtual row") copy that keeps the gathered slice of x in L2
#pragma once
#include "common.cuh"

namespace sb {

// ------------------------------------------------------------------------------------------------
// Method_Serial.  Replaces spmv_serial_cpp_{d,s} (reference src/src_spmv/serial_spmv.c:9-37) and
// Dot_Product_Avx2_{d,s} (inner_spmv.h:232-354).  The AVX2 register becomes a group of L lanes
// (L = 4 for fp64, 8 for fp32): lane l owns elements l, l+L, ... as an FMA chain from +0, the
// horizontal add is the same tree ((l0+l1)+(l2+l3) resp. ((l0+l4)+(l2+l6))+((l1+l5)+(l3+l7))) done
// with xor-shuffles, and lane 0 folds in the len%L tail exactly as the reference's compiled remainder
// loop does (see oracle/spmv_oracle.c row_dot_s for the fp32 in-order 4-wide step).  Result: y is
// bitwise equal to the reference's Method_Serial.
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void __launch_bounds__(kThreads)
csr_reforder_kernel(int m, const int *__restrict__ rowptr, const int *__restrict__ col,
                    const T *__restrict__ val, const T *__restrict__ x, T *__restrict__ y)
{
    constexpr int L = sizeof(T) == 8 ? 4 : 8;
    const long long gt = (long long)blockIdx.x * kThreads + threadIdx.x;
    const long long row_l = gt / L;
    const int lane = threadIdx.x & (L - 1);
    const bool valid = row_l < m;
    const int row = valid ? (int)row_l : 0;
    const int start = valid ? rowptr[row] : 0;
    const int end = valid ? rowptr[row + 1] : 0;
    const int len = end - start;
    const int groups = len / L;

    T acc = 0;
    for (int g = 0; g < groups; ++g) {
        const int j = start + g * L + lane;
        acc = fma_t(val[j], x[col[j]], acc);
    }
    if (L == 4) {
        acc += __shfl_xor_sync(kFull, acc, 1);
        acc += __shfl_xor_sync(kFull, acc, 2);
    } else {
        acc += __shfl_xor_sync(kFull, acc, 4);
        acc += __shfl_xor_sync(kFull, acc, 2);
        acc += __shfl_xor_sync(kFull, acc, 1);
    }
    if (valid && lane == 0) {
        T result = acc;  // all lanes are +0 when groups == 0, and (+0)+(+0) = +0 as in the reference
        int j = start + groups * L;
        if (sizeof(T) == 4 && end - j >= 4) {
            // the pinned reference build adds four UNFUSED products in order here
            float p0 = __fmul_rn((float)val[j], (float)x[col[j]]);
            float p1 = __fmul_rn((float)val[j + 1], (float)x[col[j + 1]]);
            float p2 = __fmul_rn((float)val[j + 2], (float)x[col[j + 2]]);
            float p3 = __fmul_rn((float)val[j + 3], (float)x[col[j + 3]]);
            float r = (float)result;
            r = __fadd_rn(r, p0);
            r = __fadd_rn(r, p1);
            r = __fadd_rn(r, p2);
            r = __fadd_rn(r, p3);
            result = (T)r;
            j += 4;
        }
        for (; j < end; ++j) result = fma_t(val[j], x[col[j]], result);
        y[row] = result;
    }
}

// ------------------------------------------------------------------------------------------------
// One row, cooperatively by `tpr` lanes, in predicated batches of 8 entries per lane: every stream load of a batch
// is in flight before the first gather, so a row of up to 8*tpr entries costs three dependent memory round trips
// (rowptr, col/val, x) however it is aligned -- what a latency-bound (small, L2-cold) matrix needs.  Scalar loads
// that allocate in L1 (L2 evict-first): the tpr lanes of a row walk it with stride tpr, so one 32-byte sector
// serves several lanes and is fetched from L2 once.  (Measured and dropped in round 1, fraction of the HBM peak for
// aligned 4-element chunk loads / a plain scalar loop / this: C1 0.50 / 0.60 / 0.62, C2 0.385 / 0.36 / 0.40,
// C4 0.69 / 0.74 / 0.89.)
// ------------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ T row_partial(int start, int end, int sl, int tpr, const int *__restrict__ col,
                                         const T *__restrict__ val, const T *__restrict__ x, uint64_t pl, uint64_t pf)
{
    // A lane adds at most kBlock / 2 batches into one FMA chain: a lane that walks a very long row alone (small
    // tpr on a skewed matrix) folds block sums instead of piling ~sqrt(len) ulps into a single chain, which would
    // miss the 8*eps*sum|a x| bound.  Fixed order either way: bitwise reproducible.
    constexpr int kBlock = 64;
    constexpr int B = 8;  // (4 per batch in 32 registers at full occupancy measured slower on every matrix)
    T sum = 0;
    int batches = 0;
    T acc = 0;
    for (int j = start + sl; j < end; j += B * tpr) {
        int c[B];
        T v[B];
#pragma unroll
        for (int k = 0; k < B; ++k) {
            const int jj = j + k * tpr;
            c[k] = jj < end ? ldg_cached(col + jj, pf) : -1;
        }
#pragma unroll
        for (int k = 0; k < B; ++k) {
            const int jj = j + k * tpr;
            v[k] = jj < end ? ldg_cached(val + jj, pf) : (T)0;
        }
#pragma unroll
        for (int k = 0; k < B; ++k)
            if (c[k] >= 0) acc = fma_t(v[k], ldg_x(x + c[k], pl), acc);
        if (++batches == kBlock / 2) { sum += acc; acc = 0; batches = 0; }
    }
    sum += acc;
    return sum;
}

// ------------------------------------------------------------------------------------------------
// Method_Parallel.  Replaces spmv_parallel_cpp_{d,s} (reference src/src_spmv/parallel_spmv.c:5-34):
// the OpenMP row loop becomes a grid of sub-warps, TPR lanes per row with TPR = 2^k ~ mean row
// length / 4 chosen at create.  Fixed butterfly reduction => bitwise reproducible.
// ------------------------------------------------------------------------------------------------
template <typename T, int TPR, bool FUSE, typename Store>
__device__ __forceinline__ void csr_vector_body(unsigned tid, int row0, int m, int long_thr,
                                                const int *__restrict__ rowptr, const int *__restrict__ col,
                                                const T *__restrict__ val, const T *__restrict__ x, const Store &store,
                                                int fuse_bands, int band_m, const T *__restrict__ vy)
{
    // rows [row0, m): the whole matrix in one launch, or one band / row chunk of the pipelined host path.
    // FUSE (pipelined host path only; a separate instantiation so that the plain kernel keeps its 40 registers):
    // these are rows of the LAST band of a band-major copy; the partial sums of the fuse_bands earlier bands
    // (vy, complete: written by an earlier launch) are folded in here, in band order, and the final value goes
    // to row (virtual row - fuse_bands*band_m) of y -- band_reduce_kernel without its own pass.
    const uint64_t pl = policy_evict_last(), pf = policy_evict_first();
    const long long gt = (long long)blockIdx.x * kThreads + tid;
    const long long row_l = row0 + gt / TPR;
    const int sl = tid & (TPR - 1);
    bool valid = row_l < m;
    const int row = valid ? (int)row_l : 0;
    int start = valid ? rowptr[row] : 0;
    int end = valid ? rowptr[row + 1] : 0;
    if (end - start > long_thr) { valid = false; end = start; }  // hub row: left to the long-row path
    int out_row = row;
    T prev = 0;
    if (FUSE) {
        out_row = row - fuse_bands * band_m;
        if (valid && sl == 0) {  // issued before the row walk: in flight while the row is being summed
            prev = ldg_stream(vy + out_row);
            for (int b = 1; b < fuse_bands; ++b) prev += ldg_stream(vy + (size_t)b * band_m + out_row);
        }
    }
    const auto early = store.early(valid && sl == 0, out_row);
    T sum = row_partial<T>(start, end, sl, TPR, col, val, x, pl, pf);
    sum = group_sum_c<T, TPR>(sum);
    if (valid && sl == 0) store.put(out_row, FUSE ? prev + sum : sum, early);
}

template <typename T, int TPR, bool PEERS, bool FUSE>
__global__ void __launch_bounds__(kThreads)
csr_vector_kernel(int row0, int m, int long_thr, const int *__restrict__ rowptr, const int *__restrict__ col,
                  const T *__restrict__ val, const T *__restrict__ x, T *__restrict__ y, const PeerList<T> peers,
                  int fuse_bands, int band_m, const T *__restrict__ vy)
{
    csr_vector_body<T, TPR, FUSE>(threadIdx.x, row0, m, long_thr, rowptr, col, val, x, PeerStore<PEERS, T>{y, peers},
                                  fuse_bands, band_m, vy);
}

// spmv_b200_spmv_axpby on an unbanded Method_Parallel handle with one lane per row, without row bins or long-row list:
// y <- alpha A x + beta y (instantiated for TPR = 1 only, see axpby_path)
template <typename T, int TPR>
__global__ void __launch_bounds__(kThreads)
csr_vector_axpby_kernel(int row0, int m, int long_thr, const int *__restrict__ rowptr, const int *__restrict__ col,
                        const T *__restrict__ val, const T *__restrict__ x, const ScaledStore<T> store)
{
    csr_vector_body<T, TPR, false>(threadIdx.x, row0, m, long_thr, rowptr, col, val, x, store, 0, 0,
                                   (const T *)nullptr);
}

// spmv_b200_spmv_axpby_dot on the same handles: the scaled store, and the CTA's partial of w . y (DotStore)
template <typename T, int TPR>
__global__ void __launch_bounds__(kThreads)
csr_vector_axpby_dot_kernel(int row0, int m, int long_thr, const int *__restrict__ rowptr, const int *__restrict__ col,
                            const T *__restrict__ val, const T *__restrict__ x, const DotArgs<T> d)
{
    double acc = 0;
    csr_vector_body<T, TPR, false>(threadIdx.x, row0, m, long_thr, rowptr, col, val, x, DotStore<T>{d, acc}, 0, 0,
                                   (const T *)nullptr);
    dot_partial(acc, d.partials);
}

// spmv_b200_spmv_shifted on the same handles: the shifted store, and the CTA's partials of x . y and y . y (ShiftStore)
template <typename T, int TPR>
__global__ void __launch_bounds__(kThreads)
csr_vector_shift_kernel(int row0, int m, int long_thr, const int *__restrict__ rowptr, const int *__restrict__ col,
                        const T *__restrict__ val, const T *__restrict__ x, const ShiftArgs<T> d)
{
    double xy = 0, yy = 0;
    csr_vector_body<T, TPR, false>(threadIdx.x, row0, m, long_thr, rowptr, col, val, x, ShiftStore<T>{d, xy, yy}, 0,
                                   0, (const T *)nullptr);
    shift_partials(xy, yy, d.xy, d.yy);
}

// The same row walk over a LIST of rows: Method_Parallel on matrices whose rows are short but not uniformly so
// (power-law graphs).  Rows are binned by length class at create and every bin gets the lanes per row that fit it,
// so a warp only ever holds rows of similar length (no lane group waiting for a 100-entry neighbour).
template <typename T, int TPR, bool PEERS>
__global__ void __launch_bounds__(kThreads)
csr_vector_list_kernel(int count, const int *__restrict__ list, const int *__restrict__ rowptr,
                       const int *__restrict__ col, const T *__restrict__ val, const T *__restrict__ x,
                       T *__restrict__ y, const PeerList<T> peers)
{
    const uint64_t pl = policy_evict_last(), pf = policy_evict_first();
    const long long gt = (long long)blockIdx.x * kThreads + threadIdx.x;
    const long long idx = gt / TPR;
    const int sl = threadIdx.x & (TPR - 1);
    const bool valid = idx < count;
    const int row = valid ? list[idx] : 0;
    const int start = valid ? rowptr[row] : 0;
    const int end = valid ? rowptr[row + 1] : 0;
    T sum = row_partial<T>(start, end, sl, TPR, col, val, x, pl, pf);
    sum = group_sum_c<T, TPR>(sum);
    if (valid && sl == 0) store_y<PEERS>(y, peers, row, sum);
}

// bin of a row by its length: 0 (<= 8), 1 (<= 32), 2 (<= 128), 3 (longer: long-row path)
__global__ void row_bin_kernel(int m, const int *__restrict__ rowptr, unsigned char *__restrict__ bin, int *__restrict__ ids)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= m) return;
    const int len = rowptr[r + 1] - rowptr[r];
    bin[r] = (unsigned char)(len <= 8 ? 0 : len <= 32 ? 1 : len <= 128 ? 2 : 3);
    ids[r] = r;
}

// ------------------------------------------------------------------------------------------------
// Method_Balanced.  Replaces spmv_parallel_balanced_cpp_{d,s} (reference
// src/src_spmv/parallel_balanced_spmv.c:77-125): "thread t does rows csrSplitter[t]..csrSplitter[t+1]"
// with the thread replaced by a warp and T = number of row blocks (~block_nnz non-zeros each, the
// same a9 splitter formula).  Inside its block the warp picks lanes-per-row from the block's own
// mean row length, so short-row and long-row regions of one matrix each get a fitting geometry.
// Block 0 starts at row 0 (the reference leaves leading empty rows unwritten).
// ------------------------------------------------------------------------------------------------
template <typename T, bool PEERS, int TPR>
__device__ __forceinline__ void row_block_body(int r0, int r1, int lane, const int *__restrict__ rowptr,
                                               const int *__restrict__ col, const T *__restrict__ val,
                                               const T *__restrict__ x, T *__restrict__ y, const PeerList<T> &peers,
                                               uint64_t pl, uint64_t pf)
{
    constexpr int rows_per_iter = 32 / TPR;
    const int sub = lane / TPR, sl = lane & (TPR - 1);
    // (staging the block's row pointers with one coalesced load + shuffles was measured: no gain, C4 0.72 -> 0.69)
    for (int base = r0; base < r1; base += rows_per_iter) {
        const int row = base + sub;
        const bool valid = row < r1;
        const int start = valid ? rowptr[row] : 0;
        const int end = valid ? rowptr[row + 1] : 0;
        T sum = row_partial<T>(start, end, sl, TPR, col, val, x, pl, pf);
        sum = group_sum_c<T, TPR>(sum);
        if (valid && sl == 0) store_y<PEERS>(y, peers, row, sum);
    }
}

template <typename T, bool PEERS>
__global__ void __launch_bounds__(kThreads)
row_block_kernel(int parts, const int *__restrict__ splitter, const int *__restrict__ rowptr,
                 const int *__restrict__ col, const T *__restrict__ val, const T *__restrict__ x,
                 T *__restrict__ y, const PeerList<T> peers)
{
    const uint64_t pl = policy_evict_last(), pf = policy_evict_first();
    const int w = (int)(((long long)blockIdx.x * kThreads + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (w >= parts) return;
    const int r0 = w == 0 ? 0 : splitter[w];
    const int r1 = splitter[w + 1];
    const int nrows = r1 - r0;
    if (nrows <= 0) return;
    const int nz = rowptr[r1] - rowptr[r0];
    const int avg = (nz + nrows - 1) / nrows;
    // lanes per row from the block's own mean row length (warp-uniform): compile-time bodies so that the row
    // walk unrolls and the butterfly has a fixed depth
#define SB_BODY(N) row_block_body<T, PEERS, N>(r0, r1, lane, rowptr, col, val, x, y, peers, pl, pf)
    constexpr int per_lane = 7;  // entries per lane, as pick_tpr chooses lanes for Method_Parallel
    if (avg <= per_lane) SB_BODY(1);
    else if (avg <= 2 * per_lane) SB_BODY(2);
    else if (avg <= 4 * per_lane) SB_BODY(4);
    else if (avg <= 8 * per_lane) SB_BODY(8);
    else if (avg <= 16 * per_lane) SB_BODY(16);
    else SB_BODY(32);
#undef SB_BODY
}

// a9: csrSplitter of init_csrSplitter_balanced2 (reference parallel_balanced2_spmv.c:41-53).
__global__ void splitter_kernel(int parts, int nnz, int m, const int *__restrict__ rowptr,
                                int *__restrict__ splitter)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t > parts) return;
    const long long stride = ((long long)nnz + parts - 1) / parts;
    long long b = (long long)t * stride;
    if (b > nnz) b = nnz;
    splitter[t] = right_boundary(rowptr, (int)b, m + 1) - 1;
}

// a10: the Yid scan of parallel_balanced2_get_handle (parallel_balanced2_spmv.c:72-90), reduced to
// the one bit that decides Balanced vs Balanced2: does any partition own no whole row?
__global__ void splitter_starved_kernel(int parts, int m, const int *__restrict__ splitter,
                                        int *__restrict__ flag)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= parts) return;
    if (splitter[t + 1] == splitter[t] && splitter[t] != m) *flag = 1;
}

__global__ void empty_rows_kernel(int m, const int *__restrict__ rowptr, int *__restrict__ flag)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r < m && rowptr[r] == rowptr[r + 1]) *flag = 1;
}

// ------------------------------------------------------------------------------------------------
// Band-major ("virtual row") copy of the matrix, built at handle construction when x does not fit the
// part of L2 that random gathers can use (~half of the 126 MB: measured knee at 64 MiB, see
// scripts/gather_probe.cu).  Columns are cut into K bands of band_cols; the entries of row r that fall
// into band b become virtual row b*m + r of a CSR with K*m rows, stored band after band.  Any CSR
// kernel then runs unchanged on the virtual matrix in ONE launch: CTAs are dispatched in row order, so
// at any moment all resident CTAs work inside one band and gather from an L2-resident slice of x.
// band_reduce_kernel adds the K partial vectors in band order (deterministic).
// ------------------------------------------------------------------------------------------------
constexpr int kMaxBands = 64;

// Locality probe for the automatic band decision: how many entries lie further than `halfwidth` columns
// from their row's position on the (scaled) diagonal?  Stencil / banded / FEM matrices answer "almost
// none" -- the rows in flight at any moment already share a small window of x and banding would only
// manufacture empty virtual rows; uniform-random or graph matrices answer "almost all".
__global__ void band_locality_kernel(int m, double cols_per_row, int halfwidth, const int *__restrict__ rowptr,
                                     const int *__restrict__ col, unsigned long long *__restrict__ far_count)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long far = 0;
    if (r < m) {
        const long long diag = (long long)((double)r * cols_per_row);
        for (int j = rowptr[r]; j < rowptr[r + 1]; ++j) {
            const long long d = (long long)col[j] - diag;
            far += (d > halfwidth || d < -halfwidth);
        }
    }
    for (int o = 16; o > 0; o >>= 1) far += __shfl_xor_sync(kFull, far, o);
    if ((threadIdx.x & 31) == 0 && far) atomicAdd(far_count, far);  // integer counter, builder only
}

// non-zeros that sit in rows longer than `cut` (automatic method selection: the power-law test)
__global__ void heavy_rows_kernel(int m, int cut, const int *__restrict__ rowptr, unsigned long long *__restrict__ heavy)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    unsigned long long v = 0;
    if (r < m) {
        const int len = rowptr[r + 1] - rowptr[r];
        if (len > cut) v = (unsigned long long)len;
    }
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    if ((threadIdx.x & 31) == 0 && v) atomicAdd(heavy, v);  // integer counter, builder only
}

__global__ void band_count_kernel(int m, int bands, int band_cols, const int *__restrict__ rowptr,
                                  const int *__restrict__ col, int *__restrict__ counts)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= m) return;
    int cnt[kMaxBands];
    for (int b = 0; b < bands; ++b) cnt[b] = 0;
    for (int j = rowptr[r]; j < rowptr[r + 1]; ++j) {
        int b = col[j] / band_cols;
        b = b < 0 ? 0 : (b >= bands ? bands - 1 : b);
        ++cnt[b];
    }
    for (int b = 0; b < bands; ++b) counts[(size_t)b * m + r] = cnt[b];
}

template <typename T>
__global__ void band_scatter_kernel(int m, int bands, int band_cols, const int *__restrict__ rowptr,
                                    const int *__restrict__ col, const T *__restrict__ val,
                                    const int *__restrict__ vrowptr, int *__restrict__ vcol,
                                    T *__restrict__ vval)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= m) return;
    int pos[kMaxBands];
    for (int b = 0; b < bands; ++b) pos[b] = vrowptr[(size_t)b * m + r];
    for (int j = rowptr[r]; j < rowptr[r + 1]; ++j) {  // stable: order inside a row is kept
        const int c = col[j];
        int b = c / band_cols;
        b = b < 0 ? 0 : (b >= bands ? bands - 1 : b);
        const int d = pos[b]++;
        vcol[d] = c;
        vval[d] = val[j];
    }
}

template <typename T, typename Store>
__device__ __forceinline__ void band_reduce_body(int row0, int row1, int m, int bands, const T *__restrict__ yv,
                                                 const Store &store)
{
    const int r = row0 + blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= row1) return;
    const auto early = store.early(true, r);
    T s = ldg_stream(yv + r);
    for (int b = 1; b < bands; ++b) s += ldg_stream(yv + (size_t)b * m + r);
    store.put(r, s, early);
}

template <typename T, bool PEERS>
__global__ void band_reduce_kernel(int row0, int row1, int m, int bands, const T *__restrict__ yv, T *__restrict__ y,
                                   const PeerList<T> peers)
{
    band_reduce_body<T>(row0, row1, m, bands, yv, PeerStore<PEERS, T>{y, peers});
}

// spmv_b200_spmv_axpby on a band-major handle: the fold of the band partials, scaled
template <typename T>
__global__ void band_reduce_axpby_kernel(int row0, int row1, int m, int bands, const T *__restrict__ yv,
                                         const ScaledStore<T> store)
{
    band_reduce_body<T>(row0, row1, m, bands, yv, store);
}

// spmv_b200_spmv_axpby_dot on a band-major handle: the scaled fold, and the CTA's partial of w . y
template <typename T>
__global__ void __launch_bounds__(kThreads)
band_reduce_axpby_dot_kernel(int row0, int row1, int m, int bands, const T *__restrict__ yv, const DotArgs<T> d)
{
    double acc = 0;
    band_reduce_body<T>(row0, row1, m, bands, yv, DotStore<T>{d, acc});
    dot_partial(acc, d.partials);
}

// spmv_b200_spmv_shifted on a band-major handle: the shifted fold (x read at the folded row), and the CTA's partials
template <typename T>
__global__ void __launch_bounds__(kThreads)
band_reduce_shift_kernel(int row0, int row1, int m, int bands, const T *__restrict__ yv, const ShiftArgs<T> d)
{
    double xy = 0, yy = 0;
    band_reduce_body<T>(row0, row1, m, bands, yv, ShiftStore<T>{d, xy, yy});
    shift_partials(xy, yy, d.xy, d.yy);
}

// Largest column index used by each of `chunks` equal row chunks (+1): the prefix of x a chunk needs.  Lets the
// host-pointer path start a chunk as soon as that prefix has arrived over PCIe.
__global__ void chunk_xmax_kernel(int m, int chunks, const int *__restrict__ rowptr, const int *__restrict__ col,
                                  int *__restrict__ xmax)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    int mx = 0;
    int c = 0;
    if (r < m) {
        c = (int)((long long)r * chunks / m);
        for (int j = rowptr[r]; j < rowptr[r + 1]; ++j) mx = max(mx, col[j] + 1);
    }
    // rows of one warp almost always share a chunk: reduce first, one integer atomic per warp (builder only)
    const int c0 = __shfl_sync(kFull, c, 0);
    if (__all_sync(kFull, c == c0 || r >= m)) {
        for (int o = 16; o > 0; o >>= 1) mx = max(mx, __shfl_xor_sync(kFull, mx, o));
        if ((threadIdx.x & 31) == 0 && mx > 0) atomicMax(xmax + c0, mx);
    } else if (r < m && mx > 0) {
        atomicMax(xmax + c, mx);
    }
}

// y -> peers for the kernel families whose epilogue is not fused (stream-ordered after them)
template <typename T>
__global__ void peer_copy_kernel(long long m, const T *__restrict__ y, const PeerList<T> peers)
{
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= m) return;
    const T v = y[r];
#pragma unroll
    for (int i = 0; i < kMaxPeers; ++i)
        if (i < peers.n) stg_y(peers.p[i] + r, v);
}

// spmv_b200_spmv_axpby on the handles whose last store is not a scaled kernel's: s = A x as spmv() writes it (into a
// scratch array of the handle), y <- alpha s + beta y.  s = NULL is alpha == 0: y = fl(beta y_old).
template <typename T>
__global__ void axpby_kernel(long long m, const T *__restrict__ s, const ScaledStore<T> store)
{
    const long long r = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= m) return;
    const T y_old = store.early(true, r);
    if (s) store.put(r, ldg_stream(s + r), y_old);
    else stg_y(store.y + r, mul_rn(store.beta, y_old));
}

// spmv_b200_spmv_axpby_dot's scratch pass: axpby_kernel's values (s = NULL with beta == 0: +0, the old y not read), and
// the CTA's partial of w . y
template <typename T>
__global__ void __launch_bounds__(kThreads) axpby_dot_kernel(long long m, const T *__restrict__ s, const DotArgs<T> d)
{
    const long long r = (long long)blockIdx.x * kThreads + threadIdx.x;
    double acc = 0;
    if (r < m) {
        const DotStore<T> store{d, acc};
        const DotEarly<T> e = store.early(true, r);
        if (s) store.put(r, ldg_stream(s + r), e);
        else store.keep(r, d.sc.beta != (T)0 ? mul_rn(d.sc.beta, e.y_old) : (T)0, e);
    }
    dot_partial(acc, d.partials);
}

// spmv_b200_spmv_shifted's scratch pass over s = A x (s = NULL: alpha == 0, y = fl(beta y_old), or +0 with beta == 0
// and the old y not read), and the CTA's partials
template <typename T>
__global__ void __launch_bounds__(kThreads) shift_kernel(long long m, const T *__restrict__ s, const ShiftArgs<T> d)
{
    const long long r = (long long)blockIdx.x * kThreads + threadIdx.x;
    double xy = 0, yy = 0;
    if (r < m) {
        const ShiftStore<T> store{d, xy, yy};
        const T y_old = store.early(true, r);
        if (s) store.put(r, ldg_stream(s + r), y_old);
        else store.keep(r, d.sc.beta != (T)0 ? mul_rn(d.sc.beta, y_old) : (T)0, ldg_stream(d.x + r));
    }
    shift_partials(xy, yy, d.xy, d.yy);
}

// step 4 of the dot's order (DotStore): *dot = the sum of partials[0 .. parts)
constexpr int kDotFinishThreads = 1024;
__global__ void __launch_bounds__(kDotFinishThreads) dot_finish_kernel(int parts, const double *__restrict__ partials,
                                                                       double *__restrict__ dot)
{
    __shared__ double sum[kDotFinishThreads];
    const int t = threadIdx.x;
    double acc = 0;
    for (int i = t; i < parts; i += kDotFinishThreads) acc += partials[i];
    sum[t] = acc;
    __syncthreads();
#pragma unroll
    for (int h = kDotFinishThreads / 2; h > 0; h >>= 1) {
        if (t < h) sum[t] += sum[t + h];
        __syncthreads();
    }
    if (t == 0) *dot = sum[0];
}

}  // namespace sb
