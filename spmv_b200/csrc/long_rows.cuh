// long_rows.cuh -- rows (or row tails) that are too long for the lane group / SELL slice that owns them.
//
// The reference has no counterpart: its Method_Parallel simply lets one OpenMP thread walk a hub row
// (src/src_spmv/parallel_spmv.c:12-16) and its SELL pads every row of a chunk to the longest one
// (sell_C_Sigma_spmv.c:84-101), which is harmless at C = 4 but not at C = 32 on a power-law matrix.  Here
// the main kernel of a method covers the first covered[r] entries of row r (all of them for ordinary rows)
// and the remainder is cut into segments of kLongSeg entries: one warp reduces one segment
// (long_seg_kernel), one warp per row adds the segment sums in segment order (long_final_kernel).  No
// atomics, fixed order: bitwise reproducible.
#pragma once
#include "common.cuh"

namespace sb {

constexpr int kLongSeg = 2048;

// covered[r] for the threshold rule: rows longer than thr are left to the long-row path entirely
__global__ void long_cover_threshold_kernel(int m, int row0, int thr, const int *__restrict__ rowptr,
                                            int *__restrict__ covered)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= m) return;
    const int len = rowptr[r + 1] - rowptr[r];
    if (r >= row0) covered[r] = len > thr ? 0 : len;
}

__global__ void long_count_kernel(int m, const int *__restrict__ rowptr, const int *__restrict__ covered,
                                  int *__restrict__ cnt_rows, int *__restrict__ cnt_segs)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r > m) return;
    int segs = 0;
    if (r < m) {
        const int rest = rowptr[r + 1] - rowptr[r] - covered[r];
        if (rest > 0) segs = (rest + kLongSeg - 1) / kLongSeg;
    }
    cnt_rows[r] = segs > 0;
    cnt_segs[r] = segs;
}

__global__ void long_fill_kernel(int m, const int *__restrict__ rowptr, const int *__restrict__ covered,
                                 const int *__restrict__ scan_rows, const int *__restrict__ scan_segs,
                                 int *__restrict__ row, int *__restrict__ start, int *__restrict__ seg_ptr,
                                 int *__restrict__ seg_row)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r > m) return;
    if (r == m) { seg_ptr[scan_rows[m]] = scan_segs[m]; return; }
    const int rest = rowptr[r + 1] - rowptr[r] - covered[r];
    if (rest <= 0) return;
    const int i = scan_rows[r], s0 = scan_segs[r], segs = (rest + kLongSeg - 1) / kLongSeg;
    row[i] = r;
    start[i] = rowptr[r] + covered[r];
    seg_ptr[i] = s0;
    for (int k = 0; k < segs; ++k) seg_row[s0 + k] = i;
}

// one warp per segment
template <typename T>
__global__ void __launch_bounds__(kThreads)
long_seg_kernel(int n_segs, const int *__restrict__ seg_row, const int *__restrict__ row,
                const int *__restrict__ start, const int *__restrict__ seg_ptr, const int *__restrict__ rowptr,
                const int *__restrict__ col, const T *__restrict__ val, const T *__restrict__ x,
                T *__restrict__ partial, T *__restrict__ y, int finish_single, int accumulate)
{
    // finish_single: a row with ONE segment is finished right here (its sole writer at this point of the stream)
    // and long_final_kernel skips it -- most SELL overflow rows are of that kind
    const uint64_t pl = policy_evict_last(), pf = policy_evict_first();
    const int seg = (int)(((long long)blockIdx.x * kThreads + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (seg >= n_segs) return;
    const int i = seg_row[seg];
    const int b = start[i] + (seg - seg_ptr[i]) * kLongSeg;
    const int row_end = rowptr[row[i] + 1];
    const int e = (row_end - b > kLongSeg) ? b + kLongSeg : row_end;
    // predicated batches of 8 per lane: 16 stream loads, then 8 gathers in flight together (a plain loop costs two
    // dependent round trips per element: measured 420 us -> see DESIGN.md for 35 M hub entries of C3)
    constexpr int B = 8;
    T acc = 0;
    for (int j0 = b + lane; j0 < e; j0 += 32 * B) {
        int c[B];
        T v[B];
#pragma unroll
        for (int k = 0; k < B; ++k) c[k] = (j0 + 32 * k < e) ? ldg_stream(col + j0 + 32 * k, pf) : -1;
#pragma unroll
        for (int k = 0; k < B; ++k) v[k] = (j0 + 32 * k < e) ? ldg_stream(val + j0 + 32 * k, pf) : (T)0;
        T part = 0;
#pragma unroll
        for (int k = 0; k < B; ++k)
            if (c[k] >= 0) part = fma_t(v[k], ldg_x(x + c[k], pl), part);
        acc += part;
    }
    acc = group_sum_c<T, 32>(acc);
    if (lane == 0) {
        if (finish_single && seg_ptr[i + 1] - seg_ptr[i] == 1) {
            const int r = row[i];
            stg_y(y + r, accumulate ? y[r] + acc : acc);
        } else {
            partial[seg] = acc;
        }
    }
}

// one warp per long row: y[row] = (accumulate ? y[row] : 0) + sum of its segment sums, in segment order
template <typename T, bool PEERS>
__global__ void __launch_bounds__(kThreads)
long_final_kernel(int n_rows, int accumulate, int skip_single, const int *__restrict__ row,
                  const int *__restrict__ seg_ptr, const T *__restrict__ partial, T *__restrict__ y,
                  const PeerList<T> peers)
{
    const int i = (int)(((long long)blockIdx.x * kThreads + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (i >= n_rows) return;
    const int s0 = seg_ptr[i], s1 = seg_ptr[i + 1];
    if (skip_single && s1 - s0 == 1) return;  // finished by long_seg_kernel
    T acc = 0;
    for (int s = s0 + lane; s < s1; s += 32) acc += partial[s];
    acc = group_sum_c<T, 32>(acc);
    if (lane == 0) {
        const int r = row[i];
        store_y<PEERS>(y, peers, r, accumulate ? y[r] + acc : acc);
    }
}

}  // namespace sb
