// sell.cuh -- Method_SellCSigma on the GPU: SELL-32-sigma.
//
// Replaces sell_C_Sigma_get_handle_Selected / spmv_Sigma_Blocks_init / cmp (reference
// src/src_spmv/sell_C_Sigma_spmv.c:61-247) and basic_{d,s}_lineProductGather_avx2 +
// spmv_sell_C_Sigma_cpp_{d,s} (inner_spmv.h:411-477, sell_C_Sigma_spmv.c:249-352).
//
// Same structure as the reference, re-sized for a warp: rows [0, banner), banner = sigma*floor(m/sigma),
// are sorted inside each sigma-window by (row length ascending, row index ascending) -- exactly the
// reference's cmp(), so the permutation is bit-identical to Sigma_Block.RowIndex for the same sigma --
// and cut into slices of C = 32 consecutive sorted rows (the reference: C = 4 = one AVX2 register of
// doubles).  A slice is stored column-major, width = longest row of the slice, padded with
// ColIdx = -1 / Val = 0 (the reference's padding, sell_C_Sigma_spmv.c:100-101,121-124); `full` = the
// shortest row of the slice = number of columns that need no padding test (the reference's `full`).
// One warp owns one slice, lane = row: every load is a fully coalesced 128/256-byte line.  Rows
// [banner, m) stay in CSR and go through the CSR-vector kernel (reference :291-297).
#pragma once
#include "common.cuh"

namespace sb {

constexpr int kSellC = 32;
constexpr int kSellMaxSigma = 4096;

// sort one sigma-window: 64-bit keys (len << 32 | row-in-window), bitonic network in shared memory
__global__ void __launch_bounds__(kThreads)
sell_sort_kernel(int sigma, int pow2, const int *__restrict__ rowptr, int *__restrict__ perm)
{
    extern __shared__ unsigned long long s_key[];
    const int w = blockIdx.x;
    const long long row_base = (long long)w * sigma;
    for (int i = threadIdx.x; i < pow2; i += kThreads) {
        unsigned long long k = ~0ull;  // padding sorts to the end
        if (i < sigma) {
            const int r = (int)(row_base + i);
            const unsigned len = (unsigned)(rowptr[r + 1] - rowptr[r]);
            k = ((unsigned long long)len << 32) | (unsigned)i;
        }
        s_key[i] = k;
    }
    __syncthreads();
    for (int size = 2; size <= pow2; size <<= 1) {
        for (int stride = size >> 1; stride > 0; stride >>= 1) {
            for (int i = threadIdx.x; i < (pow2 >> 1); i += kThreads) {
                const int lo = 2 * i - (i & (stride - 1));  // index with bit `stride` cleared
                const int hi = lo + stride;
                const bool up = ((lo & size) == 0);
                const unsigned long long a = s_key[lo], b = s_key[hi];
                if ((a > b) == up) { s_key[lo] = b; s_key[hi] = a; }
            }
            __syncthreads();
        }
    }
    for (int i = threadIdx.x; i < sigma; i += kThreads)
        perm[row_base + i] = (int)(row_base + (unsigned)(s_key[i] & 0xffffffffu));
}

// per slice: width, full (min row length), padded element count.  width = the longest row of the slice, as in
// the reference (ld, sell_C_Sigma_spmv.c:84-92) -- unless `cap` is set and the slice would be mostly padding
// (32*max > 2*sum of lengths: a hub row among short ones).  Then the width is the row length l_i that
// minimises  32*l_i + 2*overflow(l_i) + 64*rows_over(l_i)  and the entries beyond it (`overflow`) are left
// to the long-row path (long_rows.cuh).  The rows of a slice arrive sorted by length, so lane i holds l_i.
// In any case a slice is at most `cap` columns wide: one warp walks a slice column by column, and a slice of
// 10^5 columns would run for milliseconds after the rest of the grid has finished.
__global__ void sell_width_kernel(int slices, int cap, const int *__restrict__ rowptr, const int *__restrict__ perm,
                                  int *__restrict__ width, int *__restrict__ full,
                                  long long *__restrict__ count, int *__restrict__ covered)
{
    const int s = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (s >= slices) return;
    const int r = perm[(long long)s * kSellC + lane];
    const int len = rowptr[r + 1] - rowptr[r];
    int mx = len, mn = len;
    long long total = len;
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
        mx = max(mx, __shfl_xor_sync(kFull, mx, o));
        mn = min(mn, __shfl_xor_sync(kFull, mn, o));
        total += __shfl_xor_sync(kFull, total, o);
    }
    int w = mx;
    if (cap > 0 && (long long)kSellC * mx > 2 * total) {
        // suffix sum of the lengths after lane i (lengths ascend with the lane)
        long long incl = len;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const long long v = __shfl_up_sync(kFull, incl, o);
            if (lane >= o) incl += v;
        }
        const long long after = total - incl;  // sum of l_j, j > lane
        const long long over = after - (long long)(31 - lane) * len;
        int rows_over = 0;  // rows strictly longer than this lane's
        for (int j = 0; j < 32; ++j) rows_over += __shfl_sync(kFull, len, j) > len;
        long long cost = (long long)kSellC * len + 2 * over + 64LL * rows_over;
        int best = len;
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {  // min cost, ties -> the larger width
            const long long c2 = __shfl_xor_sync(kFull, cost, o);
            const int b2 = __shfl_xor_sync(kFull, best, o);
            if (c2 < cost || (c2 == cost && b2 > best)) { cost = c2; best = b2; }
        }
        w = best;
    }
    if (cap > 0 && w > cap) w = cap;
    if (covered) covered[r] = min(len, w);
    if (lane == 0) {
        width[s] = w;
        full[s] = min(mn, w);
        count[s] = (long long)w * kSellC;
    }
}

// scatter CSR rows into the column-major padded slices
template <typename T>
__global__ void sell_fill_kernel(int slices, const int *__restrict__ rowptr, const int *__restrict__ col,
                                 const T *__restrict__ val, const int *__restrict__ perm,
                                 const long long *__restrict__ slice_ptr, int *__restrict__ scol,
                                 T *__restrict__ sval)
{
    const int s = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (s >= slices) return;
    const long long base = slice_ptr[s];
    const int w = (int)((slice_ptr[s + 1] - base) / kSellC);
    const int r = perm[(long long)s * kSellC + lane];
    const int start = rowptr[r], len = rowptr[r + 1] - start;
    for (int j = 0; j < w; ++j) {
        const long long dst = base + (long long)j * kSellC + lane;
        if (j < len) {
            scol[dst] = col[start + j];
            sval[dst] = val[start + j];
        } else {
            scol[dst] = -1;
            sval[dst] = 0;
        }
    }
}

// U = columns per step (all 2U coalesced loads of a step are issued before its U gathers), MINB = CTAs per SM
// the register allocation is held to.  Two flavours are instantiated: U = 8 / 6 CTAs (gather-bound matrices:
// C2 0.43 vs 0.39) and U = 4 / 8 CTAs, every warp slot of the SM filled (HBM-bound ones: C4 0.86 -> 0.98).
// (Software-pipelined variants -- the next step's stream loads issued before this step's gathers -- measured no
// better and were dropped.)
template <typename T, int U, typename Store>
__device__ __forceinline__ void sell_body(unsigned tid, int slices, const long long *__restrict__ slice_ptr,
                                          const int *__restrict__ full, const int *__restrict__ perm,
                                          const int *__restrict__ scol, const T *__restrict__ sval,
                                          const T *__restrict__ x, const Store &store)
{
    const uint64_t pl = policy_evict_last(), pf = policy_evict_first();
    const int s = (int)(((long long)blockIdx.x * kThreads + tid) >> 5);
    const int lane = tid & 31;
    if (s >= slices) return;
    const long long base = slice_ptr[s];
    const int w = (int)((slice_ptr[s + 1] - base) >> 5);
    const int f = full[s];
    const int out_row = perm[(long long)s * kSellC + lane];
    const auto early = store.early(true, out_row);
    const int *c = scol + base + lane;
    const T *v = sval + base + lane;
    // blocked summation (U columns -> 512 columns -> row) keeps the rounding error of a long row at
    // ~sqrt(len/512) instead of ~sqrt(len) ulps; fixed order, so still bitwise reproducible
    constexpr int kGroups = 512 / U;
    T sum = 0, mid = 0;
    int groups = 0;
    int j = 0;
    // columns every row of the slice owns: no padding test (the reference's `full` loop)
    for (; j + U <= f; j += U) {
        int cc[U];
        T vv[U];
#pragma unroll
        for (int k = 0; k < U; ++k) cc[k] = ldg_stream(c + (size_t)(j + k) * kSellC, pf);
#pragma unroll
        for (int k = 0; k < U; ++k) vv[k] = ldg_stream(v + (size_t)(j + k) * kSellC, pf);
        T part = 0;
#pragma unroll
        for (int k = 0; k < U; ++k) part = fma_t(vv[k], ldg_x(x + cc[k], pl), part);
        mid += part;
        if (++groups == kGroups) { sum += mid; mid = 0; groups = 0; }
    }
    // remaining columns, padding (ColIdx == -1) masked as in the reference's `~idx ? ... : 0`
    for (; j < w; j += 4) {
        int cc[4];
        T vv[4];
#pragma unroll
        for (int k = 0; k < 4; ++k) {
            const bool in = j + k < w;
            cc[k] = in ? ldg_stream(c + (size_t)(j + k) * kSellC, pf) : -1;
            vv[k] = in ? ldg_stream(v + (size_t)(j + k) * kSellC, pf) : (T)0;
        }
        T part = 0;
#pragma unroll
        for (int k = 0; k < 4; ++k)
            if (cc[k] >= 0) part = fma_t(vv[k], ldg_x(x + cc[k], pl), part);
        mid += part;
        if (++groups >= kGroups) { sum += mid; mid = 0; groups = 0; }
    }
    sum += mid;
    store.put(out_row, sum, early);
}

template <typename T, bool PEERS, int U, int MINB>
__global__ void __launch_bounds__(kThreads, MINB)
sell_kernel(int slices, const long long *__restrict__ slice_ptr, const int *__restrict__ full,
            const int *__restrict__ perm, const int *__restrict__ scol, const T *__restrict__ sval,
            const T *__restrict__ x, T *__restrict__ y, const PeerList<T> peers)
{
    sell_body<T, U>(threadIdx.x, slices, slice_ptr, full, perm, scol, sval, x, PeerStore<PEERS, T>{y, peers});
}

// spmv_b200_spmv_axpby on an unbanded SELL handle without long-row list (the CSR tail: csr_tail_axpby_kernel)
template <typename T, int U, int MINB>
__global__ void __launch_bounds__(kThreads, MINB)
sell_axpby_kernel(int slices, const long long *__restrict__ slice_ptr, const int *__restrict__ full,
                  const int *__restrict__ perm, const int *__restrict__ scol, const T *__restrict__ sval,
                  const T *__restrict__ x, const ScaledStore<T> store)
{
    sell_body<T, U>(threadIdx.x, slices, slice_ptr, full, perm, scol, sval, x, store);
}

// spmv_b200_spmv_axpby_dot on the same handles (the CSR tail: csr_tail_axpby_dot_kernel)
template <typename T, int U, int MINB>
__global__ void __launch_bounds__(kThreads, MINB)
sell_axpby_dot_kernel(int slices, const long long *__restrict__ slice_ptr, const int *__restrict__ full,
                      const int *__restrict__ perm, const int *__restrict__ scol, const T *__restrict__ sval,
                      const T *__restrict__ x, const DotArgs<T> d)
{
    double acc = 0;
    sell_body<T, U>(threadIdx.x, slices, slice_ptr, full, perm, scol, sval, x, DotStore<T>{d, acc});
    dot_partial(acc, d.partials);
}

// spmv_b200_spmv_shifted on the same handles (the CSR tail: csr_tail_shift_kernel)
template <typename T, int U, int MINB>
__global__ void __launch_bounds__(kThreads, MINB)
sell_shift_kernel(int slices, const long long *__restrict__ slice_ptr, const int *__restrict__ full,
                  const int *__restrict__ perm, const int *__restrict__ scol, const T *__restrict__ sval,
                  const T *__restrict__ x, const ShiftArgs<T> d)
{
    double xy = 0, yy = 0;
    sell_body<T, U>(threadIdx.x, slices, slice_ptr, full, perm, scol, sval, x, ShiftStore<T>{d, xy, yy});
    shift_partials(xy, yy, d.xy, d.yy);
}

}  // namespace sb
