// common.cuh -- device state, error latch, and the sm_100a load/store + warp primitives shared by all
// kernel families of libspmv_b200.
#pragma once
#include <cuda_runtime.h>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>

#define SPMV_B200_NO_HOST_HEADERS 1
#include "../../include/spmv_b200.h"

namespace sb {

// ------------------------------------------------------------------------------------------------
// error latch (the public API returns void, reference include/spmv.h)
// ------------------------------------------------------------------------------------------------
void set_error(const char *fmt, ...);
bool cuda_ok(cudaError_t e, const char *what, const char *file, int line);
#define SB_CUDA(expr) ::sb::cuda_ok((expr), #expr, __FILE__, __LINE__)
#define SB_TRY(expr) do { if (!SB_CUDA(expr)) return false; } while (0)

void count_launch(int n = 1);

constexpr int kThreads = 256;       // CTA size of every spmv-path kernel
constexpr int kWarpsPerCta = kThreads / 32;
constexpr unsigned kFull = 0xffffffffu;
constexpr int kPipeChunks = 8;      // row chunks / x pieces of the pipelined host-pointer path
constexpr int kMaxPieces = 64;      // >= kMaxBands (csr_kernels.cuh)
constexpr int kMaxPeers = 8;        // extra y destinations of the fused SpMV + all-gather

static inline int ceil_div(long long a, long long b) { return (int)((a + b - 1) / b); }

// ------------------------------------------------------------------------------------------------
// Device arrays (host code).  Every device allocation the library makes for its own use is held by a DeviceArray or
// a DeviceBytes: freed when the owner is destroyed, reset or assigned over, so a builder's temporaries are freed on
// every return path and abandoning a layout is one assignment of an empty group.
// ------------------------------------------------------------------------------------------------
void count_allocation(int delta);  // spmv_b200_live_allocations

template <typename U>
class DeviceArray {
  public:
    DeviceArray() = default;
    DeviceArray(DeviceArray &&o) noexcept : p_(o.p_) { o.p_ = nullptr; }
    DeviceArray &operator=(DeviceArray &&o) noexcept
    {
        if (this != &o) {
            reset();
            p_ = o.p_;
            o.p_ = nullptr;
        }
        return *this;
    }
    DeviceArray(const DeviceArray &) = delete;
    DeviceArray &operator=(const DeviceArray &) = delete;
    ~DeviceArray() { reset(); }

    // `count` elements, at least one, in place of what the owner held; a failure latches the error (SB_CUDA)
    bool alloc(size_t count)
    {
        reset();
        void *p = nullptr;
        if (!SB_CUDA(cudaMalloc(&p, (count ? count : 1) * sizeof(U)))) return false;
        p_ = (U *)p;
        count_allocation(1);
        return true;
    }
    void reset()
    {
        if (!p_) return;
        cudaFree(p_);
        count_allocation(-1);
        p_ = nullptr;
    }
    U *get() const { return p_; }
    operator U *() const { return p_; }  // kernels and copies take the raw pointer; the owner keeps the allocation

  private:
    U *p_ = nullptr;
};

// float or double values: the element size is chosen at create (DeviceState::vsize)
class DeviceBytes {
  public:
    bool alloc(size_t count, size_t elem_bytes) { return bytes_.alloc((count ? count : 1) * elem_bytes); }
    void *get() const { return bytes_.get(); }
    template <typename T>
    T *as() const { return (T *)bytes_.get(); }

  private:
    DeviceArray<unsigned char> bytes_;
};

// ------------------------------------------------------------------------------------------------
// The options of one create (include/spmv_b200.h), read once at its start by read_create_options, which applies every
// key's rule: the builders see only these values.  seg_ctas and seg_prefetch are read at launch.
// ------------------------------------------------------------------------------------------------
struct CreateOptions {
    int sell_sigma;         // a multiple of 32 in [32, 4096]
    int sell_variant;       // 0, 2, or -1 = automatic
    int sell_cap;           // [32, 2^20], or 0 = off
    int csr5_sigma;         // 4, 8, 16, or 0 = automatic
    long long block_nnz;    // >= 32
    int tile_items;         // 4 or 8
    int tpr;                // forced lanes per row (1, 2, 4, 8, 16, 32), or 0 = from the mean
    bool row_bins;          // Method_Parallel may bin its rows: "row_bins" on and the raw "tpr" 0
    long long long_thr;     // 0 = automatic, < 0 = off, else forced
    int x_bands;            // 0 = automatic, 1 = off, 2 .. kMaxBands forced
    int seg_bands;          // 0 = automatic, -1 = never, 2 .. kSegMaxBands forced (overrides x_bands)
    bool force_merge, pipeline, auto_pick, reorder, pin_host, refresh;
    bool axpby_fused;       // false: spmv_b200_spmv_axpby takes the scratch pass on every layout
};

// ------------------------------------------------------------------------------------------------
// Device-resident state hanging off spmv_Handle::extraHandle.  The device arrays are grouped by the builder that
// fills them, each group with the sizes that describe its arrays.
// ------------------------------------------------------------------------------------------------
struct DeviceState {
    uint32_t magic = 0x5b200a11u;
    // The handle owns staging buffers, partial-sum arrays and events (the reference's handle is read-only in spmv()
    // for most methods, SURVEY 8b "Threading"): calls on ONE handle from several threads are serialised here, so
    // that their launches reach the stream call after call instead of interleaved
    std::mutex mu;
    int device = 0;
    cudaStream_t stream = nullptr;  // legacy default stream unless spmv_b200_set_stream
    int m = 0, n = 0, nnz = 0;
    int vsize = 8;                  // 8 = fp64, 4 = fp32
    int requested = 0;              // SPMV_METHODS asked for at create
    int auto_method = -1;           // option "auto": the SPMV_METHODS value create picked instead (-1: not used)
    int kernel = SPMV_B200_KERNEL_NONE;
    bool ok = false;                // false => spmv() is a no-op
    bool has_empty_rows = false;
    int dev_sms = 0;
    long long dev_l2 = 0;
    int layout_fallbacks = 0;       // optional layouts (band copy, band segments, row bins) that could not be built
    CreateOptions opts = {};        // the options in force at create
    // option "refresh": every value array below keeps its source map (refresh.cuh) in its own group, so that dropping a
    // layout drops its map too.  Starts as opts.refresh; cleared at create when a map could not be built: the handle
    // then cannot be refreshed
    bool refresh = false;
    bool map_failed = false;
    int n_peers = 0;                // spmv_b200_set_y_peers
    void *peers[kMaxPeers] = {};

    // CSR on the device: the caller's device arrays adopted in place, or our upload (32 bytes of slack behind every
    // array).  rowptr / col / val only point at one of the two.
    int *rowptr = nullptr, *col = nullptr;
    void *val = nullptr;
    struct CsrUpload { DeviceArray<int> rowptr, col; DeviceBytes val; DeviceArray<int> map; } upload;  // map: under "reorder" only
    bool released_csr = false;      // the upload was freed after a re-laid-out copy took over

    // pageable host x / y that keep coming back (the reference's drivers reuse one X and one Y for every call) are
    // page-locked in place after the second sighting, so that the copies run at PCIe speed instead of being
    // staged by the driver.  Opt-in (option "pin_host" / SPMV_B200_PIN_HOST=1): the caller must not free such a
    // buffer while the handle lives.  Undone at clear / destroy or when the caller switches buffers
    struct PinSlot { const void *ptr = nullptr; size_t bytes = 0; int seen = 0; bool registered = false; };
    PinSlot pin[2];
    // staging for host-side x / y; the pipelined host path (CSR-vector kernel) copies x in pieces on s_in,
    // computes row chunks as soon as their prefix of x has arrived, and returns finished chunks of y on s_out
    // val: host values of spmv_b200_set_values, when no upload takes them; s: A x of spmv_b200_spmv_axpby on the handles
    // whose last store has no scaled kernel (its scratch pass), allocated at the first such call; w: a host w of
    // spmv_b200_spmv_axpby_dot
    struct Staging { DeviceBytes x, y, val, s, w; } stage;
    // spmv_b200_spmv_axpby_dot: the CTA partials of its sum (allocated at the first call, sized by dot_partials_bound)
    // and, for a host dot, the device double the sum is copied back from.  spmv_b200_spmv_shifted with dots: partials
    // (x . y), yy (y . y, the same size) and, for host dots, pair (2 doubles); each allocated at its first use
    struct Dot { DeviceArray<double> partials, result, yy, pair; } dot;
    bool pipeline = false;
    cudaStream_t s_in = nullptr, s_out = nullptr;
    cudaEvent_t ev_in[kMaxPieces] = {}, ev_out[kPipeChunks] = {}, ev_start = nullptr, ev_x = nullptr;
    int chunk_xmax[kPipeChunks] = {};

    // Method_Parallel
    int tpr = 0;
    // Active matrix view used by every layout builder and kernel: the CSR itself, or (x_bands > 1) its
    // band-major copy, in which virtual row b*m + r holds the entries of row r whose column lies in band
    // b = col / band_cols.  Kernels then write the virtual y (v.y) and band_reduce_kernel folds it.
    int a_m = 0;
    int *a_rowptr = nullptr, *a_col = nullptr;
    void *a_val = nullptr;
    int x_bands = 1, band_cols = 0;
    double far_fraction = -1.0;     // share of entries far from the diagonal (automatic band decision)
    struct BandCopy { DeviceArray<int> rowptr, col, map; DeviceBytes val, y; } v;
    // Method_Balanced: row blocks; ref_splitter mirrors the reference with the caller's nthreads
    struct Splitters {
        int parts = 0, ref_T = 0;
        DeviceArray<int> splitter;      // [parts+1]
        DeviceArray<int> ref_splitter;  // [ref_T+1]
    } split;
    // tiles of Method_Balanced2 / Method_Balanced_Yid, CSR5 and band segments, and their carries
    struct Tiles {
        int count = 0, items = 0;
        DeviceArray<int> rows;          // nnz-split: row containing the first nnz of each tile [count+1]
        DeviceArray<int2> merge_coords; // merge-path: (row, nnz) start of each tile [count+1]
        DeviceBytes carry_val;          // [count] partial sum that belongs to a row started earlier
        DeviceArray<int> carry_row;     // [count] that row, or -1
        DeviceBytes carry2_val;         // level-2 carry list of the two-level fix-up: 2 entries per group of 64 tiles
        DeviceArray<int> carry2_row;
    } tile;
    // Method_SellCSigma
    struct Sell {
        int sigma = 0, banner = 0, slices = 0, variant = 0;
        long long padded = 0;
        DeviceArray<int> perm, width, full, col, map;
        DeviceArray<long long> slice_ptr;
        DeviceBytes val;
    } sell;
    // long rows / row tails left over by the main kernel of Method_Parallel and Method_SellCSigma (long_rows.cuh)
    struct LongRows {
        int thr = 0x7fffffff;           // CSR-vector kernels skip rows longer than this
        int rows = 0, segs = 0;
        bool accumulate = false;        // true: the main kernel already wrote the head of the row (SELL)
        DeviceArray<int> row, start, seg_ptr, seg_row;
        DeviceBytes partial;
        // Method_Parallel on short-row matrices with hubs: rows binned by length class (<= 8, <= 32, <= 128), one
        // launch per bin with 1 / 4 / 16 lanes per row; longer rows are on the long-row list
        bool binned = false;
        DeviceArray<int> bin_list;      // row ids, bin after bin, ascending inside a bin
        int bin_ptr[4] = {};
    } lr;
    // Method_CSR5SPMV (omega = 32)
    struct Csr5 {
        int sigma = 0, p = 0, bit_y = 0, bit_ss = 0, num_offsets = 0, tail_start = 0;
        DeviceArray<uint32_t> tile_ptr, tile_desc;
        DeviceArray<int> off_ptr, off, col, map;
        DeviceBytes val;
    } c5;
    // hyper-sparse column bands as band segments (band_seg.cuh): x_bands = K but the active view stays the CSR
    struct BandSegments {
        int bands = 0;                  // K, or 0 = no band segments (option and info key "seg_bands")
        int ptr[kMaxPieces + 1] = {};   // first slot of every band in col / ent_val (aligned to 4), [K] = end
        int cnt[kMaxPieces] = {};       // entries of every band
        int tile0[kMaxPieces + 1] = {}; // first tile of every band
        long long total = 0;            // segments = (band, row) pairs with at least one entry
        int groups = 0;                 // 32-row groups of the merge pass
        int ctas = 0;                   // persistent CTAs per SM of pass 1
        int grid = 0;                   // persistent CTAs of pass 1 (device-wide occupancy, set at the first launch)
        bool cross = false;             // some segment crosses a tile boundary: the carry fix-up is needed
        bool mask64 = false;            // K > 32: 64-bit row masks
        DeviceArray<int> col;           // column index | segment-end bit 31
        DeviceBytes ent_val;            // values, band-major
        DeviceArray<int> map;           // source map of ent_val [ptr[K]]
        DeviceBytes mask;               // per row: bands in which it has a segment
        DeviceArray<int4> tile_ent;     // per tile: (first slot, entries, L2-prefetch duty: first x element, elements)
        DeviceArray<int> tile_seg0;     // per 256-entry chunk of a tile (8 per tile): index of its first segment sum
        DeviceArray<int> gbase;         // [groups][K]: position of a row group's first segment sum in band b's list
        DeviceArray<int> ticket;        // ticket counter of pass 1's dynamic tile schedule
        DeviceBytes sums;               // [total] segment sums, band-major (written by pass 1, read by pass 2)
    } seg;
};

// ------------------------------------------------------------------------------------------------
// sm_100a memory primitives.
//  * matrix streams (ColIdx / Val) are read exactly once per SpMV: non-coherent path, L2 evict-first (the tile
//    kernels also keep them out of L1; band_seg.cuh stages them with bulk copies instead);
//  * x is the only re-used operand: read-only path with an L2 evict-last policy so the streams do
//    not push it out of the 126 MB L2.
// ------------------------------------------------------------------------------------------------
#ifdef __CUDACC__
__device__ __forceinline__ uint64_t policy_evict_last()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(p));
    return p;
}
__device__ __forceinline__ uint64_t policy_evict_first()
{
    uint64_t p;
    asm volatile("createpolicy.fractional.L2::evict_first.b64 %0, 1.0;" : "=l"(p));
    return p;
}

// ---- gathers from x (evict-last) ----
__device__ __forceinline__ double ldg_x(const double *p, uint64_t pol)
{
    double r;
    asm volatile("ld.global.nc.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ float ldg_x(const float *p, uint64_t pol)
{
    float r;
    asm volatile("ld.global.nc.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(r) : "l"(p), "l"(pol));
    return r;
}

// ---- scalar streaming loads ----
__device__ __forceinline__ int ldg_stream(const int *p)
{
    int r;
    asm volatile("ld.global.nc.L1::no_allocate.s32 %0, [%1];" : "=r"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ float ldg_stream(const float *p)
{
    float r;
    asm volatile("ld.global.nc.L1::no_allocate.f32 %0, [%1];" : "=f"(r) : "l"(p));
    return r;
}
__device__ __forceinline__ double ldg_stream(const double *p)
{
    double r;
    asm volatile("ld.global.nc.L1::no_allocate.f64 %0, [%1];" : "=d"(r) : "l"(p));
    return r;
}

// ---- scalar streaming loads with an explicit L2 policy (evict-first for the matrix streams) ----
__device__ __forceinline__ int ldg_stream(const int *p, uint64_t pol)
{
    int r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ float ldg_stream(const float *p, uint64_t pol)
{
    float r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ double ldg_stream(const double *p, uint64_t pol)
{
    double r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(r) : "l"(p), "l"(pol));
    return r;
}

// ---- scalar matrix-stream loads that DO allocate in L1 (L2 evict-first) ----
__device__ __forceinline__ int ldg_cached(const int *p, uint64_t pol)
{
    int r;
    asm volatile("ld.global.nc.L2::cache_hint.s32 %0, [%1], %2;" : "=r"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ float ldg_cached(const float *p, uint64_t pol)
{
    float r;
    asm volatile("ld.global.nc.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(r) : "l"(p), "l"(pol));
    return r;
}
__device__ __forceinline__ double ldg_cached(const double *p, uint64_t pol)
{
    double r;
    asm volatile("ld.global.nc.L2::cache_hint.f64 %0, [%1], %2;" : "=d"(r) : "l"(p), "l"(pol));
    return r;
}

// ---- y stores: written once, never re-read by the kernel ----
__device__ __forceinline__ void stg_y(double *p, double v)
{
    asm volatile("st.global.L1::no_allocate.f64 [%0], %1;" ::"l"(p), "d"(v) : "memory");
}
__device__ __forceinline__ void stg_y(float *p, float v)
{
    asm volatile("st.global.L1::no_allocate.f32 [%0], %1;" ::"l"(p), "f"(v) : "memory");
}

// ---- fused SpMV + all-gather: extra destinations of y (peer GPUs' next-x, mapped through CUDA IPC) ----
template <typename T>
struct PeerList {
    int n;
    T *p[kMaxPeers];
};
template <bool PEERS, typename T>
__device__ __forceinline__ void store_y(T *y, const PeerList<T> &peers, long long row, T v)
{
    stg_y(y + row, v);
    if (PEERS) {  // NVLink peer stores, overlapped with the SpMV (separate instantiation: the plain kernels pay nothing)
        // constant indices only: a dynamically indexed kernel-parameter array would be copied to local
        // memory by every thread (measured: +20-35 % on the L1TEX-bound kernels)
#pragma unroll
        for (int i = 0; i < kMaxPeers; ++i)
            if (i < peers.n) stg_y(peers.p[i] + row, v);
    }
}

// ---- the final store of a row value v = (A x)[row]: a template parameter of every kernel body that writes final y
// values.  PeerStore is spmv()'s (y = v, and the peer copies); ScaledStore is spmv_b200_spmv_axpby's (y <- alpha v +
// beta y).  early(pred, row) reads what put needs; most bodies call it before the row walk, so that a load of the old y
// is in flight while the row is summed.  put(row, v, early) writes.  The kernels read threadIdx.x themselves and hand it to the body (`tid`): only a
// read in the __global__ function carries the range __launch_bounds__ gives it, so the spmv() kernels keep their code.
struct NoEarly {};
template <bool PEERS, typename T>
struct PeerStore {
    T *y;
    const PeerList<T> &peers;
    __device__ __forceinline__ NoEarly early(bool, long long) const { return {}; }
    __device__ __forceinline__ void put(long long row, T v, NoEarly) const { store_y<PEERS>(y, peers, row, v); }
};

// round-to-nearest products and sums that nvcc never contracts into an FMA
__device__ __forceinline__ double mul_rn(double a, double b) { return __dmul_rn(a, b); }
__device__ __forceinline__ float mul_rn(float a, float b) { return __fmul_rn(a, b); }
__device__ __forceinline__ double add_rn(double a, double b) { return __dadd_rn(a, b); }
__device__ __forceinline__ float add_rn(float a, float b) { return __fadd_rn(a, b); }
__device__ __forceinline__ double sub_rn(double a, double b) { return __dsub_rn(a, b); }
__device__ __forceinline__ float sub_rn(float a, float b) { return __fsub_rn(a, b); }

// y[row] = fl(fl(alpha v) + fl(beta y_old)), three roundings and no FMA (what numpy computes from spmv()'s bits); beta ==
// 0: fl(alpha v), and the old y is never read, so whatever it holds does not propagate.  (alpha == 0 never reaches a
// kernel that computes v: the host then writes fl(beta y_old), or +0, without reading A or x.)
template <typename T>
struct ScaledStore {
    T *y;
    T alpha, beta;
    __device__ __forceinline__ T early(bool pred, long long row) const { return pred && beta != (T)0 ? __ldcs(y + row) : (T)0; }
    __device__ __forceinline__ T value(T v, T y_old) const
    {
        const T av = mul_rn(alpha, v);
        return beta != (T)0 ? add_rn(av, mul_rn(beta, y_old)) : av;
    }
    __device__ __forceinline__ void put(long long row, T v, T y_old) const { stg_y(y + row, value(v, y_old)); }
};

// ---- spmv_b200_spmv_axpby_dot: y <- alpha A x + beta y as ScaledStore writes it, and dot = sum_i fl(w_i y_i) over
// the rows written, in double for both precisions (an fp32 product taken in double is exact).  w == NULL is w = y.
// The sum has one fixed order, so identical inputs give identical bits:
//   1. each thread adds the products of the rows it stores to its own double (one row per thread in every body);
//   2. an xor butterfly over the warp (5 levels);
//   3. the 8 warp sums of the CTA in a fixed tree of 3 levels (dot_partial), one partial per CTA, written to
//      partials[the CTAs of earlier dot launches of the call + blockIdx.x];
//   4. dot_finish_kernel, one CTA of 1024 threads: thread t adds partials t, t + 1024, ... in that order, then a fixed
//      halving tree of 10 levels.
// So no product passes through more than L = 18 + ceil(P / 1024) additions, P the number of partials (at most m + 2),
// and |dot - sum_i p_i| <= L 2^-53 sum_i |p_i|.
template <typename T>
struct DotArgs {
    ScaledStore<T> sc;
    const T *w;         // NULL: w is the new y
    double *partials;   // this launch's first partial
};

template <typename T>
struct DotEarly {
    T y_old, w;
};

template <typename T>
struct DotStore {
    const DotArgs<T> &d;
    double &acc;
    __device__ __forceinline__ DotEarly<T> early(bool pred, long long row) const
    {
        return {d.sc.early(pred, row), pred && d.w ? ldg_stream(d.w + row) : (T)0};
    }
    __device__ __forceinline__ void put(long long row, T v, DotEarly<T> e) const { keep(row, d.sc.value(v, e.y_old), e); }
    // store the final y of the row and add its product
    __device__ __forceinline__ void keep(long long row, T y, DotEarly<T> e) const
    {
        stg_y(d.sc.y + row, y);
        acc += __dmul_rn((double)(d.w ? e.w : y), (double)y);
    }
};

// ---- spmv_b200_spmv_shifted (square handles): y <- alpha (A - sigma I) x + beta y, the step of a Chebyshev or KPM
// recurrence, with y[row] = fl(fl(alpha fl(v - fl(sigma x[row]))) + fl(beta y_old)); sigma == 0 skips the shift, so the
// value is ScaledStore's, bit for bit (v - fl(0 x) would turn a -0 into +0).  With partials, also x . y and y . y over
// the rows written, each as DotStore takes w . y (w = x and w = y): the same products, the same per-thread sums and the
// same fixed tree (shift_partials), so that with sigma == 0 both equal spmv_b200_spmv_axpby_dot's bit for bit.
template <typename T>
struct ShiftArgs {
    ScaledStore<T> sc;
    T sigma;
    const T *x;         // the x of the product, read again at the stored row
    double *xy, *yy;    // this launch's first partial of x . y and of y . y; NULL: no dots
};

template <typename T>
struct ShiftStore {
    const ShiftArgs<T> &d;
    double &xy, &yy;
    __device__ __forceinline__ T early(bool pred, long long row) const { return d.sc.early(pred, row); }
    // x[row] is a coalesced streaming read (the row walk gathers x through the evict-last path), issued here rather
    // than in early(): held through the row walk it takes two more registers, and the fp64 SELL twin spills at its 40
    __device__ __forceinline__ void put(long long row, T v, T y_old) const
    {
        const T xr = ldg_stream(d.x + row);
        keep(row, d.sc.value(d.sigma != (T)0 ? sub_rn(v, mul_rn(d.sigma, xr)) : v, y_old), xr);
    }
    // store the final y of the row and add its two products
    __device__ __forceinline__ void keep(long long row, T y, T xr) const
    {
        stg_y(d.sc.y + row, y);
        xy += __dmul_rn((double)xr, (double)y);
        yy += __dmul_rn((double)y, (double)y);
    }
};

__device__ __forceinline__ double fma_t(double a, double b, double c) { return fma(a, b, c); }
__device__ __forceinline__ float fma_t(float a, float b, float c) { return fmaf(a, b, c); }

// sub-warp butterfly sum over `width` lanes (power of two); every lane of the group gets the total
template <typename T>
__device__ __forceinline__ T group_sum(T v, int width)
{
    for (int o = width >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}
template <typename T, int WIDTH>
__device__ __forceinline__ T group_sum_c(T v)
{
#pragma unroll
    for (int o = WIDTH >> 1; o > 0; o >>= 1) v += __shfl_xor_sync(kFull, v, o);
    return v;
}

// step 3 of the dot's order: the fixed tree over the 8 warp sums of a CTA
__device__ __forceinline__ double warp_sums_tree(const double *s)
{
    static_assert(kWarpsPerCta == 8, "the fixed tree below adds 8 warp sums");
    return ((s[0] + s[1]) + (s[2] + s[3])) + ((s[4] + s[5]) + (s[6] + s[7]));
}

// steps 2 and 3 of the dot's order (DotStore); every thread of the CTA must call it, so the kernel bodies before it
// return, never exit, early, and hold no __syncthreads
__device__ __forceinline__ void dot_partial(double acc, double *partials)
{
    __shared__ double warp_sum[kWarpsPerCta];
    acc = group_sum_c<double, 32>(acc);
    if ((threadIdx.x & 31) == 0) warp_sum[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) partials[blockIdx.x] = warp_sums_tree(warp_sum);
}

// dot_partial for ShiftStore's two sums, each in that order; xy == NULL (no dots) skips it (uniform over the CTA)
__device__ __forceinline__ void shift_partials(double xy, double yy, double *pxy, double *pyy)
{
    __shared__ double warp_sum[2][kWarpsPerCta];
    if (!pxy) return;
    xy = group_sum_c<double, 32>(xy);
    yy = group_sum_c<double, 32>(yy);
    if ((threadIdx.x & 31) == 0) {
        warp_sum[0][threadIdx.x >> 5] = xy;
        warp_sum[1][threadIdx.x >> 5] = yy;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        pxy[blockIdx.x] = warp_sums_tree(warp_sum[0]);
        pyy[blockIdx.x] = warp_sums_tree(warp_sum[1]);
    }
}

// number of entries of a[0..size) that are <= key: the reference's
// binary_search_right_boundary_kernel (parallel_balanced_spmv.c:17-37), usable on host and device.
__host__ __device__ __forceinline__ int right_boundary(const int *a, int key, int size)
{
    int start = 0, stop = size - 1;
    while (stop >= start) {
        const int median = (int)(((long long)stop + start) >> 1);
        if (key >= a[median]) start = median + 1; else stop = median - 1;
    }
    return start;
}
#endif  // __CUDACC__

}  // namespace sb
