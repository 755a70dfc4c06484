// spmv_b200.cu -- the C-ABI of libspmv_b200.so: the four drop-in entry points of include/spmv.h, the
// exported name tables, and the extensions of include/spmv_b200.h.  Handle construction uploads (or
// adopts) the CSR arrays once and builds the device layout of the requested SPMV_METHODS value;
// spmv() launches the matching sm_100a kernel family.  There is no CPU compute path in this file.
#include <cstdarg>
#include <algorithm>
#include <atomic>
#include <mutex>
#include <string>
#include <map>
#include <utility>
#include <type_traits>
#include <cmath>
#include <vector>
#include <cub/device/device_scan.cuh>
#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"
#include "csr_kernels.cuh"
#include "tile_kernels.cuh"
#include "sell.cuh"
#include "csr5.cuh"
#include "long_rows.cuh"
#include "band_seg.cuh"
#include "refresh.cuh"

namespace sb {

int permute_positions(int m, const int *RowPtr, const int *ColIdx, const int *index, int *RowPtr_out, int *ColIdx_out,
                      int *pos_out);  // reorder.cu

// ------------------------------------------------------------------------------------------------
// error latch, launch counter, options
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static std::atomic<unsigned long long> g_launches{0};
static std::atomic<long long> g_live_allocations{0};

void set_error(const char *fmt, ...)
{
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
    fprintf(stderr, "[spmv_b200] %s\n", g_err);
}

bool cuda_ok(cudaError_t e, const char *what, const char *file, int line)
{
    if (e == cudaSuccess) return true;
    set_error("CUDA error %s (%s) at %s:%d in `%s`", cudaGetErrorName(e), cudaGetErrorString(e), file, line, what);
    return false;
}

void count_launch(int n) { g_launches.fetch_add((unsigned long long)n, std::memory_order_relaxed); }
void count_allocation(int delta) { g_live_allocations.fetch_add(delta, std::memory_order_relaxed); }

struct Options {
    std::mutex mu;
    std::map<std::string, long long> v{{"sell_sigma", 256}, {"csr5_sigma", 0}, {"block_nnz", 512},
                                       {"tile_items", 8},   {"tpr", 0},         {"x_bands", 0},
                                       {"force_merge", 0}, {"sell_cap", 1024},
                                       {"long_thr", 0},    {"pipeline", 1},   {"sell_variant", -1},
                                       {"seg_bands", 0},    {"seg_prefetch", 1}, {"seg_ctas", 2},  {"auto", 0},     {"reorder", 0},    {"row_bins", 1},
                                       {"pin_host", 1},     {"refresh", 0},    {"axpby_fused", 1}};
    std::map<std::string, bool> user_set;
};
static Options &options()
{
    static Options o;
    return o;
}
static long long opt(const char *key)
{
    Options &o = options();
    std::lock_guard<std::mutex> g(o.mu);
    auto it = o.v.find(key);
    if (it == o.v.end()) return -1;
    if (!o.user_set[key]) {  // environment: SPMV_B200_<KEY>
        std::string env = "SPMV_B200_";
        for (const char *p = key; *p; ++p) env.push_back((char)toupper(*p));
        if (const char *e = getenv(env.c_str())) return atoll(e);
    }
    return it->second;
}

// Every option a create reads, each read once and with its rule applied (the meaning of each field: CreateOptions)
static CreateOptions read_create_options()
{
    CreateOptions o;
    o.sell_sigma = (int)(std::clamp(opt("sell_sigma"), (long long)kSellC, (long long)kSellMaxSigma) / kSellC * kSellC);
    const long long variant = opt("sell_variant");
    o.sell_variant = variant == 0 || variant == 2 ? (int)variant : -1;
    const long long cap = opt("sell_cap");  // 0 = off (the reference's widths), else the widest slice allowed
    o.sell_cap = cap <= 0 ? 0 : (int)std::clamp(cap, 32LL, 1LL << 20);
    const long long c5 = opt("csr5_sigma");
    o.csr5_sigma = c5 == 4 || c5 == 8 || c5 == 16 ? (int)c5 : 0;
    o.block_nnz = std::max(opt("block_nnz"), 32LL);
    o.tile_items = opt("tile_items") == 4 ? 4 : 8;
    const long long tpr = opt("tpr");
    o.tpr = tpr == 1 || tpr == 2 || tpr == 4 || tpr == 8 || tpr == 16 || tpr == 32 ? (int)tpr : 0;
    // any tpr but 0 switches the row bins off, also a value such as 3 that takes the tpr from the mean
    o.row_bins = tpr == 0 && opt("row_bins") != 0;
    o.long_thr = opt("long_thr");
    const long long x_bands = opt("x_bands");
    o.x_bands = x_bands == 0 ? 0 : (int)std::clamp(x_bands, 1LL, (long long)kMaxBands);
    const long long seg_bands = opt("seg_bands");
    o.seg_bands = seg_bands == 0 ? 0 : seg_bands < 2 ? -1 : (int)std::min(seg_bands, (long long)kSegMaxBands);
    o.force_merge = opt("force_merge") != 0;
    o.pipeline = opt("pipeline") != 0;
    o.auto_pick = opt("auto") != 0;
    o.reorder = opt("reorder") != 0;
    o.pin_host = opt("pin_host") != 0;
    o.refresh = opt("refresh") != 0;
    o.axpby_fused = opt("axpby_fused") != 0;
    return o;
}

// ------------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------------
static bool is_device_ptr(const void *p)
{
    if (!p) return false;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
}

static inline int blocks_for(long long threads) { return (int)((threads + kThreads - 1) / kThreads); }

// Column bands: the n columns cut into K bands of band_cols = ceil(n / K).  Band b of K holds the columns [lo, hi);
// the last band ends at n, so K = 1 is all n columns.
static int cols_per_band(const DeviceState *st, int K) { return (int)(((long long)st->n + K - 1) / K); }
static std::pair<long long, long long> band_columns(const DeviceState *st, int b, int K)
{
    const long long n = st->n, lo = (long long)b * st->band_cols, hi = lo + st->band_cols;
    return {lo < n ? lo : n, b == K - 1 || hi > n ? n : hi};
}

// f(T()) with the handle's value type: T = double for fp64, float for fp32
template <typename F>
static auto with_precision(const DeviceState *st, F f)
{
    return st->vsize == 8 ? f(double()) : f(float());
}

// f(std::integral_constant<int, V>()) for the first V of the list equal to v, or for the last V when none is
template <int V, int... Rest, typename F>
static auto with_value(int v, F f)
{
    if constexpr (sizeof...(Rest) == 0) return f(std::integral_constant<int, V>());
    else return v == V ? f(std::integral_constant<int, V>()) : with_value<Rest...>(v, f);
}

struct DeviceGuard {  // library code is device-agnostic: run on the handle's device, then restore
    int prev = -1, want;
    explicit DeviceGuard(int dev) : want(dev)
    {
        if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
        if (prev != want) cudaSetDevice(want);
    }
    ~DeviceGuard() { if (prev >= 0 && prev != want) cudaSetDevice(prev); }
};

// Copy `count` values from the device to the host on the handle's stream and wait for them: every scalar a builder
// reads back, so that create is ordered on st->stream alone.
template <typename V>
static bool read_back(const DeviceState *st, V *host, const V *device, size_t count = 1)
{
    SB_TRY(cudaMemcpyAsync(host, device, count * sizeof(V), cudaMemcpyDeviceToHost, st->stream));
    SB_TRY(cudaStreamSynchronize(st->stream));
    return true;
}

// Zero a one-element device counter, enqueue `launch(counter)` on the handle's stream, and read the counter back.
template <typename C, typename Launch>
static bool read_counter(const DeviceState *st, C *value, Launch launch)
{
    DeviceArray<C> counter;
    if (!counter.alloc(1)) return false;
    SB_TRY(cudaMemsetAsync(counter, 0, sizeof(C), st->stream));
    launch(counter.get());
    SB_TRY(cudaGetLastError());
    return read_back(st, value, counter.get());
}

// An optional step failed: forget its CUDA and library errors and reset what it built.  Whether that counts as a
// layout fallback (spmv_b200_info "layout_fallbacks") is the caller's to say.
template <typename... Built>
static void abandon(Built &...built)
{
    cudaGetLastError();
    spmv_b200_clear_error();
    ((built = {}), ...);
}

template <typename V>
static bool exclusive_scan(const V *in, V *out, int count, cudaStream_t s)
{
    size_t bytes = 0;
    SB_TRY(cub::DeviceScan::ExclusiveSum(nullptr, bytes, in, out, count, s));
    DeviceArray<unsigned char> tmp;
    return tmp.alloc(bytes) && SB_CUDA(cub::DeviceScan::ExclusiveSum(tmp.get(), bytes, in, out, count, s)) &&
           SB_CUDA(cudaStreamSynchronize(s));
}

// ------------------------------------------------------------------------------------------------
// layout builders (handle construction, a2)
// ------------------------------------------------------------------------------------------------
static void unpin(DeviceState::PinSlot &slot)
{
    if (slot.registered && cudaHostUnregister(const_cast<void *>(slot.ptr)) != cudaSuccess) cudaGetLastError();
    slot = DeviceState::PinSlot();
}

// see DeviceState::pin
static void note_host_buffer(DeviceState *st, int which, const void *p, size_t bytes)
{
    DeviceState::PinSlot &slot = st->pin[which];
    if (slot.ptr != p || slot.bytes != bytes) {
        unpin(slot);
        slot.ptr = p;
        slot.bytes = bytes;
        slot.seen = 1;
        return;
    }
    if (slot.registered || slot.seen < 0 || bytes < (1u << 20)) return;
    if (++slot.seen < 2) return;
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) { cudaGetLastError(); slot.seen = -1; return; }
    if (a.type != cudaMemoryTypeUnregistered) { slot.seen = -1; return; }  // already pinned by the caller
    if (cudaHostRegister(const_cast<void *>(p), bytes, cudaHostRegisterDefault) == cudaSuccess) slot.registered = true;
    else { cudaGetLastError(); slot.seen = -1; }  // e.g. registered through another handle: leave it alone
}

// Option "refresh": a source map that cannot be made costs the handle its refresh, never its layout.
static void map_failure(DeviceState *st)
{
    abandon();
    st->map_failed = true;
}

// Source map of the value array `val` a builder reads: the band-major copy's, the permuted upload's (option
// "reorder"), or -- the CSR in the caller's own order -- k + 1 at k, made in `tmp`.
static const int *source_map_of(DeviceState *st, const void *val, DeviceArray<int> &tmp)
{
    if (val == st->v.val.get()) return st->v.map;
    if (st->upload.map) return st->upload.map;
    if (!tmp.alloc((size_t)st->nnz)) return nullptr;
    map_iota_kernel<<<blocks_for(st->nnz), kThreads, 0, st->stream>>>(st->nnz, tmp);
    return tmp;
}

// The source map of a layout's value array: `move(src, map)` enqueues the builder's value-moving kernel again with
// T = int, reading the source map of `val` (what the builder read the values from) and writing `map` in place of
// the values.  Padding slots get the builder's own zero, which is the map's "no source".
template <typename Move>
static void build_map(DeviceState *st, const void *val, DeviceArray<int> &map, size_t count, Move move)
{
    if (!st->refresh || st->map_failed) return;
    DeviceArray<int> tmp;
    const int *src = source_map_of(st, val, tmp);
    if (src && map.alloc(count) && move(src, map.get()) && SB_CUDA(cudaGetLastError())) return;
    map.reset();
    map_failure(st);
}

static void free_state(DeviceState *st)
{
    if (!st) return;
    DeviceGuard g(st->device);
    unpin(st->pin[0]);
    unpin(st->pin[1]);
    for (int i = 0; i < kMaxPieces; ++i) if (st->ev_in[i]) cudaEventDestroy(st->ev_in[i]);
    for (int i = 0; i < kPipeChunks; ++i) if (st->ev_out[i]) cudaEventDestroy(st->ev_out[i]);
    if (st->ev_start) cudaEventDestroy(st->ev_start);
    if (st->ev_x) cudaEventDestroy(st->ev_x);
    if (st->s_in) cudaStreamDestroy(st->s_in);
    if (st->s_out) cudaStreamDestroy(st->s_out);
    st->magic = 0;
    delete st;  // frees the device arrays, on the handle's device (g)
}

// Device facts the layout decisions need.  (The persisting-L2 carve-out, cudaLimitMaxL2FetchGranularity and an
// access-policy window over x were options in round 1; none of them moved any measured configuration -- C2 then, the
// C5 shard in round 2 -- and they are gone.)
static void apply_device_limits(DeviceState *st)
{
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, st->device) != cudaSuccess) { cudaGetLastError(); return; }
    st->dev_sms = prop.multiProcessorCount;
    st->dev_l2 = prop.l2CacheSize;
}

static int pick_tpr(const DeviceState *st)
{
    if (st->opts.tpr) return st->opts.tpr;
    const double mean = st->a_m > 0 ? (double)st->nnz / st->a_m : 0.0;
    int tpr = 1;
    // measured on B200 (scripts/sweep.py): ~7 entries per lane is the sweet spot -- fewer lanes per row
    // means more independent x gathers in flight per thread (mean 5 -> 1, 10.7 -> 2, 27 -> 4, 32 -> 8)
    while (tpr < 32 && 7.0 * tpr < mean) tpr <<= 1;
    return tpr;
}

// the bytes of x that random gathers can keep in L2
static double l2_reach(long long dev_l2) { return dev_l2 > 0 ? 0.5 * (double)dev_l2 : 63.0 * 1048576.0; }

// Locality probe (m > 0, nnz > 0): the share of entries further than 1/8 of the L2 reach from the (scaled) diagonal.
// > 25 % = gather-dominated (bound by L2 requests), else diagonal-local (bound by DRAM).  It decides whether banding
// can pay (decide_bands), which SELL kernel flavour runs (build_sell) and the method option "auto" picks.
static bool probe_locality(DeviceState *st)
{
    const int halfwidth = (int)(0.125 * l2_reach(st->dev_l2) / st->vsize);
    unsigned long long h_far = 0;
    const bool probed = read_counter(st, &h_far, [&](unsigned long long *far) {
        band_locality_kernel<<<blocks_for(st->m), kThreads, 0, st->stream>>>(
            st->m, (double)st->n / st->m, halfwidth, st->rowptr, st->col, far);
    });
    if (!probed) return false;  // a 8-byte allocation or a trivial kernel failed: the device is unusable
    st->far_fraction = (double)h_far / (double)st->nnz;
    return true;
}

// The column bands of a matrix with m > 0 rows and nnz > 0 entries: {K of the band-major copy (1 = none), bands of
// the band segments (0 = none)}.
static std::pair<int, int> decide_bands(long long m, long long n, long long nnz, int vsize, long long dev_l2,
                                        double far_fraction, const CreateOptions &o)
{
    if (o.seg_bands >= 2) return {1, o.seg_bands};  // forced band segments: no band-major copy
    int K = o.x_bands, seg = 0;
    if (K == 0) {
        K = 1;
        const double xbytes = (double)n * vsize, usable = l2_reach(dev_l2);
        // x up to ~1.2x the reach still gathers at >= 85 % of the L2 rate (profiles/r01_gather_probe.txt) and
        // banding costs 15-20 % (virtual row pointers, partial y): R-MAT s24 fp32 (x = 64 MiB) measured 7-15 %
        // FASTER unbanded, uniform fp64 (x = 128 MiB) 1.9x faster banded.  Banding only pays when the accesses
        // are NOT already diagonal-local.
        if (xbytes > 1.2 * usable && far_fraction > 0.25) {
            const long long k = (long long)ceil(xbytes / (0.75 * usable));
            if (k <= kMaxBands && (double)nnz / ((double)k * m) >= 4.0) K = (int)k;
            else if (o.seg_bands == 0) {
                // hyper-sparse bands (< 4 entries per virtual row) would cost more in row pointers than they save:
                // band segments (band_seg.cuh).  More bands = a smaller slice of x = fewer L2 misses of the gathers,
                // but more and shorter segments for the merge pass.  Measured on the C5 shard (x = 2 GiB, 16 per
                // row; scripts/c5_sweep.sh): 32 bands 5.24 ms, 40: 4.94, 44: 4.88, 48: 4.78, 52: 4.92, 56: 4.96,
                // 64: 5.19 -- a slice of about 2/3 of the reach
                const long long kc = (long long)ceil(xbytes / (0.68 * usable));
                seg = (int)(kc < 2 ? 2 : (kc > kSegMaxBands ? kSegMaxBands : kc));
            }
        }
    }
    if (m * K > 0x7fffffffLL - 8192) K = 1;  // the m·K virtual rows must stay 32-bit
    return {K, seg};
}

// Build the band-major copy of K > 1 column bands and make it the active view.
template <typename T>
static void build_band_major(DeviceState *st, int K)
{
    const int m = st->m;
    const int band_cols = cols_per_band(st, K);
    const size_t vm = (size_t)m * K;
    DeviceArray<int> counts;
    // The band-major copy is a speed-up only: when it cannot be allocated (or built) the handle keeps running the
    // plain CSR view it already holds -- never fail a handle over an optional layout.
    auto give_up = [&]() {
        abandon(st->v);
        st->layout_fallbacks++;
    };
    if (!counts.alloc(vm + 1) || !st->v.rowptr.alloc(vm + 1 + 8) || !st->v.col.alloc((size_t)st->nnz + 8) ||
        !st->v.val.alloc((size_t)st->nnz + 8, sizeof(T)) || !st->v.y.alloc(vm, sizeof(T)))
        return give_up();
    bool ok = SB_CUDA(cudaMemsetAsync(counts + vm, 0, sizeof(int), st->stream));
    if (ok) {
        band_count_kernel<<<blocks_for(m), kThreads, 0, st->stream>>>(m, K, band_cols, st->rowptr, st->col, counts);
        ok = SB_CUDA(cudaGetLastError()) && exclusive_scan(counts.get(), st->v.rowptr.get(), (int)vm + 1, st->stream);
    }
    if (ok) {
        band_scatter_kernel<T><<<blocks_for(m), kThreads, 0, st->stream>>>(m, K, band_cols, st->rowptr, st->col, (const T *)st->val,
                                                                           st->v.rowptr, st->v.col, st->v.val.as<T>());
        ok = SB_CUDA(cudaGetLastError()) && SB_CUDA(cudaStreamSynchronize(st->stream));
    }
    if (!ok) return give_up();
    build_map(st, st->val, st->v.map, (size_t)st->nnz, [&](const int *src, int *map) {
        band_scatter_kernel<int><<<blocks_for(m), kThreads, 0, st->stream>>>(m, K, band_cols, st->rowptr, st->col, src, st->v.rowptr, st->v.col, map);
        return true;
    });
    st->x_bands = K;
    st->band_cols = band_cols;
    st->a_m = (int)vm; st->a_rowptr = st->v.rowptr; st->a_col = st->v.col; st->a_val = st->v.val.get();
}

// a9 on the device for `parts` partitions; *starved = some partition owns no whole row (a10)
static bool build_splitter(DeviceState *st, int m, const int *rowptr, int parts, DeviceArray<int> &out, int *starved)
{
    if (!out.alloc((size_t)parts + 1)) return false;
    splitter_kernel<<<blocks_for(parts + 1), kThreads, 0, st->stream>>>(parts, st->nnz, m, rowptr, out);
    SB_TRY(cudaGetLastError());
    return read_counter(st, starved, [&](int *flag) {
        splitter_starved_kernel<<<blocks_for(parts), kThreads, 0, st->stream>>>(parts, m, out, flag);
    });
}

// carry arrays of the tile kernels: one (row, value) per tile + the level-2 list of the two-level fix-up
static bool alloc_carries(DeviceState *st, int tiles)
{
    const size_t t = tiles > 0 ? (size_t)tiles : 1;
    const size_t g2 = 2 * ((t + kCarryGroup - 1) / kCarryGroup);
    return st->tile.carry_val.alloc(t, st->vsize) && st->tile.carry_row.alloc(t) && st->tile.carry2_val.alloc(g2, st->vsize) &&
           st->tile.carry2_row.alloc(g2);
}

// y[row] += the carries of `tiles` consecutive tiles, in tile order; long lists in two levels
template <typename T>
static void launch_carry_fixup(DeviceState *st, cudaStream_t s, int tiles, const int *carry_row, const T *carry_val, T *y)
{
    if (tiles <= 0) return;
    if (tiles < 1024) {
        carry_fixup_kernel<T><<<blocks_for(tiles), kThreads, 0, s>>>(tiles, carry_row, carry_val, y);
        count_launch();
        return;
    }
    const int groups = (tiles + kCarryGroup - 1) / kCarryGroup;
    carry_group_kernel<T><<<blocks_for((long long)groups * 32), kThreads, 0, s>>>(tiles, carry_row, carry_val, y, st->tile.carry2_row, st->tile.carry2_val.as<T>());
    carry_fixup_kernel<T><<<blocks_for(2 * groups), kThreads, 0, s>>>(2 * groups, st->tile.carry2_row, st->tile.carry2_val.as<T>(), y);
    count_launch(2);
}

// Segment list for the entries the main kernel does not cover: covered[r] leading entries of row r are done
// by the main kernel, the rest by long_seg_kernel / long_final_kernel (long_rows.cuh).  Takes `covered` over.
static bool build_long_rows(DeviceState *st, DeviceArray<int> covered, bool accumulate)
{
    const int m = st->a_m;
    DeviceArray<int> cnt_r, cnt_s, scan_r, scan_s;
    bool ok = cnt_r.alloc((size_t)m + 1) && cnt_s.alloc((size_t)m + 1) && scan_r.alloc((size_t)m + 1) && scan_s.alloc((size_t)m + 1);
    if (ok) {
        long_count_kernel<<<blocks_for((long long)m + 1), kThreads, 0, st->stream>>>(m, st->a_rowptr, covered, cnt_r, cnt_s);
        ok = SB_CUDA(cudaGetLastError()) && exclusive_scan(cnt_r.get(), scan_r.get(), m + 1, st->stream) &&
             exclusive_scan(cnt_s.get(), scan_s.get(), m + 1, st->stream);
    }
    int totals[2] = {0, 0};
    if (ok) ok = read_back(st, &totals[0], scan_r + m) && read_back(st, &totals[1], scan_s + m);
    st->lr.rows = totals[0];
    st->lr.segs = totals[1];
    st->lr.accumulate = accumulate;
    if (ok && st->lr.rows > 0) {
        ok = st->lr.row.alloc((size_t)st->lr.rows) && st->lr.start.alloc((size_t)st->lr.rows) &&
             st->lr.seg_ptr.alloc((size_t)st->lr.rows + 1) && st->lr.seg_row.alloc((size_t)st->lr.segs) &&
             st->lr.partial.alloc((size_t)st->lr.segs, st->vsize);
        if (ok) {
            long_fill_kernel<<<blocks_for((long long)m + 1), kThreads, 0, st->stream>>>(
                m, st->a_rowptr, covered, scan_r, scan_s, st->lr.row, st->lr.start, st->lr.seg_ptr, st->lr.seg_row);
            ok = SB_CUDA(cudaGetLastError()) && SB_CUDA(cudaStreamSynchronize(st->stream));
        }
    }
    return ok;
}

// Method_Parallel: rows longer than ~256 entries per lane would keep one lane group busy long after the rest
// of the grid has drained; they go to the long-row path as a whole.
static bool build_long_rows_at(DeviceState *st, int thr)
{
    st->lr.thr = thr;
    DeviceArray<int> covered;
    if (!covered.alloc((size_t)st->a_m + 1)) return false;
    long_cover_threshold_kernel<<<blocks_for(st->a_m), kThreads, 0, st->stream>>>(st->a_m, 0, thr, st->a_rowptr, covered);
    SB_TRY(cudaGetLastError());
    return build_long_rows(st, std::move(covered), /*accumulate=*/false);
}

static bool build_long_rows_threshold(DeviceState *st)
{
    long long thr = st->opts.long_thr;  // 0 = automatic, < 0 = off
    if (thr < 0) { st->lr.thr = 0x7fffffff; return true; }
    const bool automatic = thr == 0;
    if (automatic) { thr = 256LL * st->tpr; if (thr < 512) thr = 512; if (thr > 4096) thr = 4096; }
    if (!build_long_rows_at(st, (int)thr)) return false;
    // A short-row matrix WITH hub rows (power-law graphs): one lane-group size for all rows leaves most lanes
    // waiting for the longest row of their warp.  Bin the rows by length class instead -- stable radix sort of the
    // row ids by bin -- and give every bin its own launch; rows beyond 128 entries go to the long-row path.
    // (C3: 1.26 ms with one lane-group size, 1.20 ms re-split at 128 entries, see DESIGN.md for the binned figure)
    if (automatic && st->lr.rows > 0 && st->tpr <= 4 && st->opts.row_bins) {
        st->lr = {};
        if (!build_long_rows_at(st, 128)) return false;
        const int m = st->a_m;
        DeviceArray<unsigned char> key_in, key_out, tmp;
        DeviceArray<int> ids, d_ptr;
        size_t tmp_bytes = 0;
        bool ok = key_in.alloc((size_t)m) && key_out.alloc((size_t)m) && ids.alloc((size_t)m) && st->lr.bin_list.alloc((size_t)m) &&
                  d_ptr.alloc(5);
        if (ok) {
            row_bin_kernel<<<blocks_for(m), kThreads, 0, st->stream>>>(m, st->a_rowptr, key_in, ids);
            ok = SB_CUDA(cudaGetLastError()) &&
                 SB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, key_in.get(), key_out.get(), ids.get(), st->lr.bin_list.get(), m, 0, 2, st->stream)) &&
                 tmp.alloc(tmp_bytes) &&
                 SB_CUDA(cub::DeviceRadixSort::SortPairs(tmp.get(), tmp_bytes, key_in.get(), key_out.get(), ids.get(), st->lr.bin_list.get(), m, 0, 2, st->stream));
        }
        int h_ptr[5] = {0, 0, 0, 0, 0};
        if (ok) {
            sorted_key_ptr_kernel<<<1, kThreads, 0, st->stream>>>(m, 4, key_out, d_ptr);  // first sorted row of every bin
            ok = SB_CUDA(cudaGetLastError()) && read_back(st, h_ptr, d_ptr.get(), 5);
        }
        if (!ok) return false;
        for (int b = 0; b < 4; ++b) st->lr.bin_ptr[b] = h_ptr[b];  // bin b = list[bin_ptr[b], bin_ptr[b+1]); bin 3 is unused
        st->lr.binned = true;
    }
    return true;
}

// Host-pointer pipeline of the CSR-vector kernel (option "pipeline", default on): which prefix of x each of
// the kPipeChunks row chunks needs (unbanded view; a band needs exactly its own slice of x).
static bool build_pipeline(DeviceState *st)
{
    st->pipeline = false;
    if (!st->opts.pipeline || st->lr.rows > 0 || st->m < (1 << 16)) return true;
    if (st->x_bands > 1) { st->pipeline = st->x_bands <= kMaxPieces; return true; }
    DeviceArray<int> d;
    if (!d.alloc(kPipeChunks)) return false;
    SB_TRY(cudaMemsetAsync(d, 0, kPipeChunks * sizeof(int), st->stream));
    chunk_xmax_kernel<<<blocks_for(st->m), kThreads, 0, st->stream>>>(st->m, kPipeChunks, st->rowptr, st->col, d);
    const bool ok = SB_CUDA(cudaGetLastError()) && read_back(st, st->chunk_xmax, d.get(), kPipeChunks);
    st->pipeline = ok;
    return ok;
}

static bool build_tiles(DeviceState *st, bool merge)
{
    const int ipt = st->tile.items = st->opts.tile_items;
    const long long per_tile = (long long)kThreads * ipt;
    const long long total = merge ? (long long)st->a_m + st->nnz : (long long)st->nnz;
    st->tile.count = (int)((total + per_tile - 1) / per_tile);
    if (st->tile.count < 1) st->tile.count = 1;
    if (merge) {
        if (!st->tile.merge_coords.alloc((size_t)st->tile.count + 1)) return false;
        merge_coords_kernel<<<blocks_for(st->tile.count + 1), kThreads, 0, st->stream>>>(
            st->tile.count, (int)per_tile, st->nnz, st->a_m, st->a_rowptr, st->tile.merge_coords);
    } else {
        if (!st->tile.rows.alloc((size_t)st->tile.count + 1)) return false;
        tile_rows_kernel<<<blocks_for(st->tile.count + 1), kThreads, 0, st->stream>>>(
            st->tile.count, (int)per_tile, st->nnz, st->a_m, st->a_rowptr, st->tile.rows);
    }
    SB_TRY(cudaGetLastError());
    if (!alloc_carries(st, st->tile.count)) return false;
    st->kernel = merge ? SPMV_B200_KERNEL_MERGE_PATH : SPMV_B200_KERNEL_NNZ_SPLIT;
    return true;
}

template <typename T>
static bool build_sell(DeviceState *st)
{
    st->sell.sigma = st->opts.sell_sigma;
    const int windows = st->a_m / st->sell.sigma;
    st->sell.banner = windows * st->sell.sigma;  // reference sell_C_Sigma_spmv.c:148-156
    st->sell.slices = st->sell.banner / kSellC;
    st->tpr = pick_tpr(st);  // for the CSR tail rows [banner, m)
    st->kernel = SPMV_B200_KERNEL_SELL;
    // HBM-bound (diagonal-local) matrices want every warp slot filled: 4 columns per step in 32 registers
    // (C4: 0.86 -> 0.98 of the measured peak); gather-bound ones run best with 8 columns per step (C2: 0.43 vs 0.39)
    st->sell.variant = st->opts.sell_variant >= 0 ? st->opts.sell_variant : st->far_fraction > 0.25 ? 0 : 2;
    // covered[r]: entries of row r stored in its slice (sell_width_kernel); tail rows [banner, m) stay CSR,
    // except hub rows, which csr_tail_kernel zeroes and the long-row path then adds as a whole
    const int cap = st->opts.sell_cap;
    DeviceArray<int> covered;
    if (cap) {
        if (!covered.alloc((size_t)st->a_m + 1)) return false;
        st->lr.thr = 4096;
        long_cover_threshold_kernel<<<blocks_for(st->a_m), kThreads, 0, st->stream>>>(st->a_m, st->sell.banner, st->lr.thr, st->a_rowptr, covered);
        SB_TRY(cudaGetLastError());
    }
    if (st->sell.banner == 0) return cap ? build_long_rows(st, std::move(covered), /*accumulate=*/true) : true;
    int pow2 = 1;
    while (pow2 < st->sell.sigma) pow2 <<= 1;
    if (!st->sell.perm.alloc((size_t)st->sell.banner)) return false;
    sell_sort_kernel<<<windows, kThreads, (size_t)pow2 * sizeof(unsigned long long), st->stream>>>(
        st->sell.sigma, pow2, st->a_rowptr, st->sell.perm);
    SB_TRY(cudaGetLastError());
    DeviceArray<long long> count;
    if (!st->sell.width.alloc((size_t)st->sell.slices) || !st->sell.full.alloc((size_t)st->sell.slices) ||
        !count.alloc((size_t)st->sell.slices + 1) || !st->sell.slice_ptr.alloc((size_t)st->sell.slices + 1))
        return false;
    SB_TRY(cudaMemsetAsync(count, 0, ((size_t)st->sell.slices + 1) * sizeof(long long), st->stream));
    sell_width_kernel<<<blocks_for((long long)st->sell.slices * 32), kThreads, 0, st->stream>>>(
        st->sell.slices, cap, st->a_rowptr, st->sell.perm, st->sell.width, st->sell.full, count, covered);
    SB_TRY(cudaGetLastError());
    if (cap && !build_long_rows(st, std::move(covered), /*accumulate=*/true)) return false;
    if (!exclusive_scan(count.get(), st->sell.slice_ptr.get(), st->sell.slices + 1, st->stream)) return false;
    if (!read_back(st, &st->sell.padded, st->sell.slice_ptr + st->sell.slices)) return false;
    if (!st->sell.col.alloc((size_t)st->sell.padded) || !st->sell.val.alloc((size_t)st->sell.padded, sizeof(T))) return false;
    sell_fill_kernel<T><<<blocks_for((long long)st->sell.slices * 32), kThreads, 0, st->stream>>>(
        st->sell.slices, st->a_rowptr, st->a_col, (const T *)st->a_val, st->sell.perm, st->sell.slice_ptr, st->sell.col,
        st->sell.val.as<T>());
    SB_TRY(cudaGetLastError());
    build_map(st, st->a_val, st->sell.map, (size_t)st->sell.padded, [&](const int *src, int *map) {
        sell_fill_kernel<int><<<blocks_for((long long)st->sell.slices * 32), kThreads, 0, st->stream>>>(
            st->sell.slices, st->a_rowptr, st->a_col, src, st->sell.perm, st->sell.slice_ptr, st->sell.col, map);
        return true;
    });
    return true;
}

template <typename T>
static bool build_csr5(DeviceState *st)
{
    // 0 = automatic: 16, or 8 on small matrices (twice the tiles to fill the GPU)
    const int sigma = st->c5.sigma = st->opts.csr5_sigma ? st->opts.csr5_sigma : st->nnz < (1 << 25) ? 8 : 16;
    // anonymouslib_avx2.h:124-146 at omega = 32
    int base = 2, by = 1;
    while (base < kC5Omega * sigma) { base *= 2; by++; }
    int bs = 1;
    base = 2;
    while (base < kC5Omega) { base *= 2; bs++; }
    st->c5.bit_y = by;
    st->c5.bit_ss = bs;  // by + bs + sigma <= 32 for sigma <= 16: one descriptor word per lane
    const int tile_nnz = kC5Omega * sigma;
    const int p = (int)(((long long)st->nnz + tile_nnz - 1) / tile_nnz);
    st->c5.p = p;
    st->kernel = SPMV_B200_KERNEL_CSR5;
    st->tile.count = p;
    if (p == 0) return true;
    DeviceArray<uint32_t> raw;
    DeviceArray<int> off_cnt;
    if (!raw.alloc((size_t)p + 1) || !st->c5.tile_ptr.alloc((size_t)p + 1) || !st->c5.tile_desc.alloc((size_t)p * kC5Omega) ||
        !off_cnt.alloc((size_t)p + 1) || !st->c5.off_ptr.alloc((size_t)p + 1))
        return false;
    c5_tile_ptr_kernel<<<blocks_for(p + 1), kThreads, 0, st->stream>>>(p, sigma, st->nnz, st->a_m, st->a_rowptr, raw);
    c5_tile_dirty_kernel<<<blocks_for(p + 1), kThreads, 0, st->stream>>>(p, st->a_m, st->a_rowptr, raw, st->c5.tile_ptr);
    SB_TRY(cudaMemsetAsync(off_cnt, 0, ((size_t)p + 1) * sizeof(int), st->stream));
    c5_tile_desc_kernel<<<blocks_for((long long)p * 32), kThreads, 0, st->stream>>>(
        p, sigma, by, bs, st->a_rowptr, st->c5.tile_ptr, st->c5.tile_desc, off_cnt);
    SB_TRY(cudaGetLastError());
    if (!exclusive_scan(off_cnt.get(), st->c5.off_ptr.get(), p + 1, st->stream)) return false;
    uint32_t tail_word = 0;
    if (!read_back(st, &st->c5.num_offsets, st->c5.off_ptr + p) || !read_back(st, &tail_word, st->c5.tile_ptr + (p - 1)))
        return false;
    st->c5.tail_start = (int)(tail_word & 0x7FFFFFFFu);  // anonymouslib_avx2.h:177
    if (st->c5.num_offsets > 0) {
        if (!st->c5.off.alloc((size_t)st->c5.num_offsets)) return false;
        SB_TRY(cudaMemsetAsync(st->c5.off, 0, (size_t)st->c5.num_offsets * sizeof(int), st->stream));
        c5_desc_offset_kernel<<<blocks_for((long long)p * 32), kThreads, 0, st->stream>>>(
            p, sigma, by, bs, st->a_rowptr, st->c5.tile_ptr, st->c5.tile_desc, st->c5.off_ptr, st->c5.off);
        SB_TRY(cudaGetLastError());
    }
    if (!st->c5.col.alloc((size_t)st->nnz) || !st->c5.val.alloc((size_t)st->nnz, sizeof(T))) return false;
    c5_transpose_kernel<T><<<blocks_for(st->nnz), kThreads, 0, st->stream>>>(
        st->nnz, sigma, p, st->c5.tile_ptr, st->a_col, (const T *)st->a_val, st->c5.col, st->c5.val.as<T>());
    SB_TRY(cudaGetLastError());
    build_map(st, st->a_val, st->c5.map, (size_t)st->nnz, [&](const int *src, int *map) {
        c5_transpose_kernel<int><<<blocks_for(st->nnz), kThreads, 0, st->stream>>>(st->nnz, sigma, p, st->c5.tile_ptr, st->a_col, src, st->c5.col, map);
        return true;
    });
    return alloc_carries(st, p);
}

// Band segments (band_seg.cuh): stable bucketing of the CSR entries by col / band_cols, segment-end bits, row masks,
// tile table and the per-block positions of the merge pass.
template <typename T, typename MaskT>
static bool build_band_seg_t(DeviceState *st)
{
    const int K = st->seg.bands, nnz = st->nnz, m = st->m;
    st->band_cols = cols_per_band(st, K);
    st->seg.mask64 = sizeof(MaskT) == 8;
    int tiles = 0, h_cross = 0, h_segs[2] = {0, 0};
    {  // the temporaries (about 15 bytes per entry) are freed before the segment sums are allocated
        DeviceArray<int> ent_row, idx_in, idx_out, d_tab, tile_segs, blk_cnt, blk_scan, d_cross;
        DeviceArray<unsigned char> key_in, key_out, tmp;
        size_t tmp_bytes = 0;
        int h_ptr[kMaxPieces + 1] = {};
        bool ok = ent_row.alloc((size_t)nnz) && idx_in.alloc((size_t)nnz) && idx_out.alloc((size_t)nnz) && key_in.alloc((size_t)nnz) &&
                  key_out.alloc((size_t)nnz) && d_tab.alloc(4 * (size_t)(K + 1)) && d_cross.alloc(1) &&
                  st->seg.mask.alloc((size_t)m + 1, sizeof(MaskT));
        if (ok) {
            bseg_expand_kernel<MaskT><<<blocks_for(m), kThreads, 0, st->stream>>>(m, st->band_cols, K, st->rowptr, st->col, ent_row, key_in,
                                                                                  st->seg.mask.as<MaskT>());
            bseg_iota_kernel<<<blocks_for(nnz), kThreads, 0, st->stream>>>(nnz, idx_in);
            int bits = 1;
            while ((1 << bits) < K) ++bits;
            ok = SB_CUDA(cudaGetLastError()) &&
                 SB_CUDA(cub::DeviceRadixSort::SortPairs(nullptr, tmp_bytes, key_in.get(), key_out.get(), idx_in.get(), idx_out.get(), nnz, 0, bits, st->stream)) &&
                 tmp.alloc(tmp_bytes) &&
                 SB_CUDA(cub::DeviceRadixSort::SortPairs(tmp.get(), tmp_bytes, key_in.get(), key_out.get(), idx_in.get(), idx_out.get(), nnz, 0, bits, st->stream));
        }
        if (ok) {
            sorted_key_ptr_kernel<<<1, kThreads, 0, st->stream>>>(nnz, K, key_out, d_tab);
            ok = SB_CUDA(cudaGetLastError()) && read_back(st, h_ptr, d_tab.get(), (size_t)K + 1);
        }
        if (!ok) return false;
        // band b occupies slots [seg.ptr[b], seg.ptr[b] + seg.cnt[b]); starts aligned to 4 entries (16 bytes of ColIdx)
        long long slot = 0;
        for (int b = 0; b < K; ++b) {
            st->seg.ptr[b] = (int)slot;
            st->seg.cnt[b] = h_ptr[b + 1] - h_ptr[b];
            st->seg.tile0[b] = tiles;
            tiles += ceil_div(st->seg.cnt[b], kSegTile);
            slot = (slot + st->seg.cnt[b] + 3) & ~3LL;
        }
        st->seg.ptr[K] = (int)slot;
        st->seg.tile0[K] = tiles;
        st->tile.count = tiles;
        st->seg.groups = ceil_div(m, 32);
        const size_t gk = (size_t)K * st->seg.groups;
        const size_t slots = (size_t)slot + 8;
        int h_tab[4 * (kMaxPieces + 1)];
        for (int b = 0; b <= K; ++b) {
            h_tab[b] = h_ptr[b];
            h_tab[(K + 1) + b] = st->seg.ptr[b];
            h_tab[2 * (K + 1) + b] = b < K ? st->seg.cnt[b] : 0;
            h_tab[3 * (K + 1) + b] = st->seg.tile0[b];
        }
        ok = st->seg.col.alloc(slots) && st->seg.ent_val.alloc(slots, sizeof(T)) && st->seg.tile_ent.alloc((size_t)tiles + 1) &&
             st->seg.tile_seg0.alloc((size_t)tiles * kSegChunks + 4) && tile_segs.alloc((size_t)tiles * kSegChunks + 4) &&
             blk_cnt.alloc(gk + 1) && blk_scan.alloc(gk + 1) && st->seg.gbase.alloc(gk + 1) &&
             SB_CUDA(cudaMemcpyAsync(d_tab, h_tab, 4 * (size_t)(K + 1) * sizeof(int), cudaMemcpyHostToDevice, st->stream)) &&
             SB_CUDA(cudaMemsetAsync(st->seg.col, 0, slots * sizeof(int), st->stream)) &&
             SB_CUDA(cudaMemsetAsync(st->seg.ent_val.get(), 0, slots * sizeof(T), st->stream)) &&
             SB_CUDA(cudaMemsetAsync(tile_segs, 0, ((size_t)tiles * kSegChunks + 4) * sizeof(int), st->stream)) &&
             SB_CUDA(cudaMemsetAsync(blk_cnt, 0, (gk + 1) * sizeof(int), st->stream)) &&
             SB_CUDA(cudaMemsetAsync(d_cross, 0, sizeof(int), st->stream));
        if (ok) {
            bseg_gather_kernel<T><<<blocks_for(nnz), kThreads, 0, st->stream>>>(nnz, idx_out, key_out, ent_row, st->col, (const T *)st->val, d_tab,
                                                                               d_tab + (K + 1), st->seg.col, st->seg.ent_val.as<T>());
            build_map(st, st->val, st->seg.map, (size_t)slot, [&](const int *src, int *map) {  // the gaps between bands stay 0
                if (!SB_CUDA(cudaMemsetAsync(map, 0, (size_t)slot * sizeof(int), st->stream))) return false;
                bseg_gather_kernel<int><<<blocks_for(nnz), kThreads, 0, st->stream>>>(nnz, idx_out, key_out, ent_row, st->col, src, d_tab,
                                                                                     d_tab + (K + 1), st->seg.col, map);
                return true;
            });
            bseg_tile_kernel<<<blocks_for((long long)tiles * 32), kThreads, 0, st->stream>>>(tiles, K, st->band_cols, st->n, st->vsize, d_tab + 3 * (K + 1), d_tab + (K + 1), d_tab + 2 * (K + 1),
                                                                                             st->seg.col, st->seg.tile_ent, tile_segs, d_cross);
            bseg_group_count_kernel<MaskT><<<blocks_for((long long)st->seg.groups * 32), kThreads, 0, st->stream>>>(m, K, st->seg.groups, st->seg.mask.as<MaskT>(), blk_cnt);
            ok = SB_CUDA(cudaGetLastError()) && exclusive_scan(tile_segs.get(), st->seg.tile_seg0.get(), tiles * kSegChunks + 1, st->stream) &&
                 gk + 1 < 0x7fffffffULL && exclusive_scan(blk_cnt.get(), blk_scan.get(), (int)gk + 1, st->stream);
            if (ok) {
                bseg_transpose_kernel<<<blocks_for((long long)gk), kThreads, 0, st->stream>>>(K, st->seg.groups, blk_scan, st->seg.gbase);
                ok = SB_CUDA(cudaGetLastError());
            }
            ok = ok && read_back(st, &h_segs[0], st->seg.tile_seg0 + (size_t)tiles * kSegChunks) &&
                 read_back(st, &h_segs[1], blk_scan + gk) && read_back(st, &h_cross, d_cross.get());
        }
        if (!ok) return false;
    }
    if (h_segs[0] != h_segs[1]) { set_error("band segments: %d segment ends but %d (row, band) pairs", h_segs[0], h_segs[1]); return false; }
    st->seg.total = h_segs[0];
    st->seg.cross = h_cross != 0;
    if (!st->seg.sums.alloc((size_t)st->seg.total + 8, sizeof(T)) || !st->seg.ticket.alloc(1)) return false;
    if (!alloc_carries(st, tiles * kSegChunks)) return false;  // one carry slot per 256-entry chunk
    st->x_bands = K;
    st->kernel = SPMV_B200_KERNEL_BAND_SEG;
    return true;
}

template <typename T>
static bool build_band_seg(DeviceState *st)
{
    return st->seg.bands <= 32 ? build_band_seg_t<T, uint32_t>(st) : build_band_seg_t<T, unsigned long long>(st);
}

// Mirror of the reference's demotion / promotion rule with the CALLER's nthreads (a10, parallel_balanced2_spmv.c:72-94)
// for clients that read handle->spmvMethod: Method_Balanced2 when some partition of the reference's csrSplitter owns
// no whole row, else Method_Balanced.
static bool apply_reference_balance_rule(DeviceState *st, spmv_Handle *h)
{
    st->split.ref_T = (int)(h->nthreads ? (h->nthreads > (1u << 24) ? (1u << 24) : h->nthreads) : 1);
    int ref_starved = 0;
    if (!build_splitter(st, st->m, st->rowptr, st->split.ref_T, st->split.ref_splitter, &ref_starved)) return false;
    h->spmvMethod = ref_starved ? Method_Balanced2 : Method_Balanced;
    return true;
}

template <typename T>
static bool build_method(DeviceState *st, spmv_Handle *h, int method)
{
    if (st->seg.bands > 1 && method != Method_Serial) {
        if (build_band_seg<T>(st))
            return (method != Method_Balanced && method != Method_Balanced2) || apply_reference_balance_rule(st, h);
        // an optional layout: fall back to the method's own kernel on the plain CSR view
        abandon(st->seg, st->tile);
        st->x_bands = 1;
        st->kernel = SPMV_B200_KERNEL_NONE;
        st->layout_fallbacks++;
    }
    switch (method) {
    case Method_Serial:
        st->kernel = SPMV_B200_KERNEL_CSR_REFORDER;
        return true;
    case Method_Parallel:
        st->tpr = pick_tpr(st);
        st->kernel = SPMV_B200_KERNEL_CSR_VECTOR;
        if (!build_long_rows_threshold(st)) {  // bins / long-row list are speed-ups: plain CSR-vector still works
            abandon(st->lr);
            st->layout_fallbacks++;
        }
        if (!build_pipeline(st)) abandon(st->pipeline);
        return true;
    case Method_Balanced:
    case Method_Balanced2: {
        if (!apply_reference_balance_rule(st, h)) return false;
        // the GPU geometry: row blocks of ~block_nnz non-zeros, one warp each
        const long long block_nnz = st->opts.block_nnz;
        st->split.parts = (int)(((long long)st->nnz + block_nnz - 1) / block_nnz);
        if (st->split.parts < 1) st->split.parts = 1;
        int starved = 0;
        if (!build_splitter(st, st->a_m, st->a_rowptr, st->split.parts, st->split.splitter, &starved)) return false;
        // The reference's rule (parallel_balanced2_spmv.c:87-94), applied to the GPU's own partition: a
        // starved block (some row spans more than a block) => merge-path; otherwise both methods run the
        // row-block kernel ("Balanced2 demoted to Balanced").  Option force_merge=1 keeps merge-path for
        // every Method_Balanced2 handle.
        if (starved || (method == Method_Balanced2 && st->opts.force_merge)) return build_tiles(st, /*merge=*/true);
        st->kernel = SPMV_B200_KERNEL_ROW_BLOCKS;
        return true;
    }
    case Method_Balanced_Yid:
        return build_tiles(st, /*merge=*/false);
    case Method_SellCSigma:
        return build_sell<T>(st);
    case Method_CSR5SPMV:
        return build_csr5<T>(st);
    default:
        st->kernel = SPMV_B200_KERNEL_CSR_REFORDER;
        return true;
    }
}

// "Matrix inspect and choose best method to run" (the empty heading of the reference's README.md:222), inside create:
// option "auto" = 1 lets every create whose Function is not Method_Serial pick the SPMV_METHODS value whose GPU layout
// measured fastest on matrices of that shape (profiles/r02a_bench_c2_n1.json, fraction of the measured HBM peak):
//   * more than a quarter of the non-zeros in rows much longer than the mean (power-law graphs): Method_CSR5SPMV
//     (C3: CSR5 0.390, Parallel 0.326, merge-path 0.270);
//   * short rows (mean <= 8) whose gathers are diagonal-local: Method_Parallel (C1: Parallel 0.605, SELL 0.569);
//   * everything else: Method_SellCSigma (C2: SELL 0.434, Parallel 0.398; C4: SELL 0.981, Parallel 0.883);
//   * fewer than 8192 rows: Method_Parallel (nothing to amortise a layout build).
// The statistics are the ones create gathers on the device anyway (far_fraction of the locality probe) plus one pass
// over RowPtr.  Method_Serial is never overridden: it promises the reference's bits.
// spmv_b200_recommend_method applies the same rule on the host, where the locality share is unknown (far_fraction
// < 0) and short rows alone never pick Method_Parallel.  heavy(cut, &count) counts the non-zeros in rows longer than
// cut; it is called only from 8192 rows on, and a count that fails picks Method_Parallel.
template <typename CountHeavy>
static int pick_method(long long m, long long nnz, double far_fraction, CountHeavy heavy)
{
    if (m < 8192 || nnz <= 0) return Method_Parallel;
    const double mean = (double)nnz / m;
    long long count = 0;
    if (!heavy((int)(4.0 * mean) + 16, &count)) return Method_Parallel;
    if (4 * count > nnz) return Method_CSR5SPMV;
    if (far_fraction >= 0.0 && mean <= 8.0 && far_fraction <= 0.25) return Method_Parallel;
    return Method_SellCSigma;
}

static int auto_pick_method(DeviceState *st)
{
    return pick_method(st->m, st->nnz, st->far_fraction, [&](int cut, long long *count) {
        unsigned long long h_heavy = 0;
        const bool ok = read_counter(st, &h_heavy, [&](unsigned long long *heavy) {
            heavy_rows_kernel<<<blocks_for(st->m), kThreads, 0, st->stream>>>(st->m, cut, st->rowptr, heavy);
        });
        if (!ok) abandon();
        *count = (long long)h_heavy;
        return ok;
    });
}

// reorder_map: the source map of the permuted values under options "reorder" and "refresh" (host, nnz ints)
static bool build_state(DeviceState *st, spmv_Handle *h, int m, int n, int *RowPtr, int *ColIdx, void *Val,
                        int method, const int *reorder_map = nullptr)
{
    st->requested = method;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        set_error("no CUDA device: libspmv_b200 has no CPU fallback");
        return false;
    }
    SB_TRY(cudaGetDevice(&st->device));
    apply_device_limits(st);
    if (m < 0 || n < 0 || (m > 0 && (!RowPtr))) { set_error("invalid arguments (m=%d n=%d RowPtr=%p)", m, n, (void *)RowPtr); return false; }
    st->m = m;
    st->n = n;
    st->vsize = (h->data_size == sizeof(double)) ? 8 : 4;  // reference serial_spmv.c:48-54
    st->requested = method;

    const bool dev_csr = is_device_ptr(RowPtr);
    int ends[2] = {0, 0};
    if (dev_csr) {
        if (m > 0 && !(read_back(st, &ends[0], RowPtr) && read_back(st, &ends[1], RowPtr + m))) return false;
    } else if (m > 0) {
        ends[0] = RowPtr[0];
        ends[1] = RowPtr[m];
    }
    if (ends[0] != 0 || ends[1] < 0) { set_error("RowPtr[0] must be 0 and RowPtr[m] >= 0 (got %d, %d)", ends[0], ends[1]); return false; }
    if ((long long)ends[1] > 2147483647LL - 8192) { set_error("nnz too large for 32-bit tiles"); return false; }
    st->nnz = ends[1];
    if (st->nnz > 0 && (!ColIdx || !Val)) { set_error("ColIdx / Matrix_Val are NULL"); return false; }

    if (dev_csr) {
        // device-resident CSR: adopted in place (borrowed, like the reference borrows host arrays)
        if (st->nnz > 0 && (!is_device_ptr(ColIdx) || !is_device_ptr(Val))) { set_error("RowPtr is a device pointer but ColIdx / Matrix_Val are not"); return false; }
        st->rowptr = RowPtr;
        st->col = ColIdx;
        st->val = Val;
    } else {
        // upload once
        DeviceState::CsrUpload &up = st->upload;
        if (!up.rowptr.alloc((size_t)m + 1 + 8) || !up.col.alloc((size_t)st->nnz + 8) || !up.val.alloc((size_t)st->nnz + 8, st->vsize))
            return false;
        st->rowptr = up.rowptr;
        st->col = up.col;
        st->val = up.val.get();
        if (m > 0) SB_TRY(cudaMemcpy(st->rowptr, RowPtr, ((size_t)m + 1) * sizeof(int), cudaMemcpyHostToDevice));
        else SB_TRY(cudaMemset(st->rowptr, 0, sizeof(int)));
        if (st->nnz > 0) {
            SB_TRY(cudaMemcpy(st->col, ColIdx, (size_t)st->nnz * sizeof(int), cudaMemcpyHostToDevice));
            SB_TRY(cudaMemcpy(st->val, Val, (size_t)st->nnz * st->vsize, cudaMemcpyHostToDevice));
            if (reorder_map && !st->map_failed &&
                !(up.map.alloc((size_t)st->nnz) && SB_CUDA(cudaMemcpy(up.map, reorder_map, (size_t)st->nnz * sizeof(int), cudaMemcpyHostToDevice))))
                map_failure(st);
        }
    }

    st->a_m = st->m; st->a_rowptr = st->rowptr; st->a_col = st->col; st->a_val = st->val;
    // Method_Serial keeps the reference's exact summation order: never banded
    if (method != Method_Serial && m > 0 && st->nnz > 0) {
        if (!probe_locality(st)) return false;
        const std::pair<int, int> bands = decide_bands(m, n, st->nnz, st->vsize, st->dev_l2, st->far_fraction, st->opts);
        st->seg.bands = bands.second;
        if (bands.first > 1) with_precision(st, [&](auto t) { build_band_major<decltype(t)>(st, bands.first); });
    }
    if (m > 0) {
        int e = 0;
        const bool ok = read_counter(st, &e, [&](int *flag) {
            empty_rows_kernel<<<blocks_for(st->a_m), kThreads, 0, st->stream>>>(st->a_m, st->a_rowptr, flag);
        });
        if (!ok) return false;
        st->has_empty_rows = e != 0;
    }
    if (m == 0 || st->nnz == 0) {  // nothing to lay out: spmv() only has zeros to write
        st->kernel = SPMV_B200_KERNEL_NONE;
        return true;
    }
    st->auto_method = -1;
    if (st->opts.auto_pick && method != Method_Serial) {
        method = st->auto_method = auto_pick_method(st);
        if (st->auto_method == Method_SellCSigma || st->auto_method == Method_CSR5SPMV || st->auto_method == Method_Parallel)
            h->spmvMethod = (SPMV_METHODS)st->auto_method;  // what actually runs, for clients that read the field
    }
    if (!with_precision(st, [&](auto t) { return build_method<decltype(t)>(st, h, method); })) return false;
    SB_TRY(cudaStreamSynchronize(st->stream));
    // Our own upload of the CSR is dead weight once every kernel of the handle reads a re-laid-out copy (the
    // band-major copy or the COO bands): give those gigabytes back (an adopted device CSR is the caller's).
    if (st->upload.rowptr && (st->kernel == SPMV_B200_KERNEL_BAND_SEG || st->a_rowptr != st->rowptr)) {
        st->upload = {};
        st->rowptr = st->col = nullptr;
        st->val = nullptr;
        st->released_csr = true;
    }
    if (st->map_failed) {  // a handle that cannot refresh every array it stores keeps none of the maps
        st->refresh = false;
        st->upload.map.reset();
        st->v.map.reset();
        st->sell.map.reset();
        st->c5.map.reset();
        st->seg.map.reset();
    }
    return true;
}

// ------------------------------------------------------------------------------------------------
// launch dispatch (a3: the reference's spmv_functions[] table, common.c:85-94)
// ------------------------------------------------------------------------------------------------
// the extra y destinations of spmv_b200_set_y_peers (fused all-gather); PeerList<T>{} is "none"
template <typename T>
static PeerList<T> peers_of(const DeviceState *st)
{
    PeerList<T> peers;
    peers.n = st->n_peers;
    for (int i = 0; i < kMaxPeers; ++i) peers.p[i] = (T *)st->peers[i];
    return peers;
}

// CSR-vector over rows [row0, row1) of the active view; fuse_bands > 0: they belong to the last band and y is the
// FINAL y
template <typename T>
static void launch_vector(DeviceState *st, int row0, int row1, const T *x, T *y, const PeerList<T> &peers, int fuse_bands = 0)
{
    const int grid = blocks_for((long long)(row1 - row0) * st->tpr);
    if (grid <= 0) return;
    const auto kernel = with_value<1, 2, 4, 8, 16, 32>(st->tpr, [&](auto N) {
        return fuse_bands > 0 ? csr_vector_kernel<T, N, false, true> : peers.n > 0 ? csr_vector_kernel<T, N, true, false> : csr_vector_kernel<T, N, false, false>;
    });
    kernel<<<grid, kThreads, 0, st->stream>>>(row0, row1, st->lr.thr, st->a_rowptr, st->a_col, (const T *)st->a_val, x, y, peers, fuse_bands, st->m, st->v.y.as<T>());
    count_launch();
}

// The final store of spmv_b200_spmv_axpby, spmv_b200_spmv_axpby_dot and spmv_b200_spmv_shifted on the host side: the
// scaling, for the dot w and the partials array, filled launch after launch (DotStore), and for the shifted store its
// shift and x (ShiftStore: x . y partials in `partials`, y . y partials in `yy`, both NULL without dots)
template <typename T>
struct Scaled {
    ScaledStore<T> sc;
    const T *w;              // dot: NULL = w is the new y
    double *partials;        // NULL: no dot (spmv_b200_spmv_axpby)
    int parts;               // partials written so far
    bool shifted = false;
    T sigma = 0;
    const T *x = nullptr;
    double *yy = nullptr;
    // the arguments of the next dot launch, of `grid` CTAs
    DotArgs<T> next(int grid)
    {
        const DotArgs<T> d{sc, w, partials + parts};
        parts += grid;
        return d;
    }
    // the arguments of the next shifted launch, of `grid` CTAs
    ShiftArgs<T> next_shift(int grid)
    {
        const ShiftArgs<T> d{sc, sigma, x, partials ? partials + parts : nullptr, partials ? yy + parts : nullptr};
        if (partials) parts += grid;
        return d;
    }
};

// y_out = the band partials of the virtual y (v.y) added in band order, copied to the peers too; scaled: y_out <- alpha
// (that sum) + beta y_out instead (and the dot, or the shift), and no peers
template <typename T>
static bool launch_band_fold(DeviceState *st, T *y_out, Scaled<T> *scaled = nullptr)
{
    const int grid = blocks_for(st->m);
    if (scaled && scaled->shifted) {
        band_reduce_shift_kernel<T><<<grid, kThreads, 0, st->stream>>>(0, st->m, st->m, st->x_bands, st->v.y.as<T>(), scaled->next_shift(grid));
    } else if (scaled && scaled->partials) {
        band_reduce_axpby_dot_kernel<T><<<grid, kThreads, 0, st->stream>>>(0, st->m, st->m, st->x_bands, st->v.y.as<T>(), scaled->next(grid));
    } else if (scaled) {
        band_reduce_axpby_kernel<T><<<grid, kThreads, 0, st->stream>>>(0, st->m, st->m, st->x_bands, st->v.y.as<T>(), scaled->sc);
    } else {
        const PeerList<T> peers = peers_of<T>(st);
        const auto kernel = peers.n > 0 ? band_reduce_kernel<T, true> : band_reduce_kernel<T, false>;
        kernel<<<grid, kThreads, 0, st->stream>>>(0, st->m, st->m, st->x_bands, st->v.y.as<T>(), y_out, peers);
    }
    count_launch();
    return SB_CUDA(cudaGetLastError());
}

// CSR-vector over rows [row0, m) only (the CSR tail of SELL)
template <typename T, typename Store>
__device__ __forceinline__ void csr_tail_body(unsigned tid, int row0, int m, int long_thr, const int *__restrict__ rowptr,
                                              const int *__restrict__ col, const T *__restrict__ val,
                                              const T *__restrict__ x, const Store &store)
{
    const uint64_t pl = policy_evict_last();
    const long long w = ((long long)blockIdx.x * kThreads + tid) >> 5;
    const int lane = tid & 31;
    if (row0 + w >= m) return;
    const int row = (int)(row0 + w);
    const int start = rowptr[row];
    int end = rowptr[row + 1];
    if (end - start > long_thr) end = start;  // hub row: y = 0 here, the long-row path adds the whole row
    const auto early = store.early(lane == 0, row);
    T sum = 0;
    for (int j = start + lane; j < end; j += 32) sum = fma_t(val[j], ldg_x(x + col[j], pl), sum);
    sum = group_sum_c<T, 32>(sum);
    if (lane == 0) store.put(row, sum, early);
}

// csr_tail_kernel's store: a plain one (the tail rows are few; spmv() writes them through L1 as it always has)
template <typename T>
struct TailStore {
    T *y;
    __device__ __forceinline__ NoEarly early(bool, long long) const { return {}; }
    __device__ __forceinline__ void put(long long row, T v, NoEarly) const { y[row] = v; }
};

template <typename T>
__global__ void __launch_bounds__(kThreads)
csr_tail_kernel(int row0, int m, int long_thr, const int *__restrict__ rowptr, const int *__restrict__ col,
                const T *__restrict__ val, const T *__restrict__ x, T *__restrict__ y)
{
    csr_tail_body<T>(threadIdx.x, row0, m, long_thr, rowptr, col, val, x, TailStore<T>{y});
}

template <typename T>
__global__ void __launch_bounds__(kThreads)
csr_tail_axpby_kernel(int row0, int m, int long_thr, const int *__restrict__ rowptr, const int *__restrict__ col,
                      const T *__restrict__ val, const T *__restrict__ x, const ScaledStore<T> store)
{
    csr_tail_body<T>(threadIdx.x, row0, m, long_thr, rowptr, col, val, x, store);
}

template <typename T>
__global__ void __launch_bounds__(kThreads)
csr_tail_axpby_dot_kernel(int row0, int m, int long_thr, const int *__restrict__ rowptr, const int *__restrict__ col,
                          const T *__restrict__ val, const T *__restrict__ x, const DotArgs<T> d)
{
    double acc = 0;
    csr_tail_body<T>(threadIdx.x, row0, m, long_thr, rowptr, col, val, x, DotStore<T>{d, acc});
    dot_partial(acc, d.partials);
}

template <typename T>
__global__ void __launch_bounds__(kThreads)
csr_tail_shift_kernel(int row0, int m, int long_thr, const int *__restrict__ rowptr, const int *__restrict__ col,
                      const T *__restrict__ val, const T *__restrict__ x, const ShiftArgs<T> d)
{
    double xy = 0, yy = 0;
    csr_tail_body<T>(threadIdx.x, row0, m, long_thr, rowptr, col, val, x, ShiftStore<T>{d, xy, yy});
    shift_partials(xy, yy, d.xy, d.yy);
}

static int opt_cached_seg_prefetch()
{
    static const int v = (int)opt("seg_prefetch");  // read once: spmv() is the hot path
    return v;
}

// band segments, pass 1 over the tiles of bands [b0, b0 + count)
template <typename T>
static bool launch_seg_bands(DeviceState *st, int b0, int count, const T *x)
{
    const int t0 = st->seg.tile0[b0], t1 = st->seg.tile0[b0 + count];
    if (t1 <= t0) return true;
    // persistent CTAs: option seg_ctas per SM (shared memory AND registers allow 2 or 3), read at the first launch
    if (st->seg.grid == 0) st->seg.ctas = (int)opt("seg_ctas") == 3 ? 3 : 2;
    const auto kernel = st->seg.ctas == 3 ? bseg_kernel<T, 3> : bseg_kernel<T, 2>;
    if (st->seg.grid == 0) {
        SB_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bseg_smem_bytes<T>()));
        // leave the rest of the unified array to L1: the gathers need lines for their outstanding misses
        const int carve = (int)((st->seg.ctas * (bseg_smem_bytes<T>() + 2048) * 100 + 228 * 1024 - 1) / (228 * 1024));
        SB_TRY(cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, carve > 100 ? 100 : carve));
        st->seg.grid = st->seg.ctas * (st->dev_sms > 0 ? st->dev_sms : 1);
    }
    const int grid = t1 - t0 < st->seg.grid ? t1 - t0 : st->seg.grid;
    // ticket counter of the dynamic tile schedule: tickets 0 .. 3*grid-1 are implicit (every CTA's first three tiles)
    set_int_kernel<<<1, 1, 0, st->stream>>>(st->seg.ticket, kSegStages * grid);
    // L2 prefetch of the next band's x slice pays only when two slices fit the part of L2 random gathers can use
    // (measured on the C5 shard: 64 MiB slices 5.78 -> 6.13 ms with it, 32 MiB slices 5.81 -> 5.76 ms and DRAM reads
    // 14.0 -> 9.9 GB); option seg_prefetch: 0 = never, 1 = automatic, 2 = always
    const int pf_opt = opt_cached_seg_prefetch();
    const bool two_fit = 2.0 * (double)st->band_cols * st->vsize <= 0.53 * (double)st->dev_l2;
    const int pf_on = (((uintptr_t)x & 15u) == 0 && (pf_opt == 2 || (pf_opt == 1 && two_fit))) ? 1 : 0;
    kernel<<<grid, kSegThreads, bseg_smem_bytes<T>(), st->stream>>>(t0, t1, pf_on, st->seg.ticket, st->seg.tile_ent, st->seg.tile_seg0, st->seg.col,
        st->seg.ent_val.as<T>(), x, st->seg.sums.as<T>(), st->tile.carry_val.as<T>(), st->tile.carry_row);
    count_launch();
    return SB_CUDA(cudaGetLastError());
}

// band segments: carries of segments that cross a tile boundary, then pass 2 (y written once, peers included; scaled:
// y_out <- alpha (the row sums) + beta y_out, and no peers)
template <typename T>
static bool launch_seg_finish(DeviceState *st, T *y_out, Scaled<T> *scaled = nullptr)
{
    cudaStream_t s = st->stream;
    if (st->seg.cross) launch_carry_fixup<T>(st, s, st->tile.count * kSegChunks, st->tile.carry_row, st->tile.carry_val.as<T>(), st->seg.sums.as<T>());
    const PeerList<T> pr = peers_of<T>(st);
    auto merge = [&](auto mask_word) {  // row masks of 32 or 64 bands
        using M = decltype(mask_word);
        const int grid = blocks_for((long long)st->seg.groups * 32);
        if (scaled) {  // (never with the dot or the shift: dot_path)
            bseg_merge_axpby_kernel<T, M><<<grid, kThreads, 0, s>>>(0, st->m, st->seg.bands, st->seg.mask.as<M>(), st->seg.gbase, st->seg.sums.as<T>(), scaled->sc);
            return;
        }
        const auto kernel = pr.n > 0 ? bseg_merge_kernel<T, M, true> : bseg_merge_kernel<T, M, false>;
        kernel<<<grid, kThreads, 0, s>>>(0, st->m, st->seg.bands, st->seg.mask.as<M>(), st->seg.gbase, st->seg.sums.as<T>(), y_out, pr);
    };
    if (st->seg.mask64) merge((unsigned long long)0); else merge(uint32_t(0));
    count_launch();
    return SB_CUDA(cudaGetLastError());
}

// y_out = A x.  fold_scaled (spmv_b200_spmv_axpby on a band-major or band-segment handle, _dot on a band-major one): the
// last pass, the fold of the band partials, writes y_out <- alpha A x + beta y_out instead (and the dot's partials).
template <typename T>
static bool launch(DeviceState *st, const T *x, T *y_out, Scaled<T> *fold_scaled = nullptr)
{
    cudaStream_t s = st->stream;
    if (st->m == 0) return true;
    if (st->kernel == SPMV_B200_KERNEL_NONE) {  // nnz == 0: y = 0
        return SB_CUDA(cudaMemsetAsync(y_out, 0, (size_t)st->m * sizeof(T), s));  // all-zero bits = +0.0
    }
    if (st->kernel == SPMV_B200_KERNEL_BAND_SEG) {
        // pass 1: segment sums of every tile (one launch, tiles in band order); carries of segments that cross a
        // tile boundary; pass 2: every row adds its segment sums in band order and writes y once
        return launch_seg_bands<T>(st, 0, st->seg.bands, x) && launch_seg_finish<T>(st, y_out, fold_scaled);
    }
    // the active view: the CSR itself, or its band-major copy writing the virtual y
    const int m = st->a_m;
    const bool banded = st->x_bands > 1;
    T *y = banded ? st->v.y.as<T>() : y_out;
    const T *val = (const T *)st->a_val;
    // extra y destinations (fused all-gather), written with the final y: by the band fold when banded, else here
    const PeerList<T> fused = banded ? PeerList<T>{} : peers_of<T>(st);
    bool wrote_fused = false;  // the case's kernels (and the long-row pass) wrote every final value to `fused` too
    switch (st->kernel) {
    case SPMV_B200_KERNEL_CSR_REFORDER: {
        constexpr int L = sizeof(T) == 8 ? 4 : 8;
        csr_reforder_kernel<T><<<blocks_for((long long)m * L), kThreads, 0, s>>>(m, st->a_rowptr, st->a_col, val, x, y);
        count_launch();
        break;
    }
    case SPMV_B200_KERNEL_CSR_VECTOR:
        // (one launch over all bands + band_reduce measured faster than two launches with the reduce fused into
        // the last band: 2.59 vs 2.64 ms on C2; the fused form is used by the pipelined host path, where the
        // last band runs in row chunks anyway)
        if (st->lr.binned) {
            static const int lanes[3] = {1, 4, 16};
            for (int b = 0; b < 3; ++b) {
                const int count = st->lr.bin_ptr[b + 1] - st->lr.bin_ptr[b];
                if (count <= 0) continue;
                const auto kernel = with_value<1, 4, 16>(lanes[b], [&](auto N) {
                    return fused.n > 0 ? csr_vector_list_kernel<T, N, true> : csr_vector_list_kernel<T, N, false>;
                });
                kernel<<<blocks_for((long long)count * lanes[b]), kThreads, 0, s>>>(count, st->lr.bin_list + st->lr.bin_ptr[b], st->a_rowptr, st->a_col, val, x, y, fused);
                count_launch();
            }
        } else {
            launch_vector<T>(st, 0, m, x, y, fused);
        }
        wrote_fused = true;
        break;
    case SPMV_B200_KERNEL_ROW_BLOCKS: {
        const auto kernel = fused.n > 0 ? row_block_kernel<T, true> : row_block_kernel<T, false>;
        kernel<<<blocks_for((long long)st->split.parts * 32), kThreads, 0, s>>>(st->split.parts, st->split.splitter, st->a_rowptr, st->a_col, val, x, y, fused);
        wrote_fused = true;
        count_launch();
        break;
    }
    case SPMV_B200_KERNEL_MERGE_PATH: {
        const auto kernel = st->tile.items == 4 ? merge_path_kernel<T, 4> : merge_path_kernel<T, 8>;
        kernel<<<st->tile.count, kThreads, 0, s>>>(m, st->nnz, st->tile.merge_coords, st->a_rowptr, st->a_col, val, x, y, st->tile.carry_val.as<T>(), st->tile.carry_row);
        launch_carry_fixup<T>(st, s, st->tile.count, st->tile.carry_row, st->tile.carry_val.as<T>(), y);
        count_launch();
        break;
    }
    case SPMV_B200_KERNEL_NNZ_SPLIT: {
        const auto kernel = st->tile.items == 4 ? nnz_split_kernel<T, 4> : nnz_split_kernel<T, 8>;
        kernel<<<st->tile.count, kThreads, 0, s>>>(m, st->nnz, st->tile.rows, st->a_rowptr, st->a_col, val, x, y, st->tile.carry_val.as<T>(), st->tile.carry_row);
        launch_carry_fixup<T>(st, s, st->tile.count, st->tile.carry_row, st->tile.carry_val.as<T>(), y);
        count_launch();
        break;
    }
    case SPMV_B200_KERNEL_SELL: {
        if (st->sell.slices > 0) {
            wrote_fused = st->sell.banner == m;  // no CSR tail: the SELL kernel writes every final value
            const PeerList<T> sp = wrote_fused ? fused : PeerList<T>{};
            const auto kernel = sp.n > 0 ? sell_kernel<T, true, 8, 6> : st->sell.variant == 2 ? sell_kernel<T, false, 4, 8> : sell_kernel<T, false, 8, 6>;
            kernel<<<blocks_for((long long)st->sell.slices * 32), kThreads, 0, s>>>(
                st->sell.slices, st->sell.slice_ptr, st->sell.full, st->sell.perm, st->sell.col, st->sell.val.as<T>(), x, y, sp);
            count_launch();
        }
        if (st->sell.banner < m) {
            csr_tail_kernel<T><<<blocks_for((long long)(m - st->sell.banner) * 32), kThreads, 0, s>>>(st->sell.banner, m, st->lr.thr, st->a_rowptr, st->a_col, val, x, y);
            count_launch();
        }
        break;
    }
    case SPMV_B200_KERNEL_CSR5: {
        const int p = st->c5.p;
        if (st->has_empty_rows) {
            if (!SB_CUDA(cudaMemsetAsync(y, 0, (size_t)m * sizeof(T), s))) return false;  // all-zero bits = +0.0
        }
        const T *tval = st->c5.val.as<T>();
        if (p > 1) {
            const auto kernel = with_value<4, 8, 16>(st->c5.sigma, [](auto SG) { return csr5_kernel<T, SG>; });
            kernel<<<blocks_for((long long)(p - 1) * 32), kThreads, 0, s>>>(
                p, st->c5.bit_y, st->c5.bit_ss, st->c5.tile_ptr, st->c5.tile_desc, st->c5.off_ptr, st->c5.off, st->c5.col, tval, x, y, st->tile.carry_val.as<T>(), st->tile.carry_row);
            count_launch();
        }
        const int tail_nz0 = (p - 1) * kC5Omega * st->c5.sigma;
        csr5_tail_kernel<T><<<blocks_for((long long)(m - st->c5.tail_start) * 32), kThreads, 0, s>>>(
            m, st->c5.tail_start, tail_nz0, p - 1, st->a_rowptr, st->c5.col, tval, x, y, st->tile.carry_val.as<T>(), st->tile.carry_row);
        launch_carry_fixup<T>(st, s, p, st->tile.carry_row, st->tile.carry_val.as<T>(), y);
        count_launch();
        break;
    }
    default:
        set_error("handle has no kernel (%d)", st->kernel);
        return false;
    }
    if (st->lr.rows > 0) {  // hub rows / SELL overflow: segment sums, then one ordered add per row
        const int single = fused.n == 0;  // with peer destinations every final value goes through long_final_kernel
        long_seg_kernel<T><<<blocks_for((long long)st->lr.segs * 32), kThreads, 0, s>>>(
            st->lr.segs, st->lr.seg_row, st->lr.row, st->lr.start, st->lr.seg_ptr, st->a_rowptr, st->a_col, val, x, st->lr.partial.as<T>(),
            y, single, st->lr.accumulate);
        const auto final_kernel = fused.n > 0 ? long_final_kernel<T, true> : long_final_kernel<T, false>;
        final_kernel<<<blocks_for((long long)st->lr.rows * 32), kThreads, 0, s>>>(st->lr.rows, st->lr.accumulate, single, st->lr.row, st->lr.seg_ptr, st->lr.partial.as<T>(), y, fused);
        count_launch(2);
    }
    if (banded) return launch_band_fold<T>(st, y_out, fold_scaled);  // y and the peers
    if (fused.n > 0 && !wrote_fused) {  // kernels without a fused epilogue: one stream-ordered copy to the peers
        peer_copy_kernel<T><<<blocks_for(st->m), kThreads, 0, s>>>(st->m, y_out, fused);
        count_launch();
    }
    return SB_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------
// y <- alpha A x + beta y (spmv_b200_spmv_axpby).  A x is summed by spmv()'s own kernels, bit for bit, and scaled where
// its final value is stored: in the fold of the band partials (band-major copy, band segments), in the main kernel
// (CSR-vector, row blocks, SELL and its CSR tail), or -- where the final value comes out of a carry fix-up (merge-path,
// nnz-split, CSR5), of the long-row pass, of the row bins' several launches, or of the reference-order kernel -- in a
// pass of its own over A x written to a scratch array.
// ------------------------------------------------------------------------------------------------
enum { kAxpbyScratch = 0, kAxpbyMain = 1, kAxpbyFold = 2 };  // spmv_b200_info "axpby_path"

// Whether spmv() runs SELL's 8-column flavour (variant 0, or any variant with peers and no CSR tail).  The step width
// orders the sums, so a scaled SELL kernel must step as spmv() does.  The 4-column flavour (variant 2) fits 32
// registers, which is why it exists (every warp slot of the SM filled); its scaled twin does not (fp64: 100 bytes of
// spills at 32 registers, against sell_kernel's own 76), so variant-2 handles take the scratch pass.
static bool sell_eight_columns(const DeviceState *st)
{
    return st->sell.variant != 2 || (st->n_peers > 0 && st->sell.banner == st->m);
}

static int axpby_path(const DeviceState *st)
{
    if (!st->opts.axpby_fused) return kAxpbyScratch;  // option "axpby_fused" = 0
    if (st->kernel == SPMV_B200_KERNEL_BAND_SEG) return kAxpbyFold;
    if (st->x_bands > 1) return kAxpbyFold;  // (never Method_Serial: it is not banded)
    if (st->lr.rows > 0) return kAxpbyScratch;
    // one lane per row only: at 2..32 lanes the scaled CSR-vector kernel needs 48 registers against spmv()'s 40 and
    // lost to the scratch pass on C4 (tpr 4: 1.121 against 1.086 ms), as a scaled row-block kernel did (46 registers
    // against 40, 1.387 against 1.249 ms; profiles/r04a_axpby_all_fused.json, the run before both were dropped)
    if (st->kernel == SPMV_B200_KERNEL_CSR_VECTOR) return st->lr.binned || st->tpr != 1 ? kAxpbyScratch : kAxpbyMain;
    if (st->kernel == SPMV_B200_KERNEL_SELL) return sell_eight_columns(st) ? kAxpbyMain : kAxpbyScratch;
    return kAxpbyScratch;  // also nnz == 0: s = +0
}

// spmv_b200_info "dot_path": where spmv_b200_spmv_axpby_dot scales and takes its products.  spmv_b200_spmv_axpby's
// kernel, except on band segments: their pass-2 dot twin needed 40 registers against the scaled kernel's 32 and lost to
// the scratch pass on the C5 shard (5.568 against 5.063 ms per call on one B200 at 1000 W, in the run before it was
// dropped).  The other twins beat their scratch pass (profiles/r05_axpby_dot.json: C1 0.0291 against 0.0333 ms, C2
// 2.645 against 2.696 ms).
static int dot_path(const DeviceState *st)
{
    return st->kernel == SPMV_B200_KERNEL_BAND_SEG ? kAxpbyScratch : axpby_path(st);
}

// Partials of one dot: one per CTA of its dot launches, at most -- one CTA per 256 rows (the scratch pass, alpha == 0,
// the CSR-vector kernel, the band-major fold), plus the slices and the CSR tail of an unbanded SELL handle
static long long dot_partials_bound(const DeviceState *st)
{
    long long p = blocks_for(st->m);
    if (st->kernel == SPMV_B200_KERNEL_SELL && st->x_bands == 1)
        p += blocks_for((long long)st->sell.slices * 32) + blocks_for((long long)(st->m - st->sell.banner) * 32);
    return p;
}

// the main-kernel path: the scaled (dot, shifted) twins of the kernels launch() runs on an unbanded view without long-row
// list
template <typename T>
static void launch_main_axpby(DeviceState *st, const T *x, Scaled<T> &sc)
{
    cudaStream_t s = st->stream;
    const int m = st->m;
    const T *val = (const T *)st->a_val;
    switch (st->kernel) {
    case SPMV_B200_KERNEL_CSR_VECTOR: {
        const int grid = blocks_for((long long)m * st->tpr);
        if (sc.shifted) csr_vector_shift_kernel<T, 1><<<grid, kThreads, 0, s>>>(0, m, st->lr.thr, st->a_rowptr, st->a_col, val, x, sc.next_shift(grid));
        else if (sc.partials) csr_vector_axpby_dot_kernel<T, 1><<<grid, kThreads, 0, s>>>(0, m, st->lr.thr, st->a_rowptr, st->a_col, val, x, sc.next(grid));
        else csr_vector_axpby_kernel<T, 1><<<grid, kThreads, 0, s>>>(0, m, st->lr.thr, st->a_rowptr, st->a_col, val, x, sc.sc);
        count_launch();
        break;
    }
    case SPMV_B200_KERNEL_SELL:
        if (st->sell.slices > 0) {  // (the 8-column flavour: sell_eight_columns)
            const int grid = blocks_for((long long)st->sell.slices * 32);
            if (sc.shifted) {
                sell_shift_kernel<T, 8, 6><<<grid, kThreads, 0, s>>>(
                    st->sell.slices, st->sell.slice_ptr, st->sell.full, st->sell.perm, st->sell.col, st->sell.val.as<T>(), x, sc.next_shift(grid));
            } else if (sc.partials) {
                sell_axpby_dot_kernel<T, 8, 6><<<grid, kThreads, 0, s>>>(
                    st->sell.slices, st->sell.slice_ptr, st->sell.full, st->sell.perm, st->sell.col, st->sell.val.as<T>(), x, sc.next(grid));
            } else {
                sell_axpby_kernel<T, 8, 6><<<grid, kThreads, 0, s>>>(
                    st->sell.slices, st->sell.slice_ptr, st->sell.full, st->sell.perm, st->sell.col, st->sell.val.as<T>(), x, sc.sc);
            }
            count_launch();
        }
        if (st->sell.banner < m) {
            const int grid = blocks_for((long long)(m - st->sell.banner) * 32);
            if (sc.shifted) csr_tail_shift_kernel<T><<<grid, kThreads, 0, s>>>(st->sell.banner, m, st->lr.thr, st->a_rowptr, st->a_col, val, x, sc.next_shift(grid));
            else if (sc.partials) csr_tail_axpby_dot_kernel<T><<<grid, kThreads, 0, s>>>(st->sell.banner, m, st->lr.thr, st->a_rowptr, st->a_col, val, x, sc.next(grid));
            else csr_tail_axpby_kernel<T><<<grid, kThreads, 0, s>>>(st->sell.banner, m, st->lr.thr, st->a_rowptr, st->a_col, val, x, sc.sc);
            count_launch();
        }
        break;
    }
}

// y <- alpha s + beta y over s = A x in the scratch array; s = NULL: alpha == 0
template <typename T>
static void launch_scratch_pass(DeviceState *st, const T *s, Scaled<T> &sc)
{
    const int grid = blocks_for(st->m);
    if (sc.shifted) shift_kernel<T><<<grid, kThreads, 0, st->stream>>>(st->m, s, sc.next_shift(grid));
    else if (sc.partials) axpby_dot_kernel<T><<<grid, kThreads, 0, st->stream>>>(st->m, s, sc.next(grid));
    else axpby_kernel<T><<<grid, kThreads, 0, st->stream>>>(st->m, s, sc.sc);
    count_launch();
}

// y <- alpha A x + beta y into sc.sc.y, and the dot's partials when sc.partials is set
template <typename T>
static bool launch_axpby(DeviceState *st, const T *x, Scaled<T> &sc)
{
    cudaStream_t s = st->stream;
    const int m = st->m;
    T *y = sc.sc.y;
    if (m == 0) return true;
    if (sc.sc.alpha == (T)0) {  // A and x are not read
        if (sc.sc.beta == (T)0 && !sc.partials) {
            if (!SB_CUDA(cudaMemsetAsync(y, 0, (size_t)m * sizeof(T), s))) return false;  // all-zero bits = +0.0
        } else {
            launch_scratch_pass<T>(st, (const T *)nullptr, sc);
        }
    } else {
        switch (sc.partials || sc.shifted ? dot_path(st) : axpby_path(st)) {
        case kAxpbyFold:
            if (!launch<T>(st, x, y, &sc)) return false;
            break;
        case kAxpbyMain:
            launch_main_axpby<T>(st, x, sc);
            break;
        default: {
            if (!st->stage.s.get() && !st->stage.s.alloc((size_t)m, st->vsize)) return false;
            // exactly spmv()'s launches, peers included (with peers SELL runs another flavour, whose sums differ): the
            // peers then hold A x until the copy below overwrites it with the scaled values
            if (!launch<T>(st, x, st->stage.s.as<T>())) return false;
            launch_scratch_pass<T>(st, st->stage.s.as<T>(), sc);
        }
        }
    }
    if (st->n_peers > 0) {  // the scaled kernels have no peer variants: one stream-ordered copy
        peer_copy_kernel<T><<<blocks_for(m), kThreads, 0, s>>>(m, y, peers_of<T>(st));
        count_launch();
    }
    return SB_CUDA(cudaGetLastError());
}

// launch_axpby with the dot, then *dot (a device double) = the sum of its partials; shifted: dot[0] and dot[1] = the
// sums of the x . y and the y . y partials, each in the finish kernel's one order
template <typename T>
static bool launch_axpby_dot(DeviceState *st, const T *x, Scaled<T> &sc, double *dot)
{
    if (!launch_axpby<T>(st, x, sc)) return false;
    dot_finish_kernel<<<1, kDotFinishThreads, 0, st->stream>>>(sc.parts, sc.partials, dot);
    if (sc.shifted) dot_finish_kernel<<<1, kDotFinishThreads, 0, st->stream>>>(sc.parts, sc.yy, dot + 1);
    count_launch(sc.shifted ? 2 : 1);
    return SB_CUDA(cudaGetLastError());
}

// ------------------------------------------------------------------------------------------------
// Host x and host y through the CSR-vector kernel, pipelined over PCIe: x goes up in pieces on s_in, the
// compute stream starts every band / row chunk as soon as the part of x it gathers from has arrived, and
// finished chunks of y go back on s_out while later chunks are still being computed.  Same kernels, same
// per-row arithmetic as the one-shot path: the bits of y do not depend on which path ran.
// ------------------------------------------------------------------------------------------------
template <typename T>
static bool run_pipelined(DeviceState *st, const T *hx, T *hy)
{
    if (!st->s_in) {
        SB_TRY(cudaStreamCreateWithFlags(&st->s_in, cudaStreamNonBlocking));
        SB_TRY(cudaStreamCreateWithFlags(&st->s_out, cudaStreamNonBlocking));
        for (int i = 0; i < kMaxPieces; ++i) SB_TRY(cudaEventCreateWithFlags(&st->ev_in[i], cudaEventDisableTiming));
        for (int i = 0; i < kPipeChunks; ++i) SB_TRY(cudaEventCreateWithFlags(&st->ev_out[i], cudaEventDisableTiming));
        SB_TRY(cudaEventCreateWithFlags(&st->ev_start, cudaEventDisableTiming));
    }
    cudaStream_t s = st->stream;
    T *xd = st->stage.x.as<T>(), *yd = st->stage.y.as<T>();
    const int m = st->m, n = st->n;
    const bool banded = st->x_bands > 1;
    const int pieces = banded ? st->x_bands : kPipeChunks;
    const PeerList<T> none{};
    // whatever the caller queued on the compute stream before this call stays ahead of the copies
    SB_TRY(cudaEventRecord(st->ev_start, s));
    SB_TRY(cudaStreamWaitEvent(st->s_in, st->ev_start, 0));
    SB_TRY(cudaStreamWaitEvent(st->s_out, st->ev_start, 0));
    auto piece = [&](int p) -> std::pair<long long, long long> {  // columns [lo, hi) of x in piece p
        if (banded) return band_columns(st, p, pieces);
        return {(long long)n * p / pieces, p == pieces - 1 ? n : (long long)n * (p + 1) / pieces};
    };
    for (int p = 0; p < pieces; ++p) {
        const auto [lo, hi] = piece(p);
        if (hi > lo) SB_TRY(cudaMemcpyAsync(xd + lo, hx + lo, (size_t)(hi - lo) * sizeof(T), cudaMemcpyHostToDevice, st->s_in));
        SB_TRY(cudaEventRecord(st->ev_in[p], st->s_in));
    }
    int waited = -1;
    auto need_piece = [&](int p) -> bool {
        for (; waited < p; ++waited) SB_TRY(cudaStreamWaitEvent(s, st->ev_in[waited + 1], 0));
        return true;
    };
    auto chunk_out = [&](int c, int r0, int r1) -> bool {
        SB_TRY(cudaEventRecord(st->ev_out[c], s));
        SB_TRY(cudaStreamWaitEvent(st->s_out, st->ev_out[c], 0));
        if (r1 > r0) SB_TRY(cudaMemcpyAsync(hy + r0, yd + r0, (size_t)(r1 - r0) * sizeof(T), cudaMemcpyDeviceToHost, st->s_out));
        return true;
    };
    if (banded) {
        const int K = st->x_bands;
        for (int b = 0; b + 1 < K; ++b) {
            if (!need_piece(b)) return false;
            launch_vector<T>(st, b * m, (b + 1) * m, xd, st->v.y.as<T>(), none);
        }
        if (!need_piece(K - 1)) return false;
        for (int c = 0; c < kPipeChunks; ++c) {
            const int r0 = (int)((long long)m * c / kPipeChunks), r1 = (int)((long long)m * (c + 1) / kPipeChunks);
            launch_vector<T>(st, (K - 1) * m + r0, (K - 1) * m + r1, xd, yd, none, K - 1);
            if (!chunk_out(c, r0, r1)) return false;
        }
    } else {
        for (int c = 0; c < kPipeChunks; ++c) {
            const int r0 = (int)((long long)m * c / kPipeChunks), r1 = (int)((long long)m * (c + 1) / kPipeChunks);
            int p = 0;
            while (p < pieces - 1 && piece(p).second < st->chunk_xmax[c]) ++p;
            if (!need_piece(p)) return false;
            launch_vector<T>(st, r0, r1, xd, yd, none);
            if (!chunk_out(c, r0, r1)) return false;
        }
    }
    SB_TRY(cudaGetLastError());
    SB_TRY(cudaStreamSynchronize(st->s_out));  // every chunk of y is home (and so every kernel has run)
    SB_TRY(cudaStreamSynchronize(st->s_in));   // x may be modified by the caller from here on
    return true;
}

static DeviceState *state_of(const spmv_Handle *h)
{
    if (!h || !h->extraHandle) return nullptr;
    DeviceState *st = (DeviceState *)h->extraHandle;
    return st->magic == 0x5b200a11u ? st : nullptr;
}

static void handle_init(spmv_Handle *h)  // reference gemv_Handle_init, common.c:18-29
{
    h->spmvMethod = Method_Serial;
    h->nthreads = 0;
    h->extraHandle = nullptr;
    h->RowPtr = nullptr;
    h->ColIdx = nullptr;
    h->Matrix_Val = nullptr;
    h->Y_temp = nullptr;
    h->index = nullptr;
    h->Level_3_opt_used = 0;
}

}  // namespace sb

using namespace sb;

// ================================================================================================
// exported data (reference common.c:306-339; same strings, same order)
// ================================================================================================
extern "C" {

const char *funcNames[] = {
    "Method_Serial_VECTOR_NONE", "Method_Serial_VECTOR_AVX2", "Method_Serial_VECTOR_AVX512",
    "Method_Parallel_VECTOR_NONE", "Method_Parallel_VECTOR_AVX2", "Method_Parallel_VECTOR_AVX512",
    "Method_Balanced_VECTOR_NONE", "Method_Balanced_VECTOR_AVX2", "Method_Balanced_VECTOR_AVX512",
    "Method_Balanced2_VECTOR_NONE", "Method_Balanced2_VECTOR_AVX2", "Method_Balanced2_VECTOR_AVX512",
    "Method_SellCSigma_VECTOR_NONE", "Method_SellCSigma_VECTOR_AVX2", "Method_SellCSigma_VECTOR_AVX512",
    "Method_Csr5Spmv_VECTOR_NONE", "Method_Csr5Spmv_VECTOR_AVX2", "Method_Csr5Spmv_VECTOR_AVX512"};
const char *Methods_names[] = {"Method_Serial", "Method_Parallel", "Method_Balanced", "Method_Balanced2",
                               "Method_BalancedYid", "Method_SellCSigma", "Method_Csr5Spmv"};
const char *Vectorized_names[] = {"VECTOR_NONE", "VECTOR_AVX2", "VECTOR_AVX512"};

// ================================================================================================
// the four drop-in entry points
// ================================================================================================
// everything create does to an initialised public struct (shared by create and spmv_b200_update_values)
static void create_into(spmv_Handle *h, BASIC_INT_TYPE m, BASIC_INT_TYPE n, BASIC_INT_TYPE *RowPtr, BASIC_INT_TYPE *ColIdx,
                        void *Matrix_Val, BASIC_SIZE_TYPE nthreads, int method, BASIC_SIZE_TYPE size, VECTORIZED_WAY vectorizedWay)
{
    if (method < (int)Method_Serial || method >= (int)Method_Total_Size) method = Method_Serial;  // common.c:136
    h->nthreads = nthreads;  // handle_init_common_parameters, common.c:74-83
    h->vectorizedWay = vectorizedWay;
    h->data_size = size;
    h->spmvMethod = (SPMV_METHODS)method;
    h->RowPtr = RowPtr;  // borrowed, never written (common.c:157-159)
    h->ColIdx = ColIdx;
    h->Matrix_Val = Matrix_Val;
    // (fp32 Method_CSR5SPMV: the reference silently runs SELL and stores Method_SellCSigma in the handle,
    // common.c:177-180; here it is a real fp32 CSR5 and the public field keeps Method_CSR5SPMV -- a documented
    // deviation, include/spmv.h)
    DeviceState *st = new DeviceState();
    h->extraHandle = st;
    st->opts = read_create_options();
    st->refresh = st->opts.refresh;
    // Option "reorder": the reference's level-3 hook (common.c:144-156, compiled out upstream).  Same condition as
    // there (square, > 8096 rows, > 100000 non-zeros), HOST arrays only; the device layout is then built from
    // A' = P A P^T and the permutation is handed to the caller in handle->index (reorder.cu).
    std::vector<int> p_rowptr, p_col;
    std::vector<double> p_val;  // (storage only: 8-byte aligned, holds fp32 or fp64 values)
    if (st->opts.reorder && m == n && m > 8096 && RowPtr && ColIdx && Matrix_Val && !is_device_ptr(RowPtr) &&
        RowPtr[0] == 0 && RowPtr[m] > 100000) {
        const size_t nnz = (size_t)RowPtr[m];
        int *index = (int *)malloc(((size_t)m + 1) * sizeof(int));
        bool done = false;
        if (index && spmv_b200_reorder(m, RowPtr, ColIdx, index) == 0) {
            p_rowptr.resize((size_t)m + 1);
            p_col.resize(nnz);
            p_val.resize(nnz);
            done = spmv_b200_permute_csr(m, RowPtr, ColIdx, Matrix_Val, size, index, p_rowptr.data(), p_col.data(), p_val.data()) == 0;
        }
        if (done) {
            index[m] = m;
            h->index = index;           // freed by spmv_clear_handle
            h->Level_3_opt_used = 1;
            std::vector<int> p_map;     // option "refresh": where every permuted value comes from
            if (st->refresh) {
                p_map.resize(nnz);
                // (rewrites p_rowptr / p_col with what they already hold: the same permutation)
                if (permute_positions(m, RowPtr, ColIdx, index, p_rowptr.data(), p_col.data(), p_map.data()) != 0) st->map_failed = true;
            }
            st->ok = build_state(st, h, m, n, p_rowptr.data(), p_col.data(), p_val.data(), method, p_map.empty() ? nullptr : p_map.data());
            return;
        }
        free(index);
    }
    st->ok = build_state(st, h, m, n, RowPtr, ColIdx, Matrix_Val, method);
}

void spmv_create_handle_all_in_one(spmv_Handle_t *Handle, BASIC_INT_TYPE m, BASIC_INT_TYPE n,
                                   BASIC_INT_TYPE *RowPtr, BASIC_INT_TYPE *ColIdx, void *Matrix_Val,
                                   BASIC_SIZE_TYPE nthreads, SPMV_METHODS Function, BASIC_SIZE_TYPE size,
                                   VECTORIZED_WAY vectorizedWay, const char *MtxToken)
{
    (void)MtxToken;  // only keys the reference's compiled-out METIS cache (common.c:152-154)
    if (!Handle) return;
    spmv_Handle *h = (spmv_Handle *)malloc(sizeof(spmv_Handle));  // freed by spmv_destory_handle
    *Handle = h;
    if (!h) return;
    handle_init(h);
    create_into(h, m, n, RowPtr, ColIdx, Matrix_Val, nthreads, (int)Function, size, vectorizedWay);
}

void spmv(const spmv_Handle_t handle, BASIC_INT_TYPE m, const BASIC_INT_TYPE *RowPtr,
          const BASIC_INT_TYPE *ColIdx, const void *Matrix_Val, const void *Vector_Val_X, void *Vector_Val_Y)
{
    (void)m; (void)RowPtr; (void)ColIdx; (void)Matrix_Val;  // the handle owns the device copies
    DeviceState *st = state_of(handle);  // NULL handle: silent return (common.c:285)
    if (!st || !st->ok || !Vector_Val_Y || (!Vector_Val_X && st->n > 0)) return;
    std::lock_guard<std::mutex> lock(st->mu);
    DeviceGuard guard(st->device);
    const bool x_dev = is_device_ptr(Vector_Val_X), y_dev = is_device_ptr(Vector_Val_Y);
    const void *xd = Vector_Val_X;
    void *yd = Vector_Val_Y;
    const size_t xb = (size_t)st->n * st->vsize, yb = (size_t)st->m * st->vsize;
    if (st->opts.pin_host) {
        if (!x_dev && xb) note_host_buffer(st, 0, Vector_Val_X, xb);
        if (!y_dev && yb) note_host_buffer(st, 1, Vector_Val_Y, yb);
    }
    if (!x_dev && !st->stage.x.get() && !st->stage.x.alloc(st->n, st->vsize)) return;
    if (!y_dev && !st->stage.y.get() && !st->stage.y.alloc(st->m, st->vsize)) return;
    if (!x_dev && !y_dev && st->pipeline && st->n_peers == 0 && st->kernel == SPMV_B200_KERNEL_CSR_VECTOR && xb && yb) {
        with_precision(st, [&](auto t) {
            using T = decltype(t);
            return run_pipelined<T>(st, (const T *)Vector_Val_X, (T *)Vector_Val_Y);
        });
        return;
    }
    if (!x_dev) {
        if (xb && !SB_CUDA(cudaMemcpyAsync(st->stage.x.get(), Vector_Val_X, xb, cudaMemcpyHostToDevice, st->stream))) return;
        xd = st->stage.x.get();
        if (y_dev && xb) {
            // host x, device y: the call returns without a stream sync, but the caller may reuse X at once (a pinned
            // X makes this copy truly asynchronous): wait for the copy alone
            if (!st->ev_x) { if (!SB_CUDA(cudaEventCreateWithFlags(&st->ev_x, cudaEventDisableTiming))) return; }
            if (!SB_CUDA(cudaEventRecord(st->ev_x, st->stream)) || !SB_CUDA(cudaEventSynchronize(st->ev_x))) return;
        }
    }
    if (!y_dev) yd = st->stage.y.get();
    if (!with_precision(st, [&](auto t) { using T = decltype(t); return launch<T>(st, (const T *)xd, (T *)yd); })) return;
    if (!y_dev) {
        if (yb && !SB_CUDA(cudaMemcpyAsync(Vector_Val_Y, yd, yb, cudaMemcpyDeviceToHost, st->stream))) return;
        SB_CUDA(cudaStreamSynchronize(st->stream));  // host y is complete on return, as in the reference
    }
}

// y <- alpha A x + beta y, and with_dot: *dot = w . y; sigma (spmv_b200_spmv_shifted): y <- alpha (A - sigma I) x +
// beta y instead, and with_dot: dot[0] = x . y, dot[1] = y . y (w unused) (include/spmv_b200.h).  spmv()'s pointer
// rules without the pipelined host path; fn names the entry point in the errors.
static int scaled_product(const char *fn, spmv_Handle_t handle, double alpha, const void *x, double beta, void *y,
                          bool with_dot, const void *w, double *dot, const double *sigma = nullptr)
{
    DeviceState *st = state_of(handle);
    if (!st) { set_error("%s: NULL handle", fn); return -1; }
    if (!st->ok) { set_error("%s: the handle's create failed", fn); return -1; }
    if (sigma && st->m != st->n) { set_error("%s: the handle is not square", fn); return -1; }
    if (!y) { set_error("%s: y is NULL", fn); return -1; }
    const bool with_w = with_dot && !sigma;
    if (with_w && !dot) { set_error("%s: dot is NULL", fn); return -1; }
    if (with_w && !w) { set_error("%s: w is NULL", fn); return -1; }
    if (!x && st->n > 0) { set_error("%s: x is NULL", fn); return -1; }
    if (x == y) { set_error("%s: x and y are the same array", fn); return -1; }
    const bool w_is_x = with_w && w == x, w_is_y = with_w && w == y;
    if (w_is_x && st->m != st->n) { set_error("%s: w is x on a handle that is not square", fn); return -1; }
    const size_t yb = (size_t)st->m * st->vsize;
    if (with_w && !w_is_y && (const char *)w < (const char *)y + yb && (const char *)y < (const char *)w + yb) {
        set_error("%s: w overlaps y without being y", fn);
        return -1;
    }
    std::lock_guard<std::mutex> lock(st->mu);
    DeviceGuard guard(st->device);
    const bool dot_dev = with_dot && is_device_ptr(dot);
    const int ndots = sigma ? 2 : 1;
    if (st->m == 0) {
        if (!with_dot) return 0;
        if (!dot_dev) { std::fill(dot, dot + ndots, 0.0); return 0; }
        return SB_CUDA(cudaMemsetAsync(dot, 0, ndots * sizeof(double), st->stream)) ? 0 : -1;  // all-zero bits = +0.0
    }
    const bool ok = with_precision(st, [&](auto t) {
        using T = decltype(t);
        const T a = (T)alpha, b = (T)beta;  // fp32 handles: alpha and beta rounded to float first
        const T sg = sigma ? (T)*sigma : (T)0;  // and sigma
        // the shifted kernels run when there is a shift to apply or dots to take; otherwise the call is
        // spmv_b200_spmv_axpby's, bit for bit and launch for launch
        const bool shifted = sigma && (with_dot || (a != (T)0 && sg != (T)0));
        const bool read_x = (a != (T)0 && st->n > 0) || w_is_x || (sigma && with_dot), read_y = b != (T)0;
        const bool x_dev = read_x && is_device_ptr(x), y_dev = is_device_ptr(y);
        const bool stage_w = with_w && !w_is_x && !w_is_y && !is_device_ptr(w);
        const size_t xb = (size_t)st->n * sizeof(T);
        if (st->opts.pin_host) {
            if (read_x && !x_dev) note_host_buffer(st, 0, x, xb);
            if (!y_dev) note_host_buffer(st, 1, y, yb);
        }
        const T *xd = (const T *)x;
        T *yd = (T *)y;
        if (read_x && !x_dev) {
            if (!st->stage.x.get() && !st->stage.x.alloc(st->n, sizeof(T))) return false;
            if (!SB_CUDA(cudaMemcpyAsync(st->stage.x.get(), x, xb, cudaMemcpyHostToDevice, st->stream))) return false;
            xd = st->stage.x.as<T>();
        }
        const T *wd = w_is_y ? nullptr : w_is_x ? xd : (const T *)w;  // w_is_x: a host x's staged copy
        if (stage_w) {
            if (!st->stage.w.get() && !st->stage.w.alloc(st->m, sizeof(T))) return false;
            if (!SB_CUDA(cudaMemcpyAsync(st->stage.w.get(), w, yb, cudaMemcpyHostToDevice, st->stream))) return false;
            wd = st->stage.w.as<T>();
        }
        // as in spmv(): a call that returns before its kernels end waits for the copies of host inputs alone, so that
        // the caller may reuse them at once
        if (((read_x && !x_dev) || stage_w) && y_dev && (!with_dot || dot_dev)) {
            if (!st->ev_x && !SB_CUDA(cudaEventCreateWithFlags(&st->ev_x, cudaEventDisableTiming))) return false;
            if (!SB_CUDA(cudaEventRecord(st->ev_x, st->stream)) || !SB_CUDA(cudaEventSynchronize(st->ev_x))) return false;
        }
        if (!y_dev) {
            if (!st->stage.y.get() && !st->stage.y.alloc(st->m, sizeof(T))) return false;
            yd = st->stage.y.as<T>();
            if (read_y && !SB_CUDA(cudaMemcpyAsync(yd, y, yb, cudaMemcpyHostToDevice, st->stream))) return false;
        }
        Scaled<T> sc{{yd, a, b}, wd, nullptr, 0};
        if (shifted) {
            sc.shifted = true;
            sc.sigma = sg;
            sc.x = xd;  // a host x: its staged copy
        }
        DeviceArray<double> &result = sigma ? st->dot.pair : st->dot.result;
        if (!with_dot) {
            if (!launch_axpby<T>(st, xd, sc)) return false;
        } else {
            const size_t bound = (size_t)dot_partials_bound(st);
            if (!st->dot.partials && !st->dot.partials.alloc(bound)) return false;
            if (sigma && !st->dot.yy && !st->dot.yy.alloc(bound)) return false;
            if (!dot_dev && !result && !result.alloc(ndots)) return false;
            sc.partials = st->dot.partials;
            sc.yy = st->dot.yy;
            if (!launch_axpby_dot<T>(st, xd, sc, dot_dev ? dot : result.get())) return false;
        }
        if (!y_dev && !SB_CUDA(cudaMemcpyAsync(y, yd, yb, cudaMemcpyDeviceToHost, st->stream))) return false;
        if (with_dot && !dot_dev && !SB_CUDA(cudaMemcpyAsync(dot, result.get(), ndots * sizeof(double), cudaMemcpyDeviceToHost, st->stream))) return false;
        return (y_dev && (!with_dot || dot_dev)) || SB_CUDA(cudaStreamSynchronize(st->stream));
    });
    return ok ? 0 : -1;
}

int spmv_b200_spmv_axpby(spmv_Handle_t handle, double alpha, const void *x, double beta, void *y)
{
    return scaled_product("spmv_b200_spmv_axpby", handle, alpha, x, beta, y, false, nullptr, nullptr);
}

int spmv_b200_spmv_axpby_dot(spmv_Handle_t handle, double alpha, const void *x, double beta, void *y, const void *w,
                             double *dot)
{
    return scaled_product("spmv_b200_spmv_axpby_dot", handle, alpha, x, beta, y, true, w, dot);
}

int spmv_b200_spmv_shifted(spmv_Handle_t handle, double alpha, double sigma, const void *x, double beta, void *y,
                           double *dots)
{
    return scaled_product("spmv_b200_spmv_shifted", handle, alpha, x, beta, y, dots != nullptr, nullptr, dots, &sigma);
}

void spmv_clear_handle(spmv_Handle_t this_handle)  // reference gemv_Handle_clear, common.c:31-52,69-71
{
    if (!this_handle) return;
    free_state(state_of(this_handle));
    if (this_handle->Level_3_opt_used && this_handle->index) free(this_handle->index);  // ours (option "reorder")
    handle_init(this_handle);
}

void spmv_destory_handle(spmv_Handle_t this_handle)  // reference common.c:54-61
{
    if (!this_handle) return;
    spmv_clear_handle(this_handle);
    free(this_handle);
}

// The reference re-reads the caller's Matrix_Val on every spmv() (Serial / Parallel / Balanced*); here the values are
// part of the device layout.  A client that changes values on a fixed pattern calls this instead of destroy + create:
// the handle is rebuilt in place from its own borrowed RowPtr / ColIdx, the values given here (NULL: the Matrix_Val
// it was created with, re-read), the same method, precision, nthreads and stream.  Cost: one create.
int spmv_b200_update_values(spmv_Handle_t handle, void *Matrix_Val)
{
    DeviceState *st = state_of(handle);
    if (!st || !st->ok) return -1;  // (a handle whose create failed has nothing to refresh)
    const int m = st->m, n = st->n, method = st->requested;
    cudaStream_t stream = st->stream;
    BASIC_INT_TYPE *rp = handle->RowPtr, *ci = handle->ColIdx;
    void *va = Matrix_Val ? Matrix_Val : handle->Matrix_Val;
    const BASIC_SIZE_TYPE nthreads = handle->nthreads, size = handle->data_size;
    const VECTORIZED_WAY vw = handle->vectorizedWay;
    spmv_clear_handle(handle);
    create_into(handle, m, n, rp, ci, va, nthreads, method, size, vw);
    DeviceState *fresh = state_of(handle);
    if (fresh) fresh->stream = stream;
    return fresh && fresh->ok ? 0 : -1;
}

// Option "refresh": new values on the handle's stream, through the source maps kept at create (refresh.cuh).  The
// owned upload in the caller's order takes the values as they are (one copy); every other value array is gathered
// from them in one launch.
int spmv_b200_set_values(spmv_Handle_t handle, const void *Matrix_Val)
{
    DeviceState *st = state_of(handle);
    if (!st) { set_error("spmv_b200_set_values: NULL handle"); return -1; }
    if (!st->ok) { set_error("spmv_b200_set_values: the handle's create failed"); return -1; }
    if (!st->refresh) {
        set_error("spmv_b200_set_values: the handle keeps no source maps (create it with option \"refresh\" = 1; "
                  "spmv_b200_info(h, \"refreshable\") = 0)");
        return -1;
    }
    std::lock_guard<std::mutex> lock(st->mu);
    DeviceGuard guard(st->device);
    if (st->m == 0 || st->nnz == 0) return 0;
    const void *src = Matrix_Val ? Matrix_Val : handle->Matrix_Val;
    if (st->val && !st->upload.val.get() && src != st->val) {  // an adopted device CSR is the caller's: never written
        set_error("spmv_b200_set_values: the handle adopted the caller's device Matrix_Val %p; refresh it in place and pass "
                  "NULL or that pointer (got %p)", st->val, src);
        return -1;
    }
    cudaPointerAttributes a;
    bool on_device = false;
    if (cudaPointerGetAttributes(&a, src) != cudaSuccess) cudaGetLastError();
    else on_device = a.type == cudaMemoryTypeDevice || a.type == cudaMemoryTypeManaged;
    if (on_device && a.type == cudaMemoryTypeDevice && a.device != st->device) {
        set_error("spmv_b200_set_values: Matrix_Val is on device %d, the handle on device %d", a.device, st->device);
        return -1;
    }
    RefreshTable tab = {};
    long long quads = 0;
    auto add = [&](void *dst, const int *map, long long count) {
        if (!map || count <= 0 || tab.n == kRefreshMaxTargets) return;
        tab.t[tab.n++] = {dst, map, count, quads};
        quads += (count + 3) / 4;
    };
    add(st->upload.val.get(), st->upload.map, st->nnz);
    add(st->v.val.get(), st->v.map, st->nnz);
    add(st->sell.val.get(), st->sell.map, st->sell.padded);
    add(st->c5.val.get(), st->c5.map, st->nnz);
    add(st->seg.ent_val.get(), st->seg.map, st->seg.ptr[st->seg.bands]);
    const size_t bytes = (size_t)st->nnz * st->vsize;
    const void *from = src;  // what the gather reads
    void *copy_to = nullptr;
    if (st->upload.val.get() && !st->upload.map) copy_to = st->upload.val.get();  // the identity target
    else if (!on_device && tab.n > 0) {
        if (!st->stage.val.get() && !st->stage.val.alloc((size_t)st->nnz, st->vsize)) return -1;
        copy_to = st->stage.val.get();
    }
    if (copy_to) {
        if (!SB_CUDA(cudaMemcpyAsync(copy_to, src, bytes, cudaMemcpyDefault, st->stream))) return -1;
        from = copy_to;
    }
    if (!on_device) {  // the caller may reuse a host array at once: wait for its copy alone
        if (!st->ev_x && !SB_CUDA(cudaEventCreateWithFlags(&st->ev_x, cudaEventDisableTiming))) return -1;
        if (!SB_CUDA(cudaEventRecord(st->ev_x, st->stream))) return -1;
    }
    if (tab.n > 0) {  // (not on the spmv() path: not in spmv_b200_launch_count)
        with_precision(st, [&](auto t) {
            using T = decltype(t);
            value_refresh_kernel<T><<<blocks_for(quads), kThreads, 0, st->stream>>>(tab, (const T *)from);
        });
        if (!SB_CUDA(cudaGetLastError())) return -1;
    }
    if (!on_device && !SB_CUDA(cudaEventSynchronize(st->ev_x))) return -1;
    return 0;
}

// ================================================================================================
// extensions (include/spmv_b200.h)
// ================================================================================================
int spmv_b200_version(void) { return SPMV_B200_VERSION; }
const char *spmv_b200_last_error(void) { return g_err; }
void spmv_b200_clear_error(void) { g_err[0] = 0; }
unsigned long long spmv_b200_launch_count(void) { return g_launches.load(); }
long long spmv_b200_live_allocations(void) { return g_live_allocations.load(); }

void spmv_b200_set_stream(spmv_Handle_t handle, void *cuda_stream)
{
    if (DeviceState *st = state_of(handle)) {
        std::lock_guard<std::mutex> lock(st->mu);
        st->stream = (cudaStream_t)cuda_stream;
    }
}

void spmv_b200_sync(spmv_Handle_t handle)
{
    if (DeviceState *st = state_of(handle)) {
        DeviceGuard g(st->device);
        SB_CUDA(cudaStreamSynchronize(st->stream));
    }
}

int spmv_b200_set_y_peers(spmv_Handle_t handle, int count, void *const *device_ptrs)
{
    DeviceState *st = state_of(handle);
    if (!st || count < 0 || count > kMaxPeers || (count > 0 && !device_ptrs)) return -1;
    std::lock_guard<std::mutex> lock(st->mu);
    st->n_peers = count;
    for (int i = 0; i < kMaxPeers; ++i) st->peers[i] = i < count ? device_ptrs[i] : nullptr;
    return 0;
}

// ---- column stages: the contribution of a range of column bands, then the fold ----------------------
static bool stageable(const DeviceState *st)
{
    if (!st || !st->ok || st->x_bands <= 1) return false;
    if (st->kernel == SPMV_B200_KERNEL_BAND_SEG) return true;
    return st->kernel == SPMV_B200_KERNEL_CSR_VECTOR && !st->lr.binned && st->lr.rows == 0;
}

int spmv_b200_bands(spmv_Handle_t handle)
{
    DeviceState *st = state_of(handle);
    if (!st || !st->ok) return -1;
    return stageable(st) ? st->x_bands : 1;
}

int spmv_b200_band_columns(spmv_Handle_t handle, int band, long long *col_lo, long long *col_hi)
{
    DeviceState *st = state_of(handle);
    if (!st || !st->ok || band < 0) return -1;
    const int K = stageable(st) ? st->x_bands : 1;
    if (band >= K) return -1;
    const auto cols = band_columns(st, band, K);
    if (col_lo) *col_lo = cols.first;
    if (col_hi) *col_hi = cols.second;
    return 0;
}

int spmv_b200_spmv_bands(spmv_Handle_t handle, int band_first, int band_count, const void *x_device)
{
    DeviceState *st = state_of(handle);
    if (!stageable(st) || band_first < 0 || band_count < 0 || band_first + band_count > st->x_bands) return -1;
    if (band_count == 0) return 0;
    if (!is_device_ptr(x_device)) { set_error("spmv_b200_spmv_bands: x must be a device pointer"); return -1; }
    std::lock_guard<std::mutex> lock(st->mu);
    DeviceGuard guard(st->device);
    const bool ok = with_precision(st, [&](auto t) {
        using T = decltype(t);
        if (st->kernel == SPMV_B200_KERNEL_BAND_SEG) return launch_seg_bands<T>(st, band_first, band_count, (const T *)x_device);
        const int r0 = band_first * st->m, r1 = (band_first + band_count) * st->m;  // virtual rows of these bands
        launch_vector<T>(st, r0, r1, (const T *)x_device, st->v.y.as<T>(), PeerList<T>{});
        return SB_CUDA(cudaGetLastError());
    });
    return ok ? 0 : -1;
}

int spmv_b200_spmv_finish(spmv_Handle_t handle, void *y_device)
{
    DeviceState *st = state_of(handle);
    if (!stageable(st)) return -1;
    if (!is_device_ptr(y_device)) { set_error("spmv_b200_spmv_finish: y must be a device pointer"); return -1; }
    std::lock_guard<std::mutex> lock(st->mu);
    DeviceGuard guard(st->device);
    const bool ok = with_precision(st, [&](auto t) {
        using T = decltype(t);
        return st->kernel == SPMV_B200_KERNEL_BAND_SEG ? launch_seg_finish<T>(st, (T *)y_device) : launch_band_fold<T>(st, (T *)y_device);
    });
    return ok ? 0 : -1;
}

// ---- stream-ordered building blocks of a copy-engine exchange (multigpu.py: CopyEnginePowerMethod) ----
int spmv_b200_memcpy_async(void *dst, const void *src, size_t bytes, void *cuda_stream)
{
    if (!bytes) return 0;
    return SB_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToDevice, (cudaStream_t)cuda_stream)) ? 0 : -1;
}

typedef int (*StreamValueFn)(cudaStream_t, unsigned long long /*CUdeviceptr*/, unsigned, unsigned);
static StreamValueFn driver_fn(const char *name)
{
    void *fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint(name, &fn, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) {
        cudaGetLastError();
        set_error("driver entry point %s is not available", name);
        return nullptr;
    }
    return (StreamValueFn)fn;
}

int spmv_b200_stream_write32(void *cuda_stream, void *device_ptr, unsigned value)
{
    static StreamValueFn fn = driver_fn("cuStreamWriteValue32");
    if (!fn || !device_ptr) return -1;
    const int rc = fn((cudaStream_t)cuda_stream, (unsigned long long)(uintptr_t)device_ptr, value, 0 /*CU_STREAM_WRITE_VALUE_DEFAULT*/);
    if (rc != 0) { set_error("cuStreamWriteValue32 failed (%d)", rc); return -1; }
    return 0;
}

int spmv_b200_stream_wait32_geq(void *cuda_stream, void *device_ptr, unsigned value)
{
    static StreamValueFn fn = driver_fn("cuStreamWaitValue32");
    if (!fn || !device_ptr) return -1;
    const int rc = fn((cudaStream_t)cuda_stream, (unsigned long long)(uintptr_t)device_ptr, value, 0 /*CU_STREAM_WAIT_VALUE_GEQ*/);
    if (rc != 0) { set_error("cuStreamWaitValue32 failed (%d)", rc); return -1; }
    return 0;
}

int spmv_b200_ipc_export(const void *device_ptr, void *handle_out_64)
{
    if (!device_ptr || !handle_out_64) return -1;
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    cudaIpcMemHandle_t h;
    if (!SB_CUDA(cudaIpcGetMemHandle(&h, const_cast<void *>(device_ptr)))) return -1;
    memcpy(handle_out_64, &h, sizeof(h));
    return 0;
}

void *spmv_b200_ipc_open(const void *handle_64)
{
    if (!handle_64) return nullptr;
    cudaIpcMemHandle_t h;
    memcpy(&h, handle_64, sizeof(h));
    void *p = nullptr;
    if (!SB_CUDA(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess))) return nullptr;
    return p;
}

int spmv_b200_ipc_close(void *opened_ptr)
{
    if (!opened_ptr) return -1;
    return SB_CUDA(cudaIpcCloseMemHandle(opened_ptr)) ? 0 : -1;
}

int spmv_b200_set_option(const char *key, long long value)
{
    Options &o = options();
    std::lock_guard<std::mutex> g(o.mu);
    auto it = o.v.find(key ? key : "");
    if (it == o.v.end()) return -1;
    it->second = value;
    o.user_set[key] = true;
    return 0;
}

long long spmv_b200_get_option(const char *key) { return key ? opt(key) : -1; }

long long spmv_b200_info(spmv_Handle_t handle, const char *key)
{
    DeviceState *st = state_of(handle);
    if (!st || !key) return -1;
    const std::string k(key);
    if (k == "kernel") return st->kernel;
    if (k == "requested") return st->requested;
    if (k == "ok") return st->ok;
    if (k == "m") return st->m;
    if (k == "n") return st->n;
    if (k == "nnz") return st->nnz;
    if (k == "tpr") return st->tpr;
    if (k == "parts") return st->split.parts;
    if (k == "ref_parts") return st->split.ref_T;
    if (k == "tiles") return st->tile.count;
    if (k == "tile_items") return st->tile.items;
    if (k == "sigma") return st->sell.sigma;
    if (k == "banner") return st->sell.banner;
    if (k == "slices") return st->sell.slices;
    if (k == "sell_variant") return st->sell.variant;
    if (k == "padded_nnz") return st->sell.padded;
    if (k == "csr5_p") return st->c5.p;
    if (k == "csr5_sigma") return st->c5.sigma;
    if (k == "csr5_bit_y_offset") return st->c5.bit_y;
    if (k == "csr5_bit_scansum_offset") return st->c5.bit_ss;
    if (k == "csr5_num_offsets") return st->c5.num_offsets;
    if (k == "csr5_tail_start") return st->c5.tail_start;
    if (k == "pipeline") return st->pipeline;
    if (k == "values_snapshotted") return 1;
    if (k == "refreshable") return st->refresh;
    if (k == "binned") return st->lr.binned;
    if (k == "pinned_host_buffers") return (int)st->pin[0].registered + (int)st->pin[1].registered;
    if (k == "long_rows") return st->lr.rows;
    if (k == "long_segs") return st->lr.segs;
    if (k == "long_thr") return st->lr.thr;
    if (k == "device") return st->device;
    if (k == "has_empty_rows") return st->has_empty_rows;
    if (k == "x_bands") return st->x_bands;
    if (k == "auto_method") return st->auto_method;
    if (k == "seg_bands") return st->seg.bands;
    if (k == "segments") return st->seg.total;
    if (k == "seg_cross") return st->seg.cross;
    if (k == "seg_ctas") return st->seg.ctas;
    if (k == "layout_fallbacks") return st->layout_fallbacks;
    if (k == "band_cols") return st->band_cols;
    if (k == "far_permille") return (long long)(st->far_fraction * 1000.0);
    if (k == "active_rows") return st->a_m;
    if (k == "owns_csr") return st->upload.rowptr.get() != nullptr;
    if (k == "released_csr") return st->released_csr;
    if (k == "dev_l2_bytes") return st->dev_l2;
    if (k == "axpby_path") return axpby_path(st);
    if (k == "dot_path") return dot_path(st);
    return -1;
}

long long spmv_b200_structure(spmv_Handle_t handle, const char *name, void *dst, size_t dst_bytes)
{
    DeviceState *st = state_of(handle);
    if (!st || !name) return -1;
    const std::string k(name);
    const void *src = nullptr;
    size_t bytes = 0;
    if (k == "splitter") { src = st->split.splitter; bytes = ((size_t)st->split.parts + 1) * 4; }
    else if (k == "ref_splitter") { src = st->split.ref_splitter; bytes = ((size_t)st->split.ref_T + 1) * 4; }
    else if (k == "tile_rows") { src = st->tile.rows; bytes = ((size_t)st->tile.count + 1) * 4; }
    else if (k == "merge_coords") { src = st->tile.merge_coords; bytes = ((size_t)st->tile.count + 1) * 8; }
    else if (k == "sell_perm") { src = st->sell.perm; bytes = (size_t)st->sell.banner * 4; }
    else if (k == "sell_width") { src = st->sell.width; bytes = (size_t)st->sell.slices * 4; }
    else if (k == "sell_full") { src = st->sell.full; bytes = (size_t)st->sell.slices * 4; }
    else if (k == "sell_slice_ptr") { src = st->sell.slice_ptr; bytes = ((size_t)st->sell.slices + 1) * 8; }
    else if (k == "sell_col") { src = st->sell.col; bytes = (size_t)st->sell.padded * 4; }
    else if (k == "sell_val") { src = st->sell.val.get(); bytes = (size_t)st->sell.padded * st->vsize; }
    else if (k == "csr5_tile_ptr") { src = st->c5.tile_ptr; bytes = ((size_t)st->c5.p + 1) * 4; }
    else if (k == "csr5_tile_desc") { src = st->c5.tile_desc; bytes = (size_t)st->c5.p * kC5Omega * 4; }
    else if (k == "csr5_offset_ptr") { src = st->c5.off_ptr; bytes = ((size_t)st->c5.p + 1) * 4; }
    else if (k == "csr5_offsets") { src = st->c5.off; bytes = (size_t)st->c5.num_offsets * 4; }
    else if (k == "csr5_col") { src = st->c5.col; bytes = (size_t)st->nnz * 4; }
    else if (k == "csr5_val") { src = st->c5.val.get(); bytes = (size_t)st->nnz * st->vsize; }
    else if (k == "seg_col") { src = st->seg.col; bytes = st->seg.col ? (size_t)st->seg.ptr[st->seg.bands] * 4 : 0; }
    else if (k == "seg_mask") { src = st->seg.mask.get(); bytes = src ? (size_t)st->m * (st->seg.mask64 ? 8 : 4) : 0; }
    else if (k == "seg_gbase") { src = st->seg.gbase; bytes = st->seg.gbase ? (size_t)st->seg.bands * st->seg.groups * 4 : 0; }
    else if (k == "seg_chunk_seg0") { src = st->seg.tile_seg0; bytes = st->seg.tile_seg0 ? ((size_t)st->tile.count * kSegChunks + 1) * 4 : 0; }
    else if (k == "seg_ptr" || k == "seg_cnt") {
        const int *tab = k == "seg_ptr" ? st->seg.ptr : st->seg.cnt;
        const size_t need = (size_t)(st->seg.bands + (k == "seg_ptr" ? 1 : 0)) * 4;
        if (!dst) return st->seg.bands > 1 ? (long long)need : 0;
        if (st->seg.bands <= 1 || dst_bytes < need) return -1;
        memcpy(dst, tab, need);
        return (long long)need;
    }
    else if (k == "band_rowptr") { src = st->v.rowptr; bytes = st->v.rowptr ? ((size_t)st->a_m + 1) * 4 : 0; }
    else if (k == "band_col") { src = st->v.col; bytes = st->v.col ? (size_t)st->nnz * 4 : 0; }
    else return -1;
    if (!src) bytes = 0;
    if (!dst || bytes == 0) return (long long)bytes;
    if (dst_bytes < bytes) { set_error("structure %s needs %zu bytes, got %zu", name, bytes, dst_bytes); return -1; }
    DeviceGuard g(st->device);
    if (!SB_CUDA(cudaStreamSynchronize(st->stream))) return -1;
    if (!SB_CUDA(cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost))) return -1;
    return (long long)bytes;
}

int spmv_b200_partition_rows(const int *RowPtr, int m, int parts, int *splitter_out)
{
    if (!RowPtr || !splitter_out || m < 0 || parts < 1) return -1;
    const int nnz = RowPtr[m] - RowPtr[0];
    const long long stride = ((long long)nnz + parts - 1) / parts;
    for (int g = 0; g <= parts; ++g) {
        long long b = (long long)g * stride;
        if (b > nnz) b = nnz;
        splitter_out[g] = right_boundary(RowPtr, (int)b, m + 1) - 1;
    }
    return 0;
}

int spmv_b200_recommend_method(int m, const int *RowPtr)
{
    if (!RowPtr || m < 0) return -1;
    const long long nnz = (long long)RowPtr[m] - RowPtr[0];
    return pick_method(m, nnz, /*far_fraction: unknown*/ -1.0, [&](int cut, long long *heavy) {
        for (int r = 0; r < m; ++r) {
            const long long len = (long long)RowPtr[r + 1] - RowPtr[r];
            if (len > cut) *heavy += len;
        }
        return true;
    });
}

void *spmv_b200_malloc(size_t bytes)
{
    void *p = nullptr;
    if (!SB_CUDA(cudaMalloc(&p, bytes ? bytes : 1))) return nullptr;
    return p;
}

void spmv_b200_free(void *device_ptr)
{
    if (device_ptr) cudaFree(device_ptr);
}

int spmv_b200_memcpy(void *dst, const void *src, size_t bytes, int kind)
{
    const cudaMemcpyKind k = kind == 0 ? cudaMemcpyHostToDevice : kind == 1 ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice;
    return SB_CUDA(cudaMemcpy(dst, src, bytes, k)) ? 0 : -1;
}

}  // extern "C"
