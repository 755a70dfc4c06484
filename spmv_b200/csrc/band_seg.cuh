// band_seg.cuh -- column bands for matrices whose bands are hyper-sparse ("band segments").
//
// The band-major copy of csr_kernels.cuh stores band b of row r as virtual row b*m + r of a CSR.  When x is so
// large that the number of bands K approaches the mean row length (BASELINE.json config C5: 16 non-zeros per
// row, x = 2 GiB => K = 48, a third of a non-zero per row and band) the K*m+1 virtual row pointers outweigh the matrix,
// and a y vector that is swept once per band (round 1's COO bands) costs 2*K*m*sizeof(val) bytes of DRAM traffic.
// Here the matrix is the list of its entries, stably bucketed by col / band_cols and sorted by row inside a band;
// a maximal run of entries of one row inside one band is a SEGMENT, marked by bit 31 of the column index of its
// last entry.  No row ids are stored (12 bytes per non-zero for fp64, as in CSR).  y = A x in two passes:
//
//   pass 1  bseg_kernel        persistent warp-specialised CTAs over tiles of 2048 consecutive entries (tiles never span
//                              bands; a ticket counter hands them out in band order, so the gathers of all CTAs stay
//                              inside one L2-resident slice of x).  A producer warp streams the tiles' ColIdx / Val
//                              slices into a 3-stage shared-memory ring with cp.async.bulk (TMA) + mbarriers; eight
//                              consumer warps each walk one 256-entry chunk, 8 consecutive entries per lane, with the
//                              gathers of the NEXT tile already in flight; a warp-level segmented scan numbers the
//                              segments and carries open runs across lanes; the chunk's segment sums leave as one
//                              coalesced streaming write into seg_sums, the band-major list of all segment sums.  A
//                              run still open at a chunk's end goes to carry_val[chunk] and is added to its segment by
//                              the carry fix-up kernels, in chunk order.
//   pass 2  bseg_merge_kernel  one lane per row: a K-bit mask says in which bands the row has a segment, and
//                              gbase[32-row group][band] + a ballot/popc rank gives its position in that band's
//                              list; the (up to K) partial sums are added in band order and y is written ONCE.
//
// DRAM traffic per SpMV: 12 B/nnz + x + 16 B/segment + masks + y, all of it streaming -- no read-modify-write of
// y, no atomics, fixed order: bitwise reproducible.  The reference has no counterpart (its x lives behind the CPU
// caches); this is the GPU answer to "x does not fit the last-level cache".
#pragma once
#include "common.cuh"
#include "tile_kernels.cuh"

namespace sb {

constexpr int kSegIpt = 8;
constexpr int kSegTile = kThreads * kSegIpt;  // entries per tile of pass 1
constexpr int kSegChunks = kWarpsPerCta;      // consumer warps of pass 1: each owns one chunk of a tile
constexpr int kSegChunk = kSegTile / kSegChunks;  // 256 entries, 8 per lane
constexpr int kSegMaxBands = 64;              // one mask bit per band (uint32 masks up to 32 bands)
constexpr unsigned kSegEndBit = 0x80000000u;

// ---- bulk-copy (TMA) + mbarrier primitives: PTX cp.async.bulk -> SASS UBLKCP, mbarrier -> SYNCS ----
__device__ __forceinline__ uint32_t smem_addr(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t *bar, int count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_addr(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t *bar, uint32_t bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_addr(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t *bar, uint32_t parity)
{
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "SB_WAIT:\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
        "@p bra SB_DONE;\n"
        "bra SB_WAIT;\n"
        "SB_DONE:\n"
        "}" ::"r"(smem_addr(bar)), "r"(parity) : "memory");
}
// global -> shared, `bytes` a multiple of 16, both addresses 16-byte aligned; completes on `bar`
__device__ __forceinline__ void bulk_load(void *smem_dst, const void *gmem_src, uint32_t bytes, uint64_t *bar, uint64_t policy)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint [%0], [%1], %2, [%3], %4;"
                 ::"r"(smem_addr(smem_dst)), "l"(gmem_src), "r"(bytes), "r"(smem_addr(bar)), "l"(policy) : "memory");
}

__device__ __forceinline__ void stg_stream(double *p, double v, uint64_t pol)
{
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.f64 [%0], %1, %2;" ::"l"(p), "d"(v), "l"(pol) : "memory");
}
__device__ __forceinline__ void stg_stream(float *p, float v, uint64_t pol)
{
    asm volatile("st.global.L1::no_allocate.L2::cache_hint.f32 [%0], %1, %2;" ::"l"(p), "f"(v), "l"(pol) : "memory");
}

// ------------------------------------------------------------------------------------------------
// Builders (handle construction)
// ------------------------------------------------------------------------------------------------

// per CSR entry: its row and its band (the sort key); per row: the mask of bands it has entries in
template <typename MaskT>
__global__ void bseg_expand_kernel(int m, int band_cols, int bands, const int *__restrict__ rowptr,
                                   const int *__restrict__ col, int *__restrict__ ent_row,
                                   unsigned char *__restrict__ ent_band, MaskT *__restrict__ mask)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= m) return;
    MaskT mk = 0;
    for (int j = rowptr[r]; j < rowptr[r + 1]; ++j) {
        int b = col[j] / band_cols;
        b = b < 0 ? 0 : (b >= bands ? bands - 1 : b);
        ent_row[j] = r;
        ent_band[j] = (unsigned char)b;
        mk |= (MaskT)1 << b;
    }
    mask[r] = mk;
}

__global__ void set_int_kernel(int *p, int v) { *p = v; }

__global__ void bseg_iota_kernel(int n, int *__restrict__ a)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) a[i] = i;
}

// band_ptr[b] = first sorted entry whose key is >= b (also used for the row bins of Method_Parallel)
__global__ void sorted_key_ptr_kernel(int count, int keys, const unsigned char *__restrict__ sorted_key,
                                      int *__restrict__ key_ptr)
{
    const int b = blockIdx.x * blockDim.x + threadIdx.x;
    if (b > keys) return;
    int lo = 0, hi = count;
    while (lo < hi) {
        const int mid = (int)(((long long)lo + hi) >> 1);
        if ((int)sorted_key[mid] < b) lo = mid + 1; else hi = mid;
    }
    key_ptr[b] = lo;
}

// sorted entry i -> its slot in the band-major arrays (band starts are aligned to 4 entries for the bulk copies),
// column index with the segment-end bit, value
template <typename T>
__global__ void bseg_gather_kernel(int nnz, const int *__restrict__ order, const unsigned char *__restrict__ sorted_band,
                                   const int *__restrict__ ent_row, const int *__restrict__ col, const T *__restrict__ val,
                                   const int *__restrict__ band_ptr, const int *__restrict__ band_start,
                                   int *__restrict__ bcol, T *__restrict__ bval)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nnz) return;
    const int b = sorted_band[i];
    const int j = order[i];
    const int r = ent_row[j];
    const bool last = (i + 1 == band_ptr[b + 1]) || ent_row[order[i + 1]] != r;
    const int dst = band_start[b] + (i - band_ptr[b]);
    bcol[dst] = (int)((unsigned)col[j] | (last ? kSegEndBit : 0u));
    bval[dst] = val[j];
}

// one warp per tile: its entry range, how many segments end in each of its 8 chunks of 256 entries (one chunk per
// consumer warp of pass 1), whether a segment crosses a chunk's end, and its L2-prefetch duty
__global__ void bseg_tile_kernel(int tiles, int bands, int band_cols, int n, int vsize, const int *__restrict__ band_tile0,
                                 const int *__restrict__ band_start, const int *__restrict__ band_cnt, const int *__restrict__ bcol,
                                 int4 *__restrict__ tile_ent, int *__restrict__ chunk_segs, int *__restrict__ cross_flag)
{
    const int t = (int)(((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5);
    const int lane = threadIdx.x & 31;
    if (t >= tiles) return;
    int b = 0;
    while (b + 1 < bands && band_tile0[b + 1] <= t) ++b;
    const int k = t - band_tile0[b];
    const int e0 = band_start[b] + k * kSegTile;
    const int cnt = min(kSegTile, band_cnt[b] - k * kSegTile);
    // lane l counts the 64 entries [64 l, 64 l + 64); four lanes make a chunk
    int c = 0;
    const int i0 = lane * (kSegTile / 32);
    for (int i = i0; i < i0 + kSegTile / 32 && i < cnt; ++i) c += (int)((unsigned)bcol[e0 + i] >> 31);
    c += __shfl_xor_sync(kFull, c, 1);
    c += __shfl_xor_sync(kFull, c, 2);
    if ((lane & 3) == 0) {
        const int w = lane >> 2;
        chunk_segs[(size_t)t * kSegChunks + w] = c;
        const int last = min(cnt, (w + 1) * kSegChunk) - 1;  // last valid entry of the chunk
        if (last >= w * kSegChunk && bcol[e0 + last] >= 0) *cross_flag = 1;
    }
    if (lane == 0) {
        // L2 prefetch duty of this tile: the tiles of the SECOND HALF of band b stream the x slice of band b + 1 into
        // L2 (sequentially, at DRAM speed), so that the first touch of every sector in the next band is an L2 hit
        // instead of a random DRAM access.  Chunk = slice / (tiles doing the duty), in 16-byte units.
        int pf_off = 0, pf_cnt = 0;
        const int nt = band_tile0[b + 1] - band_tile0[b];
        const int duty0 = nt / 2, duty = nt - duty0;
        if (b + 1 < bands && k >= duty0) {
            const long long lo = (long long)(b + 1) * band_cols;
            long long hi = lo + band_cols;
            if (hi > n) hi = n;
            const int per16 = 16 / vsize;  // elements per 16 bytes
            const long long units = (hi - lo) / per16;  // whole 16-byte units of the slice
            const long long u0 = units * (k - duty0) / duty, u1 = units * (k - duty0 + 1) / duty;
            if (u1 > u0 && lo % per16 == 0) { pf_off = (int)(lo + u0 * per16); pf_cnt = (int)((u1 - u0) * per16); }
        }
        tile_ent[t] = make_int4(e0, cnt, pf_off, pf_cnt);
    }
}

// per 32-row group ("row warp") and band: how many of its rows have a segment in that band (layout [band][group], so
// that ONE exclusive scan over the whole array yields positions in the band-major list of segment sums)
template <typename MaskT>
__global__ void __launch_bounds__(kThreads)
bseg_group_count_kernel(int m, int bands, int groups, const MaskT *__restrict__ mask, int *__restrict__ cnt)
{
    const long long g = ((long long)blockIdx.x * kThreads + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    if (g >= groups) return;
    const long long r = g * 32 + lane;
    const MaskT mk = r < m ? mask[r] : (MaskT)0;
    for (int b = 0; b < bands; ++b) {
        const int c = __popc(__ballot_sync(kFull, (mk >> b) & 1));
        if (lane == 0) cnt[(size_t)b * groups + g] = c;
    }
}

// [band][group] -> [group][band]: the merge pass reads a group's K positions with one coalesced load
__global__ void bseg_transpose_kernel(int bands, int groups, const int *__restrict__ in, int *__restrict__ out)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= (long long)bands * groups) return;
    const int g = (int)(i / bands), b = (int)(i - (long long)g * bands);
    out[i] = in[(size_t)b * groups + g];
}

// ------------------------------------------------------------------------------------------------
// pass 1: segment sums.  Persistent, warp-specialised CTAs over tiles [tile_lo, tile_hi).
//
// History (all measured on the C5 shard, profiles/r02_c5shard_*): one tile per CTA with block-wide scans was
// latency-bound (10.7 ms, 0.55 IPC: every tile paid DRAM latency twice in sequence -- bulk copy, then gathers -- and
// three block barriers); persistent CTAs with the gathers of tile i+1 issued before tile i is walked: 5.0 ms; a
// dynamic tile schedule + sequential L2 prefetch of the next band's x slice: 4.1 ms with DRAM reads down from 19 GB
// to 9.9 GB; what remained were block barriers and the serial cross-warp prefix.  This version has neither:
//   * one PRODUCER warp per CTA takes tiles from an integer ticket counter (dynamic schedule: all CTAs of the grid
//     work within a few hundred tiles of one another, i.e. inside one column band whose slice of x stays in L2; a
//     static stride lets CTAs drift bands apart -- 62 % of the gathers missed L2 instead of 28 %), waits for a free
//     stage of a 3-deep ring, and fills it with the tile's ColIdx / Val slices by cp.async.bulk (TMA), completing
//     on the stage's "full" mbarrier; it also issues the tile's share of the L2 prefetch of the NEXT band's x slice;
//   * eight CONSUMER warps each own one 256-entry chunk of every tile (8 consecutive entries per lane: 128-bit
//     shared loads, no bank conflicts): the gathers of the next tile's chunk are issued into registers BEFORE the
//     current chunk is walked (two register sets, swapped every step: no moves that would wait for a load); a
//     WARP-level segmented scan numbers the chunk's segments and carries open runs across lanes; the chunk's segment
//     sums are staged over its own (dead) values and leave as one coalesced streaming write at a position known
//     from the builder (chunk_seg0); the warp then arrives on the stage's "empty" mbarrier.  No __syncthreads.
//   * a run still open at a chunk's end goes to carry_val[chunk] and is added to its segment by the carry fix-up.
// ------------------------------------------------------------------------------------------------
template <typename T>
struct SegStage {
    int col[kSegTile];
    T val[kSegTile];  // raw values; after a chunk has been walked, its segment sums (staging for the coalesced store)
};
struct SegDesc {      // what the producer tells the consumers about the tile in a stage
    int tile, cnt, pad0, pad1;
    int seg0[kSegChunks];
};

constexpr int kSegStages = 3;  // tile slices in flight: the current tile, the next one (its gathers are being issued) and one landing
constexpr int kSegThreads = kThreads + 32;  // 8 consumer warps + the producer warp

template <typename T>
constexpr size_t bseg_smem_bytes() { return kSegStages * (sizeof(SegStage<T>) + sizeof(SegDesc) + 16) + 16; }

template <typename T>
__device__ __forceinline__ void load8(const T *p, T (&v)[8]);
template <>
__device__ __forceinline__ void load8<double>(const double *p, double (&v)[8])
{
    const double2 *q = reinterpret_cast<const double2 *>(p);
#pragma unroll
    for (int k = 0; k < 4; ++k) { const double2 t = q[k]; v[2 * k] = t.x; v[2 * k + 1] = t.y; }
}
template <>
__device__ __forceinline__ void load8<float>(const float *p, float (&v)[8])
{
    const float4 *q = reinterpret_cast<const float4 *>(p);
#pragma unroll
    for (int k = 0; k < 2; ++k) { const float4 t = q[k]; v[4 * k] = t.x; v[4 * k + 1] = t.y; v[4 * k + 2] = t.z; v[4 * k + 3] = t.w; }
}
__device__ __forceinline__ void load8i(const int *p, int (&c)[8])
{
    const int4 *q = reinterpret_cast<const int4 *>(p);
    const int4 a = q[0], b = q[1];
    c[0] = a.x; c[1] = a.y; c[2] = a.z; c[3] = a.w; c[4] = b.x; c[5] = b.y; c[6] = b.z; c[7] = b.w;
}
__device__ __forceinline__ void mbar_arrive(uint64_t *bar)
{
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_addr(bar)) : "memory");
}

template <typename T, int MINB>
__global__ void __launch_bounds__(kSegThreads, MINB)
bseg_kernel(int tile_lo, int tile_hi, int pf_on, int *__restrict__ next_tile, const int4 *__restrict__ tile_ent,
            const int *__restrict__ chunk_seg0, const int *__restrict__ bcol, const T *__restrict__ bval,
            const T *__restrict__ x, T *__restrict__ seg_val, T *__restrict__ carry_val, int *__restrict__ carry_row)
{
    extern __shared__ __align__(128) unsigned char seg_smem[];
    SegStage<T> *stage = reinterpret_cast<SegStage<T> *>(seg_smem);
    SegDesc *desc = reinterpret_cast<SegDesc *>(seg_smem + kSegStages * sizeof(SegStage<T>));
    uint64_t *full = reinterpret_cast<uint64_t *>(desc + kSegStages);  // [3] slices + descriptor have landed
    uint64_t *empty = full + kSegStages;                                // [3] all eight consumer warps are done with the stage

    const uint64_t pl = policy_evict_last(), pf = policy_evict_first();
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tile_lo + (int)blockIdx.x >= tile_hi) return;
    if (tid == 0) {
        for (int k = 0; k < kSegStages; ++k) { mbar_init(&full[k], 1); mbar_init(&empty[k], kSegChunks); }
    }
    __syncthreads();

    if (warp == kSegChunks) {
        // ---------------- producer ----------------
        if (lane != 0) return;
        for (int k = 0;; ++k) {
            const int s = k % kSegStages;
            // the first kSegStages tickets of a CTA are implicit, the rest come from the counter (reset by the host)
            int t = k < kSegStages ? tile_lo + (int)blockIdx.x + k * (int)gridDim.x : tile_lo + atomicAdd(next_tile, 1);
            if (t > tile_hi) t = tile_hi;
            int4 te = make_int4(0, 0, 0, 0);
            int4 sa = make_int4(0, 0, 0, 0), sb = sa;
            if (t < tile_hi) {
                te = tile_ent[t];
                const int4 *q = reinterpret_cast<const int4 *>(chunk_seg0 + (size_t)t * kSegChunks);
                sa = q[0];
                sb = q[1];
            }
            if (k >= kSegStages) mbar_wait(&empty[s], (uint32_t)(((k / kSegStages) - 1) & 1));
            SegDesc &d = desc[s];
            d.tile = t; d.cnt = te.y;
            d.seg0[0] = sa.x; d.seg0[1] = sa.y; d.seg0[2] = sa.z; d.seg0[3] = sa.w;
            d.seg0[4] = sb.x; d.seg0[5] = sb.y; d.seg0[6] = sb.z; d.seg0[7] = sb.w;
            if (t >= tile_hi) {  // end marker: the consumers stop at a stage with cnt == 0
                mbar_arrive(&full[s]);
                break;
            }
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");  // the consumers' staging writes before the bulk copy lands
            const uint32_t cnt4 = (uint32_t)(te.y + 3) & ~3u;  // the arrays carry slack: up to 3 entries past the tile are readable
            mbar_expect_tx(&full[s], cnt4 * (uint32_t)(sizeof(int) + sizeof(T)));
            bulk_load(stage[s].col, bcol + te.x, cnt4 * (uint32_t)sizeof(int), &full[s], pf);
            bulk_load(stage[s].val, bval + te.x, cnt4 * (uint32_t)sizeof(T), &full[s], pf);
            if (pf_on && te.w > 0)  // (pf_on: x is 16-byte aligned) the tile's share of the next band's x slice -> L2, evict-last
                asm volatile("cp.async.bulk.prefetch.L2.global.L2::cache_hint [%0], %1, %2;"
                             ::"l"(x + te.z), "r"((uint32_t)(te.w * (int)sizeof(T))), "l"(pl) : "memory");
        }
        return;
    }

    // ---------------- consumers: warp w owns entries [256 w, 256 w + 256) of every tile ----------------
    const int b0 = warp * kSegChunk + lane * kSegIpt;
    int slot = 0;
    bool done = false;

    // gathers of this lane's 8 entries of the tile in stage s (cnt entries in the tile); f = their segment-end bits
    auto gather = [&](int s, int cnt, unsigned &f, T (&g)[8]) {
        int c[8];
        load8i(stage[s].col + b0, c);
        f = 0;
#pragma unroll
        for (int k = 0; k < kSegIpt; ++k) {
            g[k] = (b0 + k < cnt) ? ldg_x(x + (c[k] & 0x7fffffff), pl) : (T)0;
            f |= (c[k] < 0 ? 1u : 0u) << k;  // all that is kept of the column indices
        }
    };

    auto step = [&](unsigned f_use, T (&g_use)[8], unsigned &f_pre, T (&g_pre)[8]) {
        const int cur = slot % kSegStages, nxt = (slot + 1) % kSegStages;
        const SegDesc &d = desc[cur];
        const int cnt = d.cnt;
        if (cnt == 0) { done = true; return; }  // end marker
        const int tile = d.tile, seg0 = d.seg0[warp];
        // the next tile: wait for its slices, issue this lane's gathers (they fly during the walk below)
        mbar_wait(&full[nxt], (uint32_t)(((slot + 1) / kSegStages) & 1));
        const int cn = desc[nxt].cnt;
        T v[8];
        load8<T>(stage[cur].val + b0, v);
        if (cn > 0) gather(nxt, cn, f_pre, g_pre);

        int nvalid = cnt - b0;
        nvalid = nvalid < 0 ? 0 : (nvalid > kSegIpt ? kSegIpt : nvalid);
        unsigned closed = 0;
        T run = 0;
#pragma unroll
        for (int k = 0; k < kSegIpt; ++k) {
            if (k < nvalid) {
                run = fma_t(v[k], g_use[k], run);
                if ((f_use >> k) & 1u) { v[k] = run; run = 0; closed |= 1u << k; }  // v[k] now holds the segment sum
            }
        }
        // warp-wide segmented scan over (segments closed, run still open at the lane's end): a lane that closed at least
        // one segment resets the run.  Fixed evaluation order (Kogge-Stone).
        int c = __popc(closed);
        T w = run;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const int cl = __shfl_up_sync(kFull, c, o);
            const T wl = __shfl_up_sync(kFull, w, o);
            if (lane >= o) {
                if (c == 0) w = wl + w;
                c += cl;
            }
        }
        int ex_c = __shfl_up_sync(kFull, c, 1);
        T ex_v = __shfl_up_sync(kFull, w, 1);
        if (lane == 0) { ex_c = 0; ex_v = 0; }
        const int total = __shfl_sync(kFull, c, 31);
        const T tail = __shfl_sync(kFull, w, 31);
        // the chunk's segment sums, in order, staged over its own (dead) raw values, then one coalesced streaming write
        __syncwarp();  // every lane has read its raw values
        T *s_out = stage[cur].val + warp * kSegChunk;
        bool first_close = true;
#pragma unroll
        for (int k = 0; k < kSegIpt; ++k) {
            if ((closed >> k) & 1u) {
                T o = v[k];
                if (first_close) { o = ex_v + o; first_close = false; }  // the part of the segment that sits in the preceding lanes
                s_out[ex_c + __popc(closed & ((1u << k) - 1u))] = o;
            }
        }
        __syncwarp();
        for (int j = lane; j < total; j += 32) stg_stream(seg_val + (size_t)seg0 + j, s_out[j], pf);
        // is a segment still open at the chunk's end?  The lane that owns the chunk's last valid entry knows.
        {
            const int chunk_valid = min(max(cnt - warp * kSegChunk, 0), kSegChunk);
            const int owner = chunk_valid > 0 ? (chunk_valid - 1) / kSegIpt : 0;
            const int last_k = chunk_valid > 0 ? (chunk_valid - 1) % kSegIpt : 0;
            const unsigned owner_closed = __shfl_sync(kFull, closed, owner);
            if (lane == 0) {
                const bool open = chunk_valid > 0 && ((owner_closed >> last_k) & 1u) == 0;
                carry_row[(size_t)tile * kSegChunks + warp] = open ? seg0 + total : -1;
                carry_val[(size_t)tile * kSegChunks + warp] = open ? tail : (T)0;
            }
        }
        __syncwarp();  // the staging area has been read
        if (lane == 0) mbar_arrive(&empty[cur]);
        ++slot;
    };

    unsigned f_a = 0, f_b = 0;
    T g_a[8], g_b[8];
    mbar_wait(&full[0], 0);
    gather(0, desc[0].cnt, f_a, g_a);  // (cnt > 0: the CTA has at least one tile)
    while (true) {
        step(f_a, g_a, f_b, g_b);
        if (done) break;
        step(f_b, g_b, f_a, g_a);
        if (done) break;
    }
}

// ------------------------------------------------------------------------------------------------
// pass 2: y[r] = sum over the bands of row r's segment sums, in band order.  One lane per row, no shared memory:
// gbase[group][band] is the position of the group's first segment sum in band b's list (one coalesced load per
// warp, lane b keeps band b's), a ballot over the band's mask bit + popc of the lower lanes ranks the row, and the
// (predicated) loads of a band are coalesced: the segment sums of a row group are neighbours in the band's list.
// (A ballot-free variant -- a rank byte per segment, every lane walking its own set bits -- was measured: 40 % fewer
// instructions but 1.8x the DRAM traffic, because lanes then read different bands in the same instruction.)
// ------------------------------------------------------------------------------------------------
template <typename T>
__device__ __forceinline__ void merge_half(unsigned mk, int base, unsigned lt, const T *__restrict__ seg_val, T &sum)
{
    // fully unrolled over 32 mask bits in batches of 8 loads; bits of bands that do not exist are never set
#pragma unroll
    for (int b0 = 0; b0 < 32; b0 += 8) {
        if (!__any_sync(kFull, mk & (0xffu << b0))) continue;  // (warp-uniform) nobody has a segment in these 8 bands
        T v[8];
#pragma unroll
        for (int k = 0; k < 8; ++k) {
            const bool bit = mk & (1u << (b0 + k));
            const unsigned bal = __ballot_sync(kFull, bit);
            const unsigned pos = (unsigned)__shfl_sync(kFull, base, b0 + k) + (unsigned)__popc(bal & lt);
            v[k] = bit ? __ldcs(seg_val + pos) : (T)0;  // (a C++ load: the compiler predicates it)
        }
#pragma unroll
        for (int k = 0; k < 8; ++k)
            if (mk & (1u << (b0 + k))) sum += v[k];
    }
}

template <typename T, typename MaskT, typename Store>
__device__ __forceinline__ void bseg_merge_body(unsigned tid, int row0, int m, int bands,
                                                const MaskT *__restrict__ mask, const int *__restrict__ gbase,
                                                const T *__restrict__ seg_val, const Store &store)
{
    const int lane = tid & 31;
    const long long g = row0 / 32 + (((long long)blockIdx.x * kThreads + tid) >> 5);  // row0: a multiple of 32
    const long long r = g * 32 + lane;
    if (g * 32 >= m) return;
    const MaskT mk = r < m ? __ldcs(mask + r) : (MaskT)0;
    const int base_lo = lane < bands ? __ldcs(gbase + (size_t)g * bands + lane) : 0;
    const unsigned lt = (1u << lane) - 1u;
    T sum = 0;
    merge_half<T>((unsigned)mk, base_lo, lt, seg_val, sum);
    if (sizeof(MaskT) == 8) {
        const int base_hi = lane + 32 < bands ? __ldcs(gbase + (size_t)g * bands + 32 + lane) : 0;
        merge_half<T>((unsigned)((unsigned long long)mk >> 32), base_hi, lt, seg_val, sum);
    }
    // the old y is loaded after the merge, not before it: held across the merge it costs the fp64 / 64-band kernel 8
    // registers (40 instead of 32) and a quarter of its warps, for every beta
    if (r < m) store.put(r, sum, store.early(true, r));
}

template <typename T, typename MaskT, bool PEERS>
__global__ void __launch_bounds__(kThreads)
bseg_merge_kernel(int row0, int m, int bands, const MaskT *__restrict__ mask, const int *__restrict__ gbase,
                  const T *__restrict__ seg_val, T *__restrict__ y, const PeerList<T> peers)
{
    bseg_merge_body<T>(threadIdx.x, row0, m, bands, mask, gbase, seg_val, PeerStore<PEERS, T>{y, peers});
}

// spmv_b200_spmv_axpby on a band-segment handle: pass 2, scaled
template <typename T, typename MaskT>
__global__ void __launch_bounds__(kThreads)
bseg_merge_axpby_kernel(int row0, int m, int bands, const MaskT *__restrict__ mask, const int *__restrict__ gbase,
                        const T *__restrict__ seg_val, const ScaledStore<T> store)
{
    bseg_merge_body<T>(threadIdx.x, row0, m, bands, mask, gbase, seg_val, store);
}

}  // namespace sb
