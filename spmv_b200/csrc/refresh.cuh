// refresh.cuh -- new values for a handle's device layouts without rebuilding them (option "refresh",
// spmv_b200_set_values).  Create keeps, next to every value array it stores, a source map: map[slot] = k + 1 when the
// slot holds the caller's Matrix_Val[k], 0 for a padding slot.  The maps are made by the builders' own value-moving
// kernels, run a second time with T = int over the caller's positions (spmv_b200.cu: build_map), so a map cannot
// disagree with the layout it describes.  A refresh is then one gather per stored slot, all arrays in one launch.
#pragma once
#include "common.cuh"

namespace sb {

constexpr int kRefreshMaxTargets = 4;  // upload under "reorder" or band-major copy, + SELL or CSR5; or band segments

struct RefreshTarget {
    void *dst;           // value array of a layout
    const int *map;      // its source map [count]
    long long count;     // slots to write; the allocation's slack behind them is left alone
    long long quad0;     // first thread of this target in the launch (4 slots per thread)
};
struct RefreshTable {
    int n;
    RefreshTarget t[kRefreshMaxTargets];
};

#ifdef __CUDACC__
__device__ __forceinline__ int4 ldg_stream4(const int *p, uint64_t pol)
{
    int4 r;
    asm volatile("ld.global.nc.L1::no_allocate.L2::cache_hint.v4.s32 {%0, %1, %2, %3}, [%4], %5;"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p), "l"(pol));
    return r;
}

__device__ __forceinline__ void stg_stream4(double *p, double a, double b, double c, double d)
{
    __stcs((double2 *)p, make_double2(a, b));
    __stcs((double2 *)p + 1, make_double2(c, d));
}
__device__ __forceinline__ void stg_stream4(float *p, float a, float b, float c, float d)
{
    __stcs((float4 *)p, make_float4(a, b, c, d));
}

// the caller's value k for map entry k + 1, +0.0 for padding (the bits the builders' zero padding has)
template <typename T>
__device__ __forceinline__ T refresh_value(const T *__restrict__ src, int k1)
{
    return k1 ? __ldg(src + (k1 - 1)) : T(0);  // L1-allocating: neighbouring slots of a row share src sectors
}

// dst[s] = map[s] ? src[map[s] - 1] : 0 for every slot of every target.  Each thread owns 4 consecutive slots of one
// target: the map is read as one int4 (streamed, L2 evict-first), the 4 values are stored as one vector (streaming).
// Allocations start 256-byte aligned, so a full quad is aligned; a target's last, partial quad goes scalar.
template <typename T>
__global__ void __launch_bounds__(kThreads) value_refresh_kernel(const RefreshTable tab, const T *__restrict__ src)
{
    const long long q = (long long)blockIdx.x * kThreads + threadIdx.x;
    // which target: the last one starting at or before q (constant indices only -- a dynamically indexed
    // kernel-parameter array would be copied to local memory)
    T *dst = nullptr;
    const int *map = nullptr;
    long long count = 0, q0 = 0;
#pragma unroll
    for (int i = 0; i < kRefreshMaxTargets; ++i) {
        if (i < tab.n && q >= tab.t[i].quad0) {
            dst = (T *)tab.t[i].dst;
            map = tab.t[i].map;
            count = tab.t[i].count;
            q0 = tab.t[i].quad0;
        }
    }
    const long long s = 4 * (q - q0);
    if (!dst || s >= count) return;
    if (s + 4 <= count) {
        const int4 k = ldg_stream4(map + s, policy_evict_first());
        stg_stream4(dst + s, refresh_value(src, k.x), refresh_value(src, k.y), refresh_value(src, k.z), refresh_value(src, k.w));
    } else {
        for (long long j = s; j < count; ++j) dst[j] = refresh_value(src, map[j]);
    }
}

// map[i] = i + 1: the caller's order itself (the source of a builder that reads the caller's CSR unpermuted)
__global__ void map_iota_kernel(int n, int *__restrict__ map)
{
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) map[i] = i + 1;
}
#endif  // __CUDACC__

}  // namespace sb
