// generators.cu -- on-device synthetic CSR matrices (SURVEY.md 8d), bit-identical to
// spmv_b200/matrices.py.  They stand in for the input stage of the reference's sample driver
// (src/samples/test_spmv.c:158-209: load, overwrite values with rand()%8*0.125, X = 1) so that the
// multi-GB BASELINE.json matrices are produced where they are consumed.
#include <cub/device/device_scan.cuh>
#include <cub/device/device_radix_sort.cuh>

#include "common.cuh"

namespace sb {

__host__ __device__ __forceinline__ unsigned long long splitmix64(unsigned long long z)
{
    z += 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}
constexpr unsigned long long kValSalt = 0x5A17ED0000000000ull;
constexpr unsigned long long kXSalt = 0x0C0FFEE000000000ull;

template <typename T>
__device__ __forceinline__ T hashed_value(unsigned long long seed, unsigned long long pos, int eighths)
{
    const unsigned long long h = splitmix64(seed + kValSalt + pos);
    const double k = (double)(h & 7ull);
    return (T)((eighths ? k : k + 1.0) * 0.125);
}

// ---- stencils ------------------------------------------------------------------------------------
// kind 0: 5-point on (d0, d1); kind 1: 27-point on (d0, d1, d2).  Neighbour k in ascending column order.
__device__ __forceinline__ long long stencil_neighbor(int kind, int d0, int d1, int d2, long long idx, int k)
{
    if (kind == 0) {
        const int i = (int)(idx / d1), j = (int)(idx % d1);
        const int di[5] = {-1, 0, 0, 0, 1}, dj[5] = {0, -1, 0, 1, 0};
        const int a = i + di[k], b = j + dj[k];
        if (a < 0 || a >= d0 || b < 0 || b >= d1) return -1;
        return (long long)a * d1 + b;
    }
    const int c = (int)(idx % d2), b = (int)((idx / d2) % d1), a = (int)(idx / ((long long)d1 * d2));
    const int da = k / 9 - 1, db = (k / 3) % 3 - 1, dc = k % 3 - 1;
    const int aa = a + da, bb = b + db, cc = c + dc;
    if (aa < 0 || aa >= d0 || bb < 0 || bb >= d1 || cc < 0 || cc >= d2) return -1;
    return ((long long)aa * d1 + bb) * d2 + cc;
}

__global__ void stencil_count_kernel(int kind, int d0, int d1, int d2, int m, int *__restrict__ cnt)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r > m) return;
    int c = 0;
    if (r < m) {
        const int nk = kind == 0 ? 5 : 27;
        for (int k = 0; k < nk; ++k) c += stencil_neighbor(kind, d0, d1, d2, r, k) >= 0;
    }
    cnt[r] = c;
}

template <typename T>
__global__ void stencil_fill_kernel(int kind, int d0, int d1, int d2, int m, const int *__restrict__ rowptr,
                                    int *__restrict__ col, T *__restrict__ val)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r >= m) return;
    const int nk = kind == 0 ? 5 : 27;
    const T diag = kind == 0 ? (T)4 : (T)26;
    int p = rowptr[r];
    for (int k = 0; k < nk; ++k) {
        const long long c = stencil_neighbor(kind, d0, d1, d2, r, k);
        if (c >= 0) {
            col[p] = (int)c;
            val[p] = (c == r) ? diag : (T)-1;
            ++p;
        }
    }
}

// ---- uniform random --------------------------------------------------------------------------------
constexpr int kMaxRowK = 64;
template <typename T>
__global__ void uniform_kernel(int m, int n, int k, unsigned long long seed, long long row0, int eighths,
                               int *__restrict__ rowptr, int *__restrict__ col, T *__restrict__ val)
{
    const int r = blockIdx.x * blockDim.x + threadIdx.x;
    if (r > m) return;
    rowptr[r] = r * k;
    if (r == m) return;
    int c[kMaxRowK];
    const unsigned long long base = (unsigned long long)(row0 + r) * (unsigned long long)k;
    for (int j = 0; j < k; ++j) {
        const int v = (int)((splitmix64(seed + base + j) >> 11) % (unsigned long long)n);
        int i = j;  // insertion sort, ascending, duplicates kept
        while (i > 0 && c[i - 1] > v) { c[i] = c[i - 1]; --i; }
        c[i] = v;
    }
    const long long out = (long long)r * k;
    for (int j = 0; j < k; ++j) {
        col[out + j] = c[j];
        val[out + j] = hashed_value<T>(seed, base + j, eighths);
    }
}

// ---- R-MAT ----------------------------------------------------------------------------------------
__global__ void rmat_edges_kernel(long long edges, int scale, unsigned long long seed, double ta, double tab,
                                  double tabc, unsigned long long *__restrict__ keys)
{
    const long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (e >= edges) return;
    unsigned long long row = 0, colv = 0;
    for (int lvl = 0; lvl < scale; ++lvl) {
        const unsigned long long h = splitmix64(seed + (unsigned long long)e * (unsigned long long)scale + lvl);
        const double r = (double)(h >> 11) * (1.0 / 9007199254740992.0);
        const unsigned long long rb = r >= tab;
        const unsigned long long cb = ((r >= ta) && (r < tab)) || (r >= tabc);
        row = (row << 1) | rb;
        colv = (colv << 1) | cb;
    }
    keys[e] = (row << 32) | colv;
}

template <typename T>
__global__ void rmat_finish_kernel(long long edges, int m, unsigned long long seed,
                                   const unsigned long long *__restrict__ keys, int *__restrict__ rowptr,
                                   int *__restrict__ col, T *__restrict__ val)
{
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < edges) {
        col[i] = (int)(keys[i] & 0xFFFFFFFFull);
        val[i] = hashed_value<T>(seed, (unsigned long long)i, 0);
    }
    if (i <= m) {  // rowptr[i] = first edge whose row is >= i
        const unsigned long long key = (unsigned long long)i << 32;
        long long lo = 0, hi = edges;
        while (lo < hi) {
            const long long mid = (lo + hi) >> 1;
            if (keys[mid] < key) lo = mid + 1; else hi = mid;
        }
        rowptr[i] = (int)lo;
    }
}

template <typename T>
__global__ void gen_x_kernel(long long n, unsigned long long seed, int ones, T *__restrict__ x)
{
    const long long j = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n) return;
    if (ones) { x[j] = (T)1; return; }
    const unsigned long long h = splitmix64(seed + kXSalt + (unsigned long long)j);
    x[j] = (T)(0.5 + (double)(h % 1000ull) / 1000.0);
}

static inline unsigned grid_for(long long n) { return (unsigned)((n + 255) / 256); }

static bool alloc_csr(spmv_b200_csr *out, int m, int n, long long nnz, unsigned long size)
{
    memset(out, 0, sizeof(*out));
    out->m = m; out->n = n; out->nnz = nnz; out->size = size;
    SB_TRY(cudaMalloc((void **)&out->RowPtr, ((size_t)m + 1 + 8) * sizeof(int)));
    SB_TRY(cudaMalloc((void **)&out->ColIdx, ((size_t)nnz + 8) * sizeof(int)));
    SB_TRY(cudaMalloc(&out->Val, ((size_t)nnz + 8) * size));
    return true;
}

// a generator's failure exit once *out may hold allocations: *out is freed and zeroed
static int gen_failed(spmv_b200_csr *out)
{
    spmv_b200_csr_free(out);
    return -1;
}

static int gen_stencil(int kind, int d0, int d1, int d2, unsigned long size, spmv_b200_csr *out)
{
    const long long m64 = (long long)d0 * d1 * (kind ? d2 : 1);
    if (!out || d0 < 1 || d1 < 1 || d2 < 1 || m64 > 0x7fffffffLL / 32) { set_error("bad stencil shape"); return -1; }
    const int m = (int)m64;
    memset(out, 0, sizeof(*out));
    DeviceArray<int> cnt, rp;
    DeviceArray<unsigned char> tmp;
    if (!cnt.alloc((size_t)m + 1) || !rp.alloc((size_t)m + 1)) return -1;
    stencil_count_kernel<<<grid_for(m + 1), 256>>>(kind, d0, d1, d2, m, cnt);
    size_t bytes = 0;
    int nnz = 0;
    if (!SB_CUDA(cub::DeviceScan::ExclusiveSum(nullptr, bytes, cnt.get(), rp.get(), m + 1)) || !tmp.alloc(bytes) ||
        !SB_CUDA(cub::DeviceScan::ExclusiveSum(tmp.get(), bytes, cnt.get(), rp.get(), m + 1)) ||
        !SB_CUDA(cudaMemcpy(&nnz, rp + m, sizeof(int), cudaMemcpyDeviceToHost)))
        return -1;
    if (!alloc_csr(out, m, m, nnz, size) ||
        !SB_CUDA(cudaMemcpy(out->RowPtr, rp, ((size_t)m + 1) * sizeof(int), cudaMemcpyDeviceToDevice)))
        return gen_failed(out);
    if (size == 8) stencil_fill_kernel<double><<<grid_for(m), 256>>>(kind, d0, d1, d2, m, out->RowPtr, out->ColIdx, (double *)out->Val);
    else stencil_fill_kernel<float><<<grid_for(m), 256>>>(kind, d0, d1, d2, m, out->RowPtr, out->ColIdx, (float *)out->Val);
    if (!SB_CUDA(cudaGetLastError()) || !SB_CUDA(cudaDeviceSynchronize())) return gen_failed(out);
    return 0;
}

}  // namespace sb

using namespace sb;

extern "C" {

int spmv_b200_gen_laplacian2d(int nx, int ny, unsigned long size, spmv_b200_csr *out)
{
    return gen_stencil(0, nx, ny, 1, size == 8 ? 8 : 4, out);
}

int spmv_b200_gen_stencil27(int nx, int ny, int nz, unsigned long size, spmv_b200_csr *out)
{
    return gen_stencil(1, nx, ny, nz, size == 8 ? 8 : 4, out);
}

int spmv_b200_gen_uniform(int m, int n, int k, unsigned long long seed, long long row0, int eighths,
                          unsigned long size, spmv_b200_csr *out)
{
    size = size == 8 ? 8 : 4;
    if (!out || m < 0 || n < 1 || k < 1 || k > kMaxRowK || (long long)m * k > 0x7fffffffLL - 8192) { set_error("bad uniform shape"); return -1; }
    if (!alloc_csr(out, m, n, (long long)m * k, size)) return gen_failed(out);
    if (size == 8) uniform_kernel<double><<<grid_for(m + 1), 256>>>(m, n, k, seed, row0, eighths, out->RowPtr, out->ColIdx, (double *)out->Val);
    else uniform_kernel<float><<<grid_for(m + 1), 256>>>(m, n, k, seed, row0, eighths, out->RowPtr, out->ColIdx, (float *)out->Val);
    if (!SB_CUDA(cudaGetLastError()) || !SB_CUDA(cudaDeviceSynchronize())) return gen_failed(out);
    return 0;
}

int spmv_b200_gen_rmat(int scale, int edge_factor, unsigned long long seed, unsigned long size, spmv_b200_csr *out)
{
    size = size == 8 ? 8 : 4;
    if (!out || scale < 1 || scale > 30 || edge_factor < 1) { set_error("bad rmat shape"); return -1; }
    const int m = 1 << scale;
    const long long edges = (long long)m * edge_factor;
    if (edges > 0x7fffffffLL - 8192) { set_error("rmat too large"); return -1; }
    DeviceArray<unsigned long long> keys, sorted;
    DeviceArray<unsigned char> tmp;
    if (!alloc_csr(out, m, m, edges, size) || !keys.alloc((size_t)edges) || !sorted.alloc((size_t)edges)) return gen_failed(out);
    const double a = 0.57, b = 0.19, c = 0.19;
    rmat_edges_kernel<<<grid_for(edges), 256>>>(edges, scale, seed, a, a + b, a + b + c, keys);
    size_t bytes = 0;
    cub::DeviceRadixSort::SortKeys(nullptr, bytes, keys.get(), sorted.get(), (int)edges, 0, 32 + scale);
    bool ok = tmp.alloc(bytes) && SB_CUDA(cub::DeviceRadixSort::SortKeys(tmp.get(), bytes, keys.get(), sorted.get(), (int)edges, 0, 32 + scale));
    if (ok) {
        const long long n = edges > m + 1 ? edges : m + 1;
        if (size == 8) rmat_finish_kernel<double><<<grid_for(n), 256>>>(edges, m, seed, sorted, out->RowPtr, out->ColIdx, (double *)out->Val);
        else rmat_finish_kernel<float><<<grid_for(n), 256>>>(edges, m, seed, sorted, out->RowPtr, out->ColIdx, (float *)out->Val);
        ok = SB_CUDA(cudaGetLastError()) && SB_CUDA(cudaDeviceSynchronize());
    }
    return ok ? 0 : gen_failed(out);
}

int spmv_b200_gen_x(void *device_dst, long long n, unsigned long long seed, int ones, unsigned long size)
{
    if (!device_dst || n < 0) return -1;
    if (n == 0) return 0;
    if (size == 8) gen_x_kernel<double><<<grid_for(n), 256>>>(n, seed, ones, (double *)device_dst);
    else gen_x_kernel<float><<<grid_for(n), 256>>>(n, seed, ones, (float *)device_dst);
    return (SB_CUDA(cudaGetLastError()) && SB_CUDA(cudaDeviceSynchronize())) ? 0 : -1;
}

void spmv_b200_csr_free(spmv_b200_csr *csr)
{
    if (!csr) return;
    if (csr->RowPtr) cudaFree(csr->RowPtr);
    if (csr->ColIdx) cudaFree(csr->ColIdx);
    if (csr->Val) cudaFree(csr->Val);
    memset(csr, 0, sizeof(*csr));
}

}  // extern "C"
