// reorder.cu -- locality reordering at create (SURVEY.md 8(f)-4): host code only.
//
// The reference has a compiled-out "level 3" hook (src/src_spmv/common.c:144-156, HyperGraphInterface.cpp:59-146):
// for square matrices create computes a symmetric permutation (METIS k-way parts sorted into blocks), rebuilds the
// CSR as A' = P A P^T, stores the permutation in handle->index (index[i] = original row at position i) and sets
// Level_3_opt_used; the caller then passes x' with x'[i] = x[index[i]] and scatters y[index[i]] = y'[i]
// (src/samples/test_spmv.c:95-101,130-137).  METIS is not vendored upstream and the option is off there.
//
// Here the same hook is filled by a reverse Cuthill-McKee ordering (breadth-first over the row adjacency, every
// component entered at its lowest-degree vertex, neighbours in ascending degree, whole order reversed): it pulls
// the non-zeros of matrices whose x fits L2 but whose rows are scattered towards the diagonal, which is what the
// gathers of the GPU kernels want (neighbouring rows then share sectors of x).  Everything below runs on the host
// arrays the caller hands to create; the device path is the ordinary one on the permuted matrix.
#include <algorithm>
#include <cstdint>
#include <cstring>
#include <numeric>
#include <vector>

#define SPMV_B200_NO_HOST_HEADERS 1
#include "../../include/spmv_b200.h"

namespace {

template <typename V>
void permute_values(int m, const int *rowptr, const int *col, const V *val, const int *index, const int *inv,
                    const int *rowptr_out, int *col_out, V *val_out)
{
    std::vector<std::pair<int, int>> tmp;  // (new column, original position): stable for duplicate columns
    for (int i = 0; i < m; ++i) {
        const int r = index[i];
        const int a = rowptr[r], b = rowptr[r + 1];
        tmp.clear();
        for (int j = a; j < b; ++j) tmp.emplace_back(inv[col[j]], j);
        std::sort(tmp.begin(), tmp.end());
        int d = rowptr_out[i];
        for (const auto &e : tmp) {
            col_out[d] = e.first;
            val_out[d] = val[e.second];
            ++d;
        }
    }
}

template <typename V>
int permute_csr(int m, const int *RowPtr, const int *ColIdx, const V *Val, const int *index, int *RowPtr_out, int *ColIdx_out,
                V *Val_out)
{
    if (m < 0 || !RowPtr || !index || !RowPtr_out) return -1;
    const int nnz = RowPtr[m] - RowPtr[0];
    if (nnz > 0 && (!ColIdx || !Val || !ColIdx_out || !Val_out)) return -1;
    std::vector<int> inv((size_t)m, -1);
    for (int i = 0; i < m; ++i) {
        if (index[i] < 0 || index[i] >= m || inv[index[i]] != -1) return -1;  // not a permutation
        inv[index[i]] = i;
    }
    for (int j = RowPtr[0]; j < RowPtr[m]; ++j)
        if (ColIdx[j] < 0 || ColIdx[j] >= m) return -1;  // a symmetric permutation needs a square pattern
    RowPtr_out[0] = 0;
    for (int i = 0; i < m; ++i) RowPtr_out[i + 1] = RowPtr_out[i] + (RowPtr[index[i] + 1] - RowPtr[index[i]]);
    permute_values<V>(m, RowPtr, ColIdx, Val, index, inv.data(), RowPtr_out, ColIdx_out, Val_out);
    return 0;
}

}  // namespace

namespace sb {

// Options "reorder" + "refresh": pos_out[d] = 1 + the caller's position of the entry A' stores at d (the source map of
// the permuted upload, refresh.cuh), placed exactly as spmv_b200_permute_csr places the values.
int permute_positions(int m, const int *RowPtr, const int *ColIdx, const int *index, int *RowPtr_out, int *ColIdx_out, int *pos_out)
{
    if (m < 0 || !RowPtr || RowPtr[m] < 0) return -1;
    std::vector<int> pos((size_t)RowPtr[m]);  // the values are read as Val[j], j in [RowPtr[0], RowPtr[m])
    std::iota(pos.begin(), pos.end(), 1);
    return permute_csr<int>(m, RowPtr, ColIdx, pos.data(), index, RowPtr_out, ColIdx_out, pos_out);
}

}  // namespace sb

extern "C" {

int spmv_b200_reorder(int m, const int *RowPtr, const int *ColIdx, int *index_out)
{
    if (m < 0 || !RowPtr || !index_out || (RowPtr[m] > RowPtr[0] && !ColIdx)) return -1;
    std::vector<int> deg((size_t)m), start((size_t)m);
    for (int i = 0; i < m; ++i) deg[i] = RowPtr[i + 1] - RowPtr[i];
    std::iota(start.begin(), start.end(), 0);
    std::stable_sort(start.begin(), start.end(), [&](int a, int b) { return deg[a] < deg[b]; });
    std::vector<unsigned char> seen((size_t)m, 0);
    std::vector<int> nbr;
    int head = 0, tail = 0;  // index_out doubles as the BFS queue
    for (int s = 0; s < m; ++s) {
        const int root = start[s];
        if (seen[root]) continue;
        seen[root] = 1;
        index_out[tail++] = root;
        while (head < tail) {
            const int u = index_out[head++];
            nbr.clear();
            for (int j = RowPtr[u]; j < RowPtr[u + 1]; ++j) {
                const int v = ColIdx[j];
                if (v >= 0 && v < m && !seen[v]) {
                    seen[v] = 1;
                    nbr.push_back(v);
                }
            }
            std::sort(nbr.begin(), nbr.end(), [&](int a, int b) { return deg[a] != deg[b] ? deg[a] < deg[b] : a < b; });
            for (int v : nbr) index_out[tail++] = v;
        }
    }
    std::reverse(index_out, index_out + m);
    return 0;
}

int spmv_b200_permute_csr(int m, const int *RowPtr, const int *ColIdx, const void *Val, unsigned long size,
                          const int *index, int *RowPtr_out, int *ColIdx_out, void *Val_out)
{
    if (size == sizeof(double))
        return permute_csr<double>(m, RowPtr, ColIdx, (const double *)Val, index, RowPtr_out, ColIdx_out, (double *)Val_out);
    return permute_csr<float>(m, RowPtr, ColIdx, (const float *)Val, index, RowPtr_out, ColIdx_out, (float *)Val_out);
}

}  // extern "C"
