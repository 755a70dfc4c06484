/*
 * spmv_b200.h -- non-breaking extensions next to the drop-in API of spmv.h.
 *
 * Nothing here exists in the reference; a client that only knows spmv.h never needs it.  These entry
 * points cover what moving the path to a GPU adds: stream control for device-resident x/y, error
 * retrieval (the reference API returns void everywhere), introspection of the device layouts for
 * bit-exact structure tests, the equal-nnz row partition used to shard a matrix across GPUs, and
 * on-device synthetic matrix generators so that multi-GB benchmark matrices never cross PCIe.
 *
 * Plain C ABI: pointers, sizes, ints.  No CUDA or torch types appear in any signature (a CUDA stream
 * is passed as void*).
 */
#ifndef SPMV_B200_EXT_H
#define SPMV_B200_EXT_H
#include <stddef.h>
#include "spmv.h"

#if defined(__cplusplus)
extern "C" {
#endif

#define SPMV_B200_VERSION 200 /* round 2 */

/* ---- errors ------------------------------------------------------------------------------------
 * The reference swallows every error (common.c:136,285; csr5_spmv.cpp:31-35).  Same void API here,
 * plus: the last failure message of the calling thread ("" when none). */
SPMV_B200_API int spmv_b200_version(void);
SPMV_B200_API const char *spmv_b200_last_error(void);
SPMV_B200_API void spmv_b200_clear_error(void);

/* ---- refreshing the values -------------------------------------------------------------------------
 * spmv() ignores its Matrix_Val argument: the values are part of the device layout built at create (the reference
 * re-reads the caller's array on every call for Serial / Parallel / Balanced*).  After changing values on a FIXED
 * pattern call spmv_b200_update_values(handle, Matrix_Val): the handle is rebuilt in place from the RowPtr / ColIdx
 * it borrowed at create and the values given (NULL = re-read the array given at create), same method, precision and
 * stream.  Costs one create.  Returns 0, or -1 (spmv_b200_last_error()). */
SPMV_B200_API int spmv_b200_update_values(spmv_Handle_t handle, void *Matrix_Val);
/* A handle created with option "refresh" = 1 can take new values without a rebuild: create then keeps, for every value
 * array it stores, a source map (4 bytes per stored slot: where in the caller's Matrix_Val, in the caller's order, the
 * value of that slot comes from).  spmv_b200_set_values(handle, Matrix_Val) then writes the new values into every layout
 * in place.  Matrix_Val holds nnz values of the handle's precision in the order of the ColIdx given at create (before
 * any option-"reorder" permutation), as a HOST or DEVICE pointer; NULL = re-read the array given at create (the
 * reference's usage: change that array in place, then call).  With an adopted device CSR only NULL or that same adopted
 * pointer is accepted: the library never writes the caller's arrays.
 * The call is stream-ordered on the handle's stream: every product enqueued before it uses the old values, every one
 * enqueued after it the new ones (device or host x / y, the pipelined host path, spmv_b200_spmv_bands /
 * spmv_b200_spmv_finish, y peers).  A DEVICE source (on the handle's device) returns without a host synchronisation
 * and allocates nothing; the caller keeps the array unchanged until the stream has passed the refresh, as for a device
 * x in spmv().  A HOST source has been copied out on return, so the caller may reuse the array at once; it goes
 * through a staging array of nnz values, allocated at the first such call and owned by the handle, unless the handle's
 * own CSR upload takes it as it is.  Afterwards every spmv() result is bit for bit what a handle newly created with
 * these values under the same options computes.  spmv_b200_info(h, "refreshable") says whether a handle can be
 * refreshed (0 without the option, or when a map could not be allocated at create; the handle still works).
 * m == 0 or nnz == 0: returns 0 and does nothing.  Returns 0, or -1 (spmv_b200_last_error()): NULL handle, failed
 * create, no option "refresh", another pointer than an adopted one, a device pointer on another device.
 * Refresh kernels are not counted by spmv_b200_launch_count(). */
SPMV_B200_API int spmv_b200_set_values(spmv_Handle_t handle, const void *Matrix_Val);

/* ---- scaled products ----------------------------------------------------------------------------------
 * y <- alpha * A x + beta * y, the update of a CG residual, a Jacobi or Chebyshev step, PageRank or a Lanczos step,
 * and what MKL's mkl_sparse_?_mv and cuSPARSE's cusparseSpMV compute.  With s = the y that spmv() on this handle writes
 * for this x, bit for bit, every row gets y[i] = fl(fl(alpha s[i]) + fl(beta y_old[i])): three roundings, no FMA, so
 * the result is reproducible on a CPU.  beta == 0: y[i] = fl(alpha s[i]) and the old y is never read (it may hold
 * anything, NaN included); alpha == 0: y[i] = fl(beta y_old[i]) and A and x are not read; both 0: every row +0.0.  So
 * alpha = 1, beta = 0 is exactly spmv().  fp32 handles round alpha and beta to float first.  nnz == 0 follows the rule
 * with s = +0; m == 0 does nothing.
 * x and y may be HOST or DEVICE pointers as in spmv() (option "pin_host" applies; the pipelined host path does not):
 * with device x and y the call is enqueued on the handle's stream, with a host y it is synchronous (and with beta != 0
 * the old y is uploaded first).  y peers (spmv_b200_set_y_peers) receive the scaled values.  x and y must not overlap.
 * The scaling is done by the kernel that stores each final y value -- the fold of the column bands, or the main kernel
 * of an unbanded CSR-vector, row-block or 8-column SELL handle -- at the cost of one read of the old y when beta != 0;
 * the other layouts (carry fix-ups, long-row list, row bins, SELL's 4-column flavour "sell_variant" 2, Method_Serial,
 * nnz == 0) write A x into a scratch array of m values, allocated at the first such call and owned by the handle, and
 * scale it in one more pass.
 * spmv_b200_info(h, "axpby_path") says which: 0 = scratch pass, 1 = main kernel, 2 = fold (option "axpby_fused" = 0
 * at create: always 0).  With device pointers the call can be captured in a CUDA graph after one call outside the
 * capture (which may allocate the scratch array).
 * Returns 0, or -1 (spmv_b200_last_error()): NULL handle, failed create, NULL y, NULL x with n > 0, or x == y (all
 * with y untouched), or a failed allocation or launch (a failed scratch allocation also leaves y untouched; the
 * handle keeps working). */
SPMV_B200_API int spmv_b200_spmv_axpby(spmv_Handle_t handle, double alpha, const void *x, double beta, void *y);

/* y <- alpha * A x + beta * y as spmv_b200_spmv_axpby writes it, bit for bit and under all of its rules (rounding,
 * beta == 0 and alpha == 0, fp32 rounding alpha and beta to float first, host and device pointers, "pin_host", y peers
 * receiving the scaled values, x == y rejected), and *dot = sum over i of p_i = w[i] * y[i] over the y this call wrote:
 * the dot product a CG step (p . Ap), a Lanczos step (v . w) or a normalised power method (|y|^2, x . y) needs next,
 * taken by the kernel that stores each final y value instead of a second pass over y.
 * p_i is fl(w[i] y[i]) on fp64 handles (one rounding, no FMA) and the exact product of the two floats in double on fp32
 * handles; the sum is taken in double, and *dot is a double for both precisions.
 * w: m values of the handle's precision, on the host or the device.  w == y is the new y (so |y|^2 is
 * spmv_b200_spmv_axpby_dot(h, 1, x, 0, y, y, &d)); w == x is allowed on a square handle (CG's p . Ap; a host x is then
 * read from its staged copy); any other w must not overlap y.  A host w goes through a staging array of m values,
 * owned by the handle and allocated at its first use.
 * dot: a host or a device pointer to one double.  A device dot is written in stream order on the handle's stream,
 * without a host synchronisation (with device x, y and w the call is only enqueued, so a whole CG step can stay on the
 * device and be captured in a CUDA graph after one call outside the capture); with a host dot the call is synchronous.
 * Reproducible: identical inputs on one handle give the same bits in every call, on any stream and in graph replay (no
 * float atomics; one fixed summation tree: per CTA of 256 rows an xor butterfly over each warp and a fixed tree over the
 * 8 warp sums, then one CTA of 1024 threads that adds partials t, t + 1024, ... in order and halves in a fixed tree).
 * Accuracy: no product passes through more than L = 18 + ceil(P / 1024) additions, P <= m + 2 the number of CTA
 * partials, so |*dot - sum p_i| <= L 2^-53 sum |p_i|.
 * alpha == beta == 0: y = +0 without reading the old y, and *dot is taken over those zeros (NaN if w holds +-Inf or
 * NaN); nnz == 0 follows the rule; m == 0 writes *dot = +0 and nothing else.
 * spmv_b200_info(h, "dot_path") says where the dot is taken, with the encoding of "axpby_path": the same kernel as
 * spmv_b200_spmv_axpby, except band-segment handles, which take the scratch pass ("axpby_fused" = 0: always the scratch
 * pass).  The partials (one double per CTA) are owned by the handle, allocated at the first call.
 * Returns 0, or -1 (spmv_b200_last_error()): NULL handle, failed create, NULL y, NULL dot, NULL w, NULL x with n > 0,
 * x == y, w == x on a handle that is not square, w overlapping y without being y (all with y and *dot untouched), or a
 * failed allocation or launch. */
SPMV_B200_API int spmv_b200_spmv_axpby_dot(spmv_Handle_t handle, double alpha, const void *x, double beta, void *y,
                                           const void *w, double *dot);

/* y <- alpha * (A - sigma I) x + beta * y on a square handle (m == n), and optionally x . y and y . y over the y this
 * call wrote: one step of a Chebyshev iteration or smoother, a Chebyshev filter or the kernel polynomial method
 * (t_{k+1} = 2 ((A - c I) / e) t_k - t_{k-1}: alpha = 2 / e, sigma = c, beta = -1, x = t_k, y = t_{k-1} overwritten),
 * or of a normalised power method on A - sigma I (the Rayleigh quotient x . y and |y|^2), in the kernel that stores
 * each final y value instead of an axpy and two dot passes over x and y.
 * With s = the y that spmv() on this handle writes for this x, bit for bit, every row gets
 * y[i] = fl(fl(alpha fl(s[i] - fl(sigma x[i]))) + fl(beta y_old[i])): five roundings, no FMA, so the result is
 * reproducible on a CPU.  sigma == 0 skips the shift term entirely (s - fl(0 x) would turn a -0 into +0): the call then
 * writes spmv_b200_spmv_axpby's y, bit for bit.  Every rule of spmv_b200_spmv_axpby applies unchanged: beta == 0 never
 * reads the old y (y[i] = fl(alpha fl(s[i] - fl(sigma x[i])))); alpha == 0 reads neither A nor x for y and writes
 * fl(beta y_old[i]), or +0 when beta == 0; fp32 handles round alpha, beta and sigma to float first; nnz == 0 follows
 * the rule with s = +0; host and device x and y, "pin_host"; y peers receive the final values; x == y is rejected.
 * dots: NULL = no dots.  Otherwise a host or a device pointer to 2 doubles: dots[0] = sum over i of fl(x[i] y[i]) and
 * dots[1] = sum over i of fl(y[i] y[i]), over the y this call wrote, each with spmv_b200_spmv_axpby_dot's products
 * (one rounding in double on fp64 handles, exact on fp32), its one fixed summation order, its reproducibility and its
 * bound |dots[k] - sum p_i| <= L 2^-53 sum |p_i|, L = 18 + ceil(P / 1024), P <= m + 2.  So with sigma == 0, dots[0] and
 * dots[1] are, bit for bit, the *dot of spmv_b200_spmv_axpby_dot(h, alpha, x, beta, y, w, &d) with w = x and with
 * w = y.  With alpha == 0 and dots, x is read only for dots[0].  A device dots is written in stream order on the
 * handle's stream without a host synchronisation (with device x and y the call is only enqueued and can be captured
 * in a CUDA graph after one call outside the capture); with host dots the call is synchronous.  m == 0 writes dots +0,
 * +0 (when given) and nothing else.
 * The call takes the paths spmv_b200_info(h, "dot_path") reports, with or without dots.  The partials (two doubles per
 * CTA) and, for host dots, 2 device doubles are owned by the handle, allocated at their first use.
 * Returns 0, or -1 (spmv_b200_last_error()): NULL handle, failed create, a handle that is not square, NULL y, NULL x
 * with n > 0, x == y (all with y and dots untouched), or a failed allocation or launch. */
SPMV_B200_API int spmv_b200_spmv_shifted(spmv_Handle_t handle, double alpha, double sigma, const void *x, double beta,
                                         void *y, double *dots);

/* ---- streams -----------------------------------------------------------------------------------
 * spmv() with HOST x/y is synchronous (reference semantics).  With DEVICE x/y it is enqueued on the
 * handle's stream (default: the legacy default stream 0) and returns immediately. */
SPMV_B200_API void spmv_b200_set_stream(spmv_Handle_t handle, void *cuda_stream);
SPMV_B200_API void spmv_b200_sync(spmv_Handle_t handle);

/* ---- options (process-global, read when a handle is created) --------------------------------------
 * Also settable through the environment as SPMV_B200_<KEY IN CAPITALS>.  Keys:
 *   "sell_sigma"      sorting window of Method_SellCSigma (multiple of 32, <= 4096; default 256)
 *   "csr5_sigma"      nnz per lane of a CSR5 tile (4, 8 or 16; default 0 = 16, or 8 below 2^25 non-zeros)
 *   "block_nnz"       nnz per row block of Method_Balanced (default 512)
 *   "tile_items"      items per thread of the merge-path / equal-nnz tiles (4 or 8; default 8, any other value is 8)
 *   "tpr"             force threads-per-row of Method_Parallel (power of two <= 32; 0 = from mean)
 *   "x_bands"         column bands of the band-major layout that keeps the gathered slice of x inside L2
 *                     (0 = automatic from n and the L2 size, 1 = off, 2..64 forced); every method except
 *                     Method_Serial can run on the band-major copy
 *   "seg_bands"       column bands stored as band segments (entry lists sorted by row inside a band, segment sums
 *                     merged per row in a second pass), for matrices whose bands would hold fewer than 4 non-zeros
 *                     per row (0 = automatic, -1 = never, 2..64 forced); replaces the kernel of every method except
 *                     Method_Serial
 *   "seg_ctas"        persistent CTAs per SM of the band-segment pass 1 (2 = default, or 3); read at a handle's FIRST
 *                     band-segment launch, not at create
 *   "seg_prefetch"    L2 prefetch of the next band's slice of x in the band-segment pass 1 (0 = never, 1 = automatic
 *                     (default), 2 = always); read once per process, at the first band-segment launch; no effect on y
 *   "force_merge"     1 = Method_Balanced2 always runs the merge-path kernel (default: only when a row is
 *                     long enough to starve a row block, the reference's own Balanced2 -> Balanced rule)
 *   "sell_variant"    SELL kernel flavour: -1 = automatic (default: 2 on diagonal-local matrices, else 0),
 *                     0 = 8 columns per step / 40 registers, 2 = 4 columns per step / 32 registers (every warp slot filled)
 *   "sell_cap"        widest SELL slice in columns (default 1024); slices that would be mostly padding are
 *                     narrowed by a cost rule and the cut-off row tails go to the long-row path.  0 = the
 *                     reference's widths (every slice as wide as its longest row)
 *   "long_thr"        Method_Parallel leaves rows longer than this to the long-row path (0 = automatic:
 *                     256 x lanes-per-row clamped to [512, 4096]; < 0 = never)
 *   "row_bins"        1 (default) = Method_Parallel on short-row matrices that also have hub rows bins the rows by
 *                     length class (<= 8, <= 32, <= 128 entries: 1, 4, 16 lanes per row, one launch each; longer
 *                     rows on the long-row path); 0 = one lane-group size for all rows
 *   "pin_host"        1 (default) = a pageable HOST x or y (>= 1 MiB) that is passed to spmv() twice in a row is
 *                     page-locked in place (cudaHostRegister) so that its copies run at PCIe speed (3x on the
 *                     reference's sample driver, which reuses one X and one Y for every call); released when the
 *                     caller switches buffers and at clear / destroy.  The caller must not free such a buffer while
 *                     the handle lives.  0 = never touch the caller's pages
 *   "auto"            1 = every create whose Function is not Method_Serial picks the method itself from statistics it
 *                     gathers on the device (share of non-zeros in very long rows, mean row length, locality of the
 *                     column indices): Method_CSR5SPMV for power-law matrices, Method_Parallel for short diagonal-
 *                     local rows and small matrices, Method_SellCSigma otherwise -- the table of measured winners is
 *                     in DESIGN.md.  handle->spmvMethod then holds the method that runs, spmv_b200_info(h,
 *                     "auto_method") too.  0 (default) = run what Function says
 *   "pipeline"        1 (default) = spmv() with HOST x and y on a Method_Parallel handle overlaps the PCIe
 *                     copies with the kernels (x in pieces, y in row chunks); 0 = copy, run, copy
 *   "refresh"         1 = create also keeps a source map of every value array the handle stores, so that
 *                     spmv_b200_set_values can refresh the values in place (4 bytes per stored slot); 0 (default) = no
 *                     maps, create is unchanged
 *   "axpby_fused"     1 (default) = spmv_b200_spmv_axpby (_dot, _shifted) scales in the kernel that stores each final y
 *                     value where the layout has such a kernel; 0 = always A x into the scratch array, then one
 *                     scaling pass (the same y bits; for timing one against the other)
 * Returns 0, or -1 for an unknown key. */
SPMV_B200_API int spmv_b200_set_option(const char *key, long long value);
SPMV_B200_API long long spmv_b200_get_option(const char *key);

/* ---- introspection -----------------------------------------------------------------------------
 * spmv_b200_info: scalar facts about a handle.  Keys: "kernel" (internal kernel family, see
 * SPMV_B200_KERNEL_*), "requested", "m", "n", "nnz", "tpr", "parts", "tiles", "tile_items", "sigma", "banner",
 * "slices", "sell_variant" (0 or 2: the SELL kernel flavour that runs), "padded_nnz", "csr5_p", "csr5_sigma",
 * "csr5_num_offsets", "csr5_tail_start", "device", "has_empty_rows", "x_bands", "seg_bands", "segments", "seg_cross",
 * "seg_ctas" (persistent CTAs per SM of the band-segment pass 1; 0 until the handle's first launch), "band_cols",
 * "active_rows", "owns_csr", "released_csr",
 * "layout_fallbacks", "auto_method", "values_snapshotted", "refreshable", "pipeline", "dev_l2_bytes", "axpby_path" (where
 * spmv_b200_spmv_axpby scales: 0 = scratch pass, 1 = main kernel, 2 = fold), "dot_path" (the same for
 * spmv_b200_spmv_axpby_dot).  Returns -1 for an unknown key /
 * NULL handle.
 *
 * spmv_b200_structure: copy a device layout array to HOST memory.  Returns its size in bytes (call
 * with dst = NULL to size it), or -1.  Names: "splitter" (int[parts+1], a9), "ref_splitter"
 * (int[nthreads+1], a9 with the caller's nthreads), "tile_rows" (int[tiles+1]), "merge_coords"
 * (int[2*(tiles+1)]), "sell_perm" (int[banner], a13), "sell_width" (int[slices]), "sell_slice_ptr"
 * (long long[slices+1]), "sell_col" (int[padded]), "sell_val", "csr5_tile_ptr" (unsigned[p+1], a16),
 * "csr5_tile_desc" (unsigned[p*32], a17), "csr5_offset_ptr" (int[p+1]), "csr5_offsets" (int[num]),
 * "csr5_col" (int[nnz], a18), "csr5_val", "band_rowptr" (int[x_bands*m+1]), "band_col" (int[nnz]); band segments:
 * "seg_ptr" (int[K+1], first slot of every band), "seg_cnt" (int[K]), "seg_col" (unsigned[slots], bit 31 = last entry of
 * a segment), "seg_mask" (uint32 / uint64 [m]), "seg_gbase" (int[groups*K]), "seg_chunk_seg0" (int[tiles*8+1]). */
enum {
    SPMV_B200_KERNEL_NONE = 0,
    SPMV_B200_KERNEL_CSR_REFORDER = 1, /* Method_Serial   */
    SPMV_B200_KERNEL_CSR_VECTOR = 2,   /* Method_Parallel */
    SPMV_B200_KERNEL_ROW_BLOCKS = 3,   /* Method_Balanced */
    SPMV_B200_KERNEL_MERGE_PATH = 4,   /* Method_Balanced2 */
    SPMV_B200_KERNEL_NNZ_SPLIT = 5,    /* Method_Balanced_Yid */
    SPMV_B200_KERNEL_SELL = 6,         /* Method_SellCSigma */
    SPMV_B200_KERNEL_CSR5 = 7,         /* Method_CSR5SPMV */
    SPMV_B200_KERNEL_BAND_SEG = 8      /* any method but Method_Serial when x needs so many column bands that
                                          they are hyper-sparse (see "seg_bands") */
};
SPMV_B200_API long long spmv_b200_info(spmv_Handle_t handle, const char *key);
SPMV_B200_API long long spmv_b200_structure(spmv_Handle_t handle, const char *name, void *dst, size_t dst_bytes);

/* ---- method recommendation ("Matrix inspect and choose best method to run": an empty heading in the
 * reference's README.md:222) ---------------------------------------------------------------------------
 * Looks at the row-length distribution of a CSR (HOST RowPtr; pure host code, usable without a GPU) and
 * returns the SPMV_METHODS value whose GPU layout measured fastest on matrices of that shape: Method_CSR5SPMV
 * when more than a quarter of the non-zeros sit in rows much longer than the mean (power-law graphs),
 * Method_Parallel for small matrices (fewer than 8192 rows: nothing to amortise a layout build), otherwise
 * Method_SellCSigma.  Returns -1 on invalid arguments. */
SPMV_B200_API int spmv_b200_recommend_method(int m, const int *RowPtr);

/* ---- locality reordering at create (the reference's compiled-out level-3 hook, common.c:144-156) ----------------------
 * Option "reorder" = 1 (SPMV_B200_REORDER=1): for a square matrix with more than 8096 rows and 100000 non-zeros given
 * as HOST arrays (the reference's own condition, common.c:145), create computes a symmetric permutation, builds the
 * device layout of A' = P A P^T, stores the permutation in handle->index (malloc'ed, m+1 ints, index[i] = original row at
 * position i; freed by clear / destroy) and sets handle->Level_3_opt_used.  The caller then follows the reference's
 * protocol (src/samples/test_spmv.c:95-101,130-137): x'[i] = x[index[i]] goes in, y[index[i]] = y'[i] comes out.
 * The two host functions below are what create uses; pure host code, usable without a GPU:
 *   spmv_b200_reorder      reverse Cuthill-McKee over the row adjacency (components entered at their lowest-degree
 *                          vertex); index_out[m];
 *   spmv_b200_permute_csr  A' = P A P^T for a square CSR: row i of A' is row index[i] of A with column c renamed to the
 *                          position of c, columns ascending inside a row (duplicates keep their order).
 * Return 0, or -1 (bad arguments, index not a permutation, column outside [0, m)). */
SPMV_B200_API int spmv_b200_reorder(int m, const int *RowPtr, const int *ColIdx, int *index_out);
SPMV_B200_API int spmv_b200_permute_csr(int m, const int *RowPtr, const int *ColIdx, const void *Val, unsigned long size,
                                        const int *index, int *RowPtr_out, int *ColIdx_out, void *Val_out);

/* kernels launched by this process on the spmv() path since load (for benchmark accounting) */
SPMV_B200_API unsigned long long spmv_b200_launch_count(void);
/* device allocations the library currently holds for its own use, in all handles and calls of this process (for leak
 * checks).  Generated matrices handed to the caller and spmv_b200_malloc blocks are the caller's and not counted. */
SPMV_B200_API long long spmv_b200_live_allocations(void);

/* ---- multi-GPU row partition -------------------------------------------------------------------
 * splitter[g] = right_boundary(RowPtr, min(g*ceil(nnz/parts), nnz), m+1) - 1, g = 0..parts: the
 * reference's init_csrSplitter_balanced2 (parallel_balanced2_spmv.c:41-53) with nthreads = parts.
 * RowPtr is a HOST pointer; pure host code, usable without a GPU.  Returns 0 or -1. */
SPMV_B200_API int spmv_b200_partition_rows(const int *RowPtr, int m, int parts, int *splitter_out);

/* ---- fused SpMV + all-gather over NVLink peer memory -----------------------------------------------
 * In the iterated x <- A x loop on several GPUs every rank's y slice must reach every rank's next x.
 * Instead of a separate collective, a handle can store each y value to up to 8 EXTRA destinations while
 * it computes: device_ptrs[i] is the address where this rank's slice starts inside peer i's next-x buffer
 * (a peer mapping obtained through spmv_b200_ipc_open, or any local device buffer).  The stores are
 * issued by the kernel that produces the final y (CSR-vector, row blocks, SELL, the band reduce); the other
 * kernel families fall back to one stream-ordered copy kernel.  count = 0 switches it off.  The caller
 * synchronises the ranks (e.g. a 1-element NCCL all-reduce) before the next x is read.
 * ipc_export writes a 64-byte handle for a pointer returned by spmv_b200_malloc; ipc_open maps a handle
 * exported by another process on the same node (peer access is enabled lazily).  Return 0 / pointer, or
 * -1 / NULL with spmv_b200_last_error() set. */
SPMV_B200_API int spmv_b200_set_y_peers(spmv_Handle_t handle, int count, void *const *device_ptrs);
SPMV_B200_API int spmv_b200_ipc_export(const void *device_ptr, void *handle_out_64);
SPMV_B200_API void *spmv_b200_ipc_open(const void *handle_64);
SPMV_B200_API int spmv_b200_ipc_close(void *opened_ptr);

/* ---- column stages: an SpMV in pieces, for overlapping the y -> x exchange of an iterated loop with compute ------
 * A handle whose layout is banded by columns (the band-major copy of Method_Parallel, or band segments) computes the
 * contribution of every column band separately and folds them at the end.  These entry points expose that: band b
 * only reads x[col_lo, col_hi), so in x <- A x on several GPUs a rank can start on the bands whose slice of the new
 * x has already arrived while the rest is still in flight over NVLink (spmv_b200/multigpu.py: PipelinedPowerMethod).
 *   spmv_b200_bands         number of column bands that can be staged (1: not banded -- use spmv());
 *   spmv_b200_band_columns  the half-open column range band `band` reads;
 *   spmv_b200_spmv_bands    enqueue the partial products of bands [band_first, band_first + band_count) on the
 *                           handle's stream (x: DEVICE pointer to the full-length vector; any order, each band once);
 *   spmv_b200_spmv_finish   enqueue the fold: y (DEVICE pointer) = sum over all bands, in band order -- bit for bit
 *                           the y that spmv() writes, whatever order the bands were staged in; extra destinations
 *                           set with spmv_b200_set_y_peers are written here.
 * All return 0, or -1 (not stageable / bad arguments; spmv_b200_last_error()). */
SPMV_B200_API int spmv_b200_bands(spmv_Handle_t handle);
SPMV_B200_API int spmv_b200_band_columns(spmv_Handle_t handle, int band, long long *col_lo, long long *col_hi);
SPMV_B200_API int spmv_b200_spmv_bands(spmv_Handle_t handle, int band_first, int band_count, const void *x_device);
SPMV_B200_API int spmv_b200_spmv_finish(spmv_Handle_t handle, void *y_device);

/* ---- stream-ordered copies and flags: a copy-engine exchange over NVLink ---------------------------------------------
 * The y -> x exchange of the iterated loop moves hundreds of megabytes per GPU; done by kernels (NCCL or peer stores)
 * it competes with the SpMV for SMs, done by the copy engines it does not.  These three calls are all such an exchange
 * needs next to the IPC mappings above: a device-to-device copy (dst may be a peer mapping) enqueued on a stream, a
 * 32-bit flag written after everything earlier on the stream (cuStreamWriteValue32; the flag may live in a peer's
 * memory), and a wait that holds everything later on the stream until a flag is >= value (cuStreamWaitValue32).  The
 * flags carry iteration numbers: "my slice of x_k has landed in your buffer", "I have finished reading buffer p".
 * `cuda_stream` is a cudaStream_t passed as void*.  Return 0 or -1 (spmv_b200_last_error()). */
SPMV_B200_API int spmv_b200_memcpy_async(void *dst, const void *src, size_t bytes, void *cuda_stream);
SPMV_B200_API int spmv_b200_stream_write32(void *cuda_stream, void *device_ptr, unsigned value);
SPMV_B200_API int spmv_b200_stream_wait32_geq(void *cuda_stream, void *device_ptr, unsigned value);

/* ---- device memory helpers for C clients (Python clients use torch tensors) ----------------------- */
SPMV_B200_API void *spmv_b200_malloc(size_t bytes);
SPMV_B200_API void spmv_b200_free(void *device_ptr);
/* kind: 0 host->device, 1 device->host, 2 device->device; synchronous.  Returns 0 or -1. */
SPMV_B200_API int spmv_b200_memcpy(void *dst, const void *src, size_t bytes, int kind);

/* ---- on-device synthetic matrices (SURVEY.md 8d; bit-identical to spmv_b200/matrices.py) ----------
 * Each fills *out with DEVICE pointers owned by the caller (release with spmv_b200_csr_free).
 * `size` = sizeof(double) or sizeof(float).  Returns 0 or -1 (see spmv_b200_last_error); on failure *out holds
 * nothing to free (arguments that are rejected leave it untouched). */
typedef struct spmv_b200_csr {
    int m, n;
    long long nnz;
    int *RowPtr;
    int *ColIdx;
    void *Val;
    unsigned long size;
} spmv_b200_csr;

SPMV_B200_API int spmv_b200_gen_laplacian2d(int nx, int ny, unsigned long size, spmv_b200_csr *out);
SPMV_B200_API int spmv_b200_gen_stencil27(int nx, int ny, int nz, unsigned long size, spmv_b200_csr *out);
/* rows [row0, row0+m) of the global uniform-random matrix with k entries per row over n columns */
SPMV_B200_API int spmv_b200_gen_uniform(int m, int n, int k, unsigned long long seed, long long row0, int eighths,
                          unsigned long size, spmv_b200_csr *out);
SPMV_B200_API int spmv_b200_gen_rmat(int scale, int edge_factor, unsigned long long seed, unsigned long size,
                       spmv_b200_csr *out);
/* x_j for j in [0, n): 0.5 + (hash(j) mod 1000)/1000, or all ones */
SPMV_B200_API int spmv_b200_gen_x(void *device_dst, long long n, unsigned long long seed, int ones, unsigned long size);
SPMV_B200_API void spmv_b200_csr_free(spmv_b200_csr *csr);

#if defined(__cplusplus)
}
#endif
#endif /* SPMV_B200_EXT_H */
