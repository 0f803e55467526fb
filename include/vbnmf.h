/* libvbnmf — C ABI of the B200-native variational-Bayes Poisson-NMF engine.
 *
 * This is the drop-in boundary for ONE path of the R package ccfindR: the per-iteration VB update
 * and the loop that drives it.  Citations are file:line in the reference tree.
 *
 *   reference interface replaced                                     entry point here
 *   ---------------------------------------------------------------  -------------------------
 *   .Call(`_ccfindR_vbnmf_update`, X, wh, hyper, fudge)               vbnmf_create + vbnmf_set_state
 *     R/RcppExports.R:4-6, src/RcppExports.cpp:11-22                  + vbnmf_step + vbnmf_get_state
 *   vbnmf_update(): one VB iteration, src/vbnmf_update.cpp:16-102     vbnmf_step
 *   return list w,h,lw,lh,ew,eh,lkh,dw,dh, src/vbnmf_update.cpp:92-100 vbnmf_get_state (+ *lkh)
 *   for(it in seq_len(Itmax)) loop of vb_iterate, R/bayesian.R:336-352 vbnmf_run
 *   hyper_update(), R/bayesian.R:2-53                                  (inside vbnmf_run)
 *   uniform-column test, R/bayesian.R:368-369                          vbnmf_uniform_columns
 *   cluster_id(): apply(h,2,which.max), R/utils.R:903-909              vbnmf_cluster_id
 *   nmf_updateR() + likelihood() loop, R/factorize.R:189-212           mlnmf_run, mlnmf_run2 (both criteria)
 *   vb_init(): 'random', 'svd', 'svd2', R/bayesian.R:111-149,150-159   vbnmf_init_random, vbnmf_init_svd,
 *                                                                      vbnmf_init_svd2
 *   read_10x(): readMM + as(., 'dgCMatrix'), R/utils.R:34               vbnmf_create_from_mtx
 *   filter_cells(): colSums(counts), R/utils.R:78-95                   vbnmf_qc_stats +
 *                                                                      vbnmf_create_subset
 *   filter_genes(): rowSums, VMR, cells expressed, R/utils.R:134-218   vbnmf_qc_stats +
 *                                                                      vbnmf_create_subset
 *   normalize_count(): counts scaled per cell, R/utils.R:318-327       vbnmf_create_subset (col_scale)
 *   factorize(randomize = TRUE): each column of the counts shuffled    vbnmf_create_shuffled
 *     over the genes, R/factorize.R:172-173
 *   factorize(): dispersion() and cophenet() of the consensus          vbnmf_consensus
 *     connectivity, R/factorize.R:51-78,214-216,226 (average linkage)
 *   Rmpi task farm over restarts, R/bayesian.R:263                     one handle per process/GPU;
 *                                                                      cells sharded: vbnmf_attach_comm
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on failure; vbnmf_last_error() gives the text.
 *     No C++ exception crosses this boundary.
 *   - all matrices are column-major doubles exactly as R stores them: lw/ew/dw are n x r,
 *     lh/eh/dh are r x m.  hyper = {aw, bw, ah, bh}.
 *   - the count matrix is CSC as in Matrix::dgCMatrix: colptr = @p (length m+1), rowidx = @i
 *     (0-based), values = @x.  Column pointers may be 32- or 64-bit; on the device they are 64-bit.
 *   - a handle owns one CUDA device and is not thread-safe.  There is no CPU fallback: creating a
 *     handle without a usable CUDA device fails.
 *   - when cells are sharded over several GPUs (one process and one handle per GPU), m is the
 *     LOCAL number of cells, lh/eh/dh are the local columns, lw/ew/dw are replicated, and every
 *     rank must make the same sequence of calls (set_state/step/run are collective).
 */
#ifndef VBNMF_H
#define VBNMF_H
#include <stdint.h>

#if defined(__GNUC__)
#define VBNMF_API __attribute__((visibility("default")))
#else
#define VBNMF_API
#endif

#ifdef __cplusplus
extern "C" {
#endif

typedef struct vbnmf_handle vbnmf_handle;

/* mirrors the `bundle` of vb_factorize (R/bayesian.R:252-259) for the fields the loop reads */
typedef struct {
    int itmax;            /* Itmax */
    double tol;           /* Tol */
    int hyper_update[4];  /* hyper.update: aw, bw, ah, bh */
    int n0;               /* hyper.update.n0 */
    int dn;               /* hyper.update.dn */
    double fudge;         /* fudge (R passes .Machine$double.eps when NULL, R/bayesian.R:238) */
} vbnmf_cfg;

enum { VBNMF_FP64 = 0, VBNMF_FP32_STORAGE = 1 };
enum { VBNMF_STOP_ITMAX = 0, VBNMF_STOP_CONVERGED = 1, VBNMF_STOP_NAN = 2 };
enum {
    VBNMF_OK = 0,
    VBNMF_ERR_ARG = 1,
    VBNMF_ERR_HYPER = 2, /* 'Hyper-parameter update failed to converge', R/bayesian.R:43 */
    VBNMF_ERR_CUDA = 3,
    VBNMF_ERR_STATE = 4,
    VBNMF_ERR_NCCL = 5,
    VBNMF_ERR_EMPTY = 6, /* 'Input matrix contains empty rows/columns', R/bayesian.R:244-247 */
    VBNMF_ERR_MEMORY = 7 /* vbnmf_consensus: more label groups than max_groups or device memory allow */
};

/* Upload a CSC count matrix from HOST memory and build the device-side layouts.
 * Exactly one of colptr32 / colptr64 is non-NULL.  device = CUDA ordinal. */
VBNMF_API int vbnmf_create(vbnmf_handle **out, int64_t n, int64_t m, int64_t nnz, const int32_t *colptr32,
                 const int64_t *colptr64, const int32_t *rowidx, const double *values, int device);

/* Same, from arrays already resident on `device` (int64 colptr, int32 rowidx, fp32 counts).
 * The arrays are borrowed: they must outlive the handle.  They are read on the handle's own
 * stream, starting inside this call: the work that produces them must have COMPLETED (synchronise
 * the producing stream first) -- the library cannot know that stream. */
VBNMF_API int vbnmf_create_from_device(vbnmf_handle **out, int64_t n, int64_t m, int64_t nnz,
                             const int64_t *d_colptr, const int32_t *d_rowidx, const float *d_values,
                             int device);

/* Host threads that stage uploads (copy / fp64 -> fp32 conversion into pinned buffers).  Default
 * min(16, hardware threads) or VBNMF_HOST_THREADS; with one process per GPU pass cores / processes.
 * Process-wide.  (The reference holds X in R memory; this replaces as.matrix(), R/bayesian.R:339.) */
VBNMF_API int vbnmf_set_host_threads(int nthreads);

/* Return the device memory the engine's stream-ordered pool keeps cached to the driver. */
VBNMF_API int vbnmf_trim_pool(int device);

/* Read a MatrixMarket coordinate file (the `matrix.mtx` of a 10x directory, R/utils.R:28-54:
 * Matrix::readMM + as(., 'dgCMatrix')) straight into a device-resident handle: the host reads the
 * bytes and the header, the text is parsed, sorted into CSC and validated on the GPU.  Supports
 * `matrix coordinate real|integer general`.  dims (may be NULL) receives n, m, nnz. */
VBNMF_API int vbnmf_create_from_mtx(vbnmf_handle **out, const char *path, int device, int64_t dims[3]);

/* The CSC arrays of a handle copied to the host: colptr (m+1), rowidx (nnz), values (nnz); any may
 * be NULL.  (After vbnmf_create_from_mtx the front end needs them for the row/column filters.) */
VBNMF_API int vbnmf_get_csc(vbnmf_handle *h, int64_t *colptr, int32_t *rowidx, double *values);

/* QC statistics of the matrix a handle holds (filter_cells / filter_genes / calc_vmr,
 * R/utils.R:78-95,134-218).  Any pointer may be NULL.  cell_sum (m), gene_sum, gene_sumsq (n):
 * fp64 sums of x and x^2; gene_cells (n), cell_genes (m): entries with a non-zero value.
 * The sums are exact for integer counts (any summation order gives the same bits).  A handle with
 * a communicator of more than one rank attached is refused (VBNMF_ERR_STATE). */
VBNMF_API int vbnmf_qc_stats(vbnmf_handle *h, double *cell_sum, double *gene_sum,
                             double *gene_sumsq, int64_t *gene_cells, int64_t *cell_genes);

/* A new handle on src's device holding the rows i with keep_rows[i] != 0 and the columns j with
 * keep_cols[j] != 0 of src's matrix (order kept, rows renumbered), each kept entry of column j
 * multiplied by col_scale[j] when col_scale != NULL (normalize_count, R/utils.R:318-327).
 * Built from src's device arrays; src is not modified and stays valid.  keep_rows has src's n
 * entries, keep_cols and col_scale its m.  Stored entries are kept as stored (explicit zeros
 * included); the values are held as by vbnmf_create (fp32 when every one is exact in fp32), so
 * the handle equals vbnmf_create on the same CSC.  No rows, columns or entries selected:
 * VBNMF_ERR_ARG; src with more than one rank attached: VBNMF_ERR_STATE. */
VBNMF_API int vbnmf_create_subset(vbnmf_handle **out, vbnmf_handle *src, const uint8_t *keep_rows,
                                  const uint8_t *keep_cols, const double *col_scale);

/* A new handle on src's device holding src's matrix with each column shuffled over the genes: the
 * null matrix of factorize(randomize = TRUE) (R/factorize.R:172-173).  colptr, nnz and each
 * column's values (stored zeros included) are kept; only the rows are drawn.  Column j with k
 * entries: u_t = the (t+1)-th next() of the counter stream (seed, 3 << 62 | j) of
 * vbnmf_init_random, row of draw t = (u_t * n) >> 64, s_0 .. s_{k-1} = the first k distinct rows
 * drawn; the t-th stored entry goes to row s_t, and the column is stored sorted by row (csrc/
 * shuffle.cuh, restated in ccfindr_b200/synth.py:shuffle_columns_reference).  Built from src's
 * device arrays after src's stream has finished; src is not modified.  The values keep src's
 * format, so the handle equals vbnmf_create on the same CSC.  A gene left without entries is
 * accepted here and refused when a factorization is set up (VBNMF_ERR_EMPTY).  n above 929,792
 * rows (one column's row bitmap must fit one CTA's 227 KB of shared memory) or a column with more
 * entries than rows: VBNMF_ERR_ARG; src with more than one rank attached: VBNMF_ERR_STATE. */
VBNMF_API int vbnmf_create_shuffled(vbnmf_handle **out, vbnmf_handle *src, uint64_t seed);

/* Consensus measures of factorize() (R/factorize.R:51-78,214-216,226) from the labels of nrun
 * restarts, without the m(m-1)/2 connectivity vector.  Handle-free: runs on `device` and releases
 * everything it allocated before returning.  labels: HOST memory, run-major (nrun x m), values
 * 0 ... nlabels - 1.  Let a_xy = number of runs in which cells x and y share a label.
 *   moments[0] = S1 = sum_{x<y} a_xy = sum_t sum_c C(n^t_c, 2),
 *   moments[1] = S2 = sum_{x<y} a_xy^2 = S1 + 2 sum_{t<u} sum_{c,c'} C(M^tu_cc', 2)
 *   (exact; M^tu = K x K contingency table of runs t and u); dispersion follows from S1, S2.
 * merges == NULL: moments only.  Otherwise also the average-linkage tree of 1 - a / nrun:
 *   groups = the distinct columns of labels in the order of (L[0], L[1], ...); *ngroups = G;
 *   IP_ab = n_a n_b #{t: T_at = T_bt} for groups a < b;
 *   G - 1 greedy steps: among active a < b take the largest q_ab = IP_ab / (nrun N_a N_b) (both
 *   exact int64 values converted to fp64, IEEE division), ties to the smallest a, then the
 *   smallest b; record (a, b, IP_ab, N_a, N_b) as row s of merges ((G - 1) x 5, row-major);
 *   IP_ak += IP_bk for every active k, N_a += N_b, retire b.  (The Lance-Williams update of
 *   average linkage is exact on the integers IP.)  *rescans = rows rescanned by the row cache of
 *   the merge loop.
 * The tree needs 8 G (G - 1) / 2 bytes of device memory for the IP triangle.  G above max_groups
 * (0: no limit) or above what device memory allows: VBNMF_ERR_MEMORY, with G in *ngroups.
 * VBNMF_ERR_ARG: nrun < 1, m < 1 or m >= 2^31; nlabels outside 1 ... 240 (a K x K table of
 * counters must fit one CTA's shared memory); a label outside 0 ... nlabels - 1;
 * nrun * ceil(m / 2)^2 >= 2^53; merge_cap < G - 1 (G still in *ngroups).
 * Error text: vbnmf_last_error(NULL). */
VBNMF_API int vbnmf_consensus(int device, int64_t m, int nrun, int nlabels, const int32_t *labels,
                              int64_t max_groups, int64_t moments[2], int64_t *ngroups,
                              int64_t *merges, int64_t merge_cap, int64_t *rescans);

VBNMF_API void vbnmf_destroy(vbnmf_handle *h);
VBNMF_API const char *vbnmf_last_error(const vbnmf_handle *h); /* h may be NULL: error of the last create */

/* VBNMF_FP64 (default): all arithmetic IEEE double, as the reference.
 * VBNMF_FP32_STORAGE: lw/lh panels held in fp32, per-nonzero arithmetic fp32, all sums fp64. */
VBNMF_API int vbnmf_set_precision(vbnmf_handle *h, int precision);

/* Run the engine's kernels on a caller-provided CUDA stream (cudaStream_t cast to void*). */
VBNMF_API int vbnmf_set_stream(vbnmf_handle *h, void *cuda_stream);

/* Multi-GPU: an NCCL communicator of `nranks` processes (one per GPU) that hold disjoint cell
 * ranges of one matrix.  The communicator belongs to the process, not to a handle: create it once
 * (uid = 128-byte ncclUniqueId from vbnmf_nccl_unique_id() on rank 0, distributed by the host, e.g.
 * over MPI where the reference uses Rmpi, R/bayesian.R:263) and attach it to each handle. */
typedef struct vbnmf_comm vbnmf_comm;
VBNMF_API int vbnmf_nccl_unique_id(void *uid128);
VBNMF_API int vbnmf_comm_create(vbnmf_comm **out, int nranks, int rank, const void *uid128, int device);
VBNMF_API void vbnmf_comm_destroy(vbnmf_comm *c);
VBNMF_API int vbnmf_attach_comm(vbnmf_handle *h, vbnmf_comm *c);

/* Load the state list `wh` (R/bayesian.R:170: lw, lh, ew, eh).  ew may be NULL (it is overwritten
 * before use, src/vbnmf_update.cpp:44); eh NULL means eh = lh (vb_init). */
VBNMF_API int vbnmf_set_state(vbnmf_handle *h, int r, const double *lw, const double *lh, const double *ew,
                    const double *eh);

/* vb_init(initializer = 'random') (R/bayesian.R:111-115,170) drawn on the device instead of
 * vbnmf_set_state from host matrices: w_ik ~ Gamma(shape aw, scale bw/aw), h_kj ~ Gamma(shape ah,
 * scale bh/ah), lw = ew = w, lh = eh = h.  R's RNG stream cannot be reproduced; the draw is defined
 * by a counter RNG keyed by (seed, gene i or GLOBAL cell index cell_offset + j, k) (csrc/
 * kernels_common.cuh, restated in ccfindr_b200/synth.py:device_random_init_reference), so it does
 * not depend on the device layout or on how the cells are sharded.  hyper = {aw, bw, ah, bh}. */
VBNMF_API int vbnmf_init_random(vbnmf_handle *h, int r, const double hyper[4], uint64_t seed,
                                int64_t cell_offset);

/* vb_init(initializer = 'svd2') (R/bayesian.R:150-159) on the device: w = |u| / scale,
 * h = |diag(d) v^T| * scale, scale = bh / mean(h), from a rank-r truncated SVD of the count matrix
 * computed where it lives (randomized subspace iteration with oversampling 20, run until the r
 * leading Ritz values stop moving, in place of irlba; k x k factorizations on the host).  Singular
 * vectors are defined up to sign, which abs() removes; they match an exact truncated SVD to ~1e-7.
 * seed keys the Gaussian test matrix by GLOBAL cell index (cell_offset + j): the result does not
 * depend on the sharding.  hyper = {aw, bw, ah, bh} (only bh is used, as in the reference). */
VBNMF_API int vbnmf_init_svd2(vbnmf_handle *h, int r, const double hyper[4], uint64_t seed,
                              int64_t cell_offset);

/* vb_init(initializer = 'svd') (R/bayesian.R:116-149) on the device, from the same truncated SVD
 * as vbnmf_init_svd2 (same seed, same cell_offset rule), U = (u_k) n x r, d, V = (v_k) m x r:
 *   component 0, as the reference: w_0 = sqrt(d_0) u_0, h_0 = sqrt(d_0) v_0, both multiplied by
 *     sgn = sign(w_00) (gene 0), and w_0 kept unflipped with h_0 = 0 when w_00 is exactly 0;
 *   components k >= 1, NNDSVD (Boutsidis & Gallopoulos 2008): P = |u_k+| |v_k+|, N = |u_k-| |v_k-|
 *     (norms of the positive and negative parts over all genes and all cells); when N > P the
 *     pair becomes (-u_k, -v_k) (ties keep it); then w_k = sqrt(d_k P) u_k+ / |u_k+|,
 *     h_k = sqrt(d_k P) v_k+ / |v_k+|.
 * The reference computes its negative-part norms from the positive parts (:136-137), so it always
 * takes the positive parts of whatever signs irlba returned, and gives NaN when both are <= 0.
 * Orienting each pair first makes the result independent of the SVD's sign choice, equal to the
 * reference whenever irlba returned the dominant orientation, and finite: for a nonnegative matrix
 * and d_k > 0, P = N = 0 would force u_k^T X v_k <= 0.  lw = ew = w, lh = eh = h; no hyper-
 * parameter enters.  Numerical rank below r: VBNMF_ERR_ARG, as vbnmf_init_svd2. */
VBNMF_API int vbnmf_init_svd(vbnmf_handle *h, int r, uint64_t seed, int64_t cell_offset);

/* One call of vbnmf_update (src/vbnmf_update.cpp:16-102): state <- update(state); *lkh = bound. */
VBNMF_API int vbnmf_step(vbnmf_handle *h, const double hyper[4], double fudge, double *lkh);

/* The loop of vb_iterate for one rank (R/bayesian.R:336-352) on the loaded state.
 * hyper: in = initial {aw,bw,ah,bh}, out = final.  lkh_trace (itmax doubles, may be NULL):
 * lkh of every executed iteration.  hyper_trace (4*itmax, may be NULL): hyper after each iteration.
 * *lml = lk0 as stored at R/bayesian.R:379 (NOT updated by the iteration that breaks). */
VBNMF_API int vbnmf_run(vbnmf_handle *h, const vbnmf_cfg *cfg, double hyper[4], double *lkh_trace,
              double *hyper_trace, int *niter, double *lml, int *stop_reason);

/* Copy the state out; any pointer may be NULL.  dw, dh are variances (the R driver stores their
 * square roots, R/bayesian.R:382-383). */
VBNMF_API int vbnmf_get_state(vbnmf_handle *h, double *lw, double *lh, double *ew, double *eh, double *dw,
                    double *dh);

/* inputs of hyper_update for the current state: mean(log lw), mean(log lh), mean(ew), mean(eh) */
VBNMF_API int vbnmf_get_means(vbnmf_handle *h, double means[4]);

/* cid[j] = 1-based index of the first maximum of column j of eh (local cells) */
VBNMF_API int vbnmf_cluster_id(vbnmf_handle *h, int32_t *cid);

/* flags[k] = 1 when column k of ew has |max - min| < tol (R/bayesian.R:368-369) */
VBNMF_API int vbnmf_uniform_columns(vbnmf_handle *h, double tol, int32_t *flags);

/* Maximum-likelihood path: the it-loop of factorize() with criterion='likelihood'
 * (R/factorize.R:189-212) from initial w0 (n x r), h0 (r x m).  lik_trace may be NULL. */
VBNMF_API int mlnmf_run(vbnmf_handle *h, int r, const double *w0, const double *h0, int itmax, double tol,
              double *w, double *h_out, double *lik_trace, int *niter);

/* Same loop with the stopping rule of factorize() selectable (R/factorize.R:194-212):
 * criterion = VBNMF_ML_LIKELIHOOD: |lkold - lk0| < tol |lkold| (:207, what mlnmf_run does);
 * criterion = VBNMF_ML_CONNECTIVITY: stop when the connectivity matrix of the cells
 * (outer(cid, cid, '=='), cid = which.max of each column of h, :51-60) has not changed for
 * ncnn_step consecutive iterations (:195-203).  The m(m-1)/2 connectivity vector is never formed:
 * sum(cnn != cnn0) is taken from the r x r contingency table of consecutive labelings.
 * nchange_trace (itmax doubles, may be NULL): that count per iteration (npair at iteration 1). */
enum { VBNMF_ML_LIKELIHOOD = 0, VBNMF_ML_CONNECTIVITY = 1 };
VBNMF_API int mlnmf_run2(vbnmf_handle *h, int r, const double *w0, const double *h0, int itmax,
               double tol, int criterion, int ncnn_step, double *w, double *h_out,
               double *lik_trace, double *nchange_trace, int *niter);

/* Measurement hooks (bench.py).  Runs `iters` steady-state VB iterations (posterior update +
 * nonzero sweep [+ all-reduce]) with fixed hypers and reports CUDA-event times in ms:
 * ms[0] = whole timed region, ms[1] = sum over the column-sweep kernel, ms[2] = row-sweep kernel,
 * ms[3] = everything else.  launches = kernels launched inside the timed region.
 * hyper_on = 1: hyper_update (R/bayesian.R:2-53) after every iteration as in the reference loop past
 * hyper.update.n0, hyper[] in/out; 0: hyper-parameters held fixed. */
VBNMF_API int vbnmf_bench_iterations(vbnmf_handle *h, double hyper[4], double fudge, int iters,
                           int hyper_on, double ms[4], int64_t *launches, double *lkh_last);

/* shape / layout facts for the host side */
VBNMF_API int vbnmf_info(const vbnmf_handle *h, int64_t info[8]); /* n, m, nnz, r, rs, precision, nranks, m_global */
/* facts about the tiled device layout in use (valid after vbnmf_set_state / mlnmf_run):
 * info[0] storage format of the nonzeros: 0 = {int32 row, float count} (8 bytes), 1 = int32 row +
 *         double count (12 bytes; counts not exact in fp32), 2 = packed {count << 16 | row}
 *         (4 bytes; integer counts below 2^16);
 * info[1] tile rows T, info[2] gene slabs, info[3] cell slabs,
 * info[4], info[5] entries stored for the cell-owner / gene-owner pass (nonzeros + schedule holes),
 * info[6] nonzeros per 8-lane group step, info[7] bytes of both passes' entry and pointer arrays */
VBNMF_API int vbnmf_layout_info(const vbnmf_handle *h, int64_t info[8]);

#ifdef __cplusplus
}
#endif
#endif
