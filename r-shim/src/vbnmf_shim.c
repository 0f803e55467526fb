/* R .Call shim over libvbnmf (include/vbnmf.h).  R is not installed in the build environment of
 * this repository: there this file is compiled, linked against libvbnmf.so and EXECUTED against
 * stand-in headers and a minimal runtime for the R C API subset it uses (tests/rstub/,
 * tests/test_rshim.py); it uses nothing beyond the documented API (Rinternals.h,
 * R_ext/Rdynload.h).
 *
 * It replaces, in ccfindR, the generated glue src/RcppExports.cpp:11-32 (one .Call per ITERATION,
 * `_ccfindR_vbnmf_update`) by one .Call per RUN of iterations on a device-resident handle.
 * Build inside an R package:  PKG_LIBS = -L<dir of libvbnmf.so> -lvbnmf ; PKG_CPPFLAGS = -I<repo>/include
 */
#include <R.h>
#include <Rinternals.h>
#include <R_ext/Rdynload.h>
#include <stdint.h>
#include <string.h>

#include "vbnmf.h"

static void chk(int rc, vbnmf_handle *h) {
    if (rc != 0) Rf_error("libvbnmf: %s", vbnmf_last_error(h)); /* like END_RCPP, RcppExports.cpp:21 */
}

static void handle_finalizer(SEXP ptr) {
    vbnmf_handle *h = (vbnmf_handle *)R_ExternalPtrAddr(ptr);
    if (h) vbnmf_destroy(h);
    R_ClearExternalPtr(ptr);
}

static vbnmf_handle *get_handle(SEXP ptr) {
    vbnmf_handle *h = (vbnmf_handle *)R_ExternalPtrAddr(ptr);
    if (!h) Rf_error("libvbnmf: handle has been released");
    return h;
}

/* dgCMatrix slots: p = @p (int, m+1), i = @i (int, 0-based), x = @x (double), dim = @Dim */
SEXP C_vbnmf_create(SEXP p, SEXP i, SEXP x, SEXP dim, SEXP device) {
    vbnmf_handle *h = NULL;
    const int n = INTEGER(dim)[0], m = INTEGER(dim)[1];
    const int64_t nnz = (int64_t)XLENGTH(x);
    int rc = vbnmf_create(&h, n, m, nnz, INTEGER(p), NULL, INTEGER(i), REAL(x), Rf_asInteger(device));
    if (rc != 0) Rf_error("libvbnmf: %s", vbnmf_last_error(NULL));
    SEXP ptr = PROTECT(R_MakeExternalPtr(h, R_NilValue, R_NilValue));
    R_RegisterCFinalizerEx(ptr, handle_finalizer, TRUE);
    UNPROTECT(1);
    return ptr;
}

SEXP C_vbnmf_destroy(SEXP ptr) {
    handle_finalizer(ptr);
    return R_NilValue;
}

/* wh list fields lw, lh, ew, eh as numeric matrices (column-major, as R stores them) */
SEXP C_vbnmf_set_state(SEXP ptr, SEXP lw, SEXP lh, SEXP ew, SEXP eh) {
    vbnmf_handle *h = get_handle(ptr);
    const int r = Rf_ncols(lw);
    chk(vbnmf_set_state(h, r, REAL(lw), REAL(lh), Rf_isNull(ew) ? NULL : REAL(ew),
                        Rf_isNull(eh) ? NULL : REAL(eh)), h);
    return R_NilValue;
}

/* vb_init(initializer = 'random') drawn on the device (R/bayesian.R:111-115,170): no n x r and
 * r x m matrices cross the bus.  hyper = c(aw, bw, ah, bh); seed: numeric(1) (an integer value) */
SEXP C_vbnmf_init_random(SEXP ptr, SEXP rank, SEXP hyper, SEXP seed) {
    vbnmf_handle *h = get_handle(ptr);
    chk(vbnmf_init_random(h, Rf_asInteger(rank), REAL(hyper), (uint64_t)Rf_asReal(seed), 0), h);
    return R_NilValue;
}

/* vb_init(initializer = 'svd2') computed on the device from the resident matrix
 * (R/bayesian.R:150-159): randomized truncated SVD keyed by seed.  hyper = c(aw, bw, ah, bh) */
SEXP C_vbnmf_init_svd2(SEXP ptr, SEXP rank, SEXP hyper, SEXP seed) {
    vbnmf_handle *h = get_handle(ptr);
    chk(vbnmf_init_svd2(h, Rf_asInteger(rank), REAL(hyper), (uint64_t)Rf_asReal(seed), 0), h);
    return R_NilValue;
}

/* vb_init(initializer = 'svd') computed on the device (R/bayesian.R:116-149), each pair of
 * singular vectors k >= 1 oriented first (include/vbnmf.h) */
SEXP C_vbnmf_init_svd(SEXP ptr, SEXP rank, SEXP seed) {
    vbnmf_handle *h = get_handle(ptr);
    chk(vbnmf_init_svd(h, Rf_asInteger(rank), (uint64_t)Rf_asReal(seed), 0), h);
    return R_NilValue;
}

/* one vbnmf_update (src/vbnmf_update.cpp:16-102); hyper = c(aw, bw, ah, bh) */
SEXP C_vbnmf_step(SEXP ptr, SEXP hyper, SEXP fudge) {
    vbnmf_handle *h = get_handle(ptr);
    double lkh = NA_REAL;
    chk(vbnmf_step(h, REAL(hyper), Rf_asReal(fudge), &lkh), h);
    return Rf_ScalarReal(lkh);
}

/* the it-loop of vb_iterate (R/bayesian.R:336-352) */
SEXP C_vbnmf_run(SEXP ptr, SEXP hyper, SEXP itmax, SEXP tol, SEXP hyper_update, SEXP n0, SEXP dn,
                 SEXP fudge) {
    vbnmf_handle *h = get_handle(ptr);
    vbnmf_cfg cfg;
    cfg.itmax = Rf_asInteger(itmax);
    cfg.tol = Rf_asReal(tol);
    for (int k = 0; k < 4; k++) cfg.hyper_update[k] = LOGICAL(hyper_update)[k] ? 1 : 0;
    cfg.n0 = Rf_asInteger(n0);
    cfg.dn = Rf_asInteger(dn);
    cfg.fudge = Rf_asReal(fudge);
    SEXP hy = PROTECT(Rf_duplicate(hyper));
    SEXP trace = PROTECT(Rf_allocVector(REALSXP, cfg.itmax));
    int niter = 0, reason = 0;
    double lml = 0.0;
    chk(vbnmf_run(h, &cfg, REAL(hy), REAL(trace), NULL, &niter, &lml, &reason), h);
    const char *names[] = {"hyper", "lml", "niter", "stop_reason", "lkh_trace", ""};
    SEXP out = PROTECT(Rf_mkNamed(VECSXP, names));
    SET_VECTOR_ELT(out, 0, hy);
    SET_VECTOR_ELT(out, 1, Rf_ScalarReal(lml));
    SET_VECTOR_ELT(out, 2, Rf_ScalarInteger(niter));
    SET_VECTOR_ELT(out, 3, Rf_ScalarInteger(reason));
    SET_VECTOR_ELT(out, 4, Rf_lengthgets(trace, niter));
    UNPROTECT(3);
    return out;
}

/* list(lw, lh, ew, eh, dw, dh) with the shapes of src/vbnmf_update.cpp:92-100 */
SEXP C_vbnmf_get_state(SEXP ptr) {
    vbnmf_handle *h = get_handle(ptr);
    int64_t info[8];
    chk(vbnmf_info(h, info), h);
    const int n = (int)info[0], m = (int)info[1], r = (int)info[3];
    const char *names[] = {"lw", "lh", "ew", "eh", "dw", "dh", ""};
    SEXP out = PROTECT(Rf_mkNamed(VECSXP, names));
    for (int k = 0; k < 6; k++) {
        const int wside = (k % 2 == 0);
        SET_VECTOR_ELT(out, k, Rf_allocMatrix(REALSXP, wside ? n : r, wside ? r : m));
    }
    chk(vbnmf_get_state(h, REAL(VECTOR_ELT(out, 0)), REAL(VECTOR_ELT(out, 1)),
                        REAL(VECTOR_ELT(out, 2)), REAL(VECTOR_ELT(out, 3)),
                        REAL(VECTOR_ELT(out, 4)), REAL(VECTOR_ELT(out, 5))), h);
    UNPROTECT(1);
    return out;
}

SEXP C_vbnmf_uniform_columns(SEXP ptr, SEXP tol) {
    vbnmf_handle *h = get_handle(ptr);
    int64_t info[8];
    chk(vbnmf_info(h, info), h);
    SEXP out = PROTECT(Rf_allocVector(LGLSXP, (R_xlen_t)info[3]));
    chk(vbnmf_uniform_columns(h, Rf_asReal(tol), (int32_t *)LOGICAL(out)), h);
    UNPROTECT(1);
    return out;
}

SEXP C_vbnmf_cluster_id(SEXP ptr) {
    vbnmf_handle *h = get_handle(ptr);
    int64_t info[8];
    chk(vbnmf_info(h, info), h);
    SEXP out = PROTECT(Rf_allocVector(INTSXP, (R_xlen_t)info[1]));
    chk(vbnmf_cluster_id(h, (int32_t *)INTEGER(out)), h);
    UNPROTECT(1);
    return out;
}

/* it-loop of factorize(), criterion = 'likelihood' (R/factorize.R:189-212) */
SEXP C_mlnmf_run(SEXP ptr, SEXP w0, SEXP h0, SEXP itmax, SEXP tol) {
    vbnmf_handle *h = get_handle(ptr);
    const int n = Rf_nrows(w0), r = Rf_ncols(w0), m = Rf_ncols(h0), it = Rf_asInteger(itmax);
    const char *names[] = {"ew", "eh", "lik_trace", "niter", ""};
    SEXP out = PROTECT(Rf_mkNamed(VECSXP, names));
    SET_VECTOR_ELT(out, 0, Rf_allocMatrix(REALSXP, n, r));
    SET_VECTOR_ELT(out, 1, Rf_allocMatrix(REALSXP, r, m));
    SEXP trace = PROTECT(Rf_allocVector(REALSXP, it));
    int niter = 0;
    chk(mlnmf_run(h, r, REAL(w0), REAL(h0), it, Rf_asReal(tol), REAL(VECTOR_ELT(out, 0)),
                  REAL(VECTOR_ELT(out, 1)), REAL(trace), &niter), h);
    SET_VECTOR_ELT(out, 2, Rf_lengthgets(trace, niter));
    SET_VECTOR_ELT(out, 3, Rf_ScalarInteger(niter));
    UNPROTECT(2);
    return out;
}

/* 0 = fp64 (the reference's arithmetic), 1 = fp32 storage / fp64 accumulation */
SEXP C_vbnmf_set_precision(SEXP ptr, SEXP precision) {
    vbnmf_handle *h = get_handle(ptr);
    chk(vbnmf_set_precision(h, Rf_asInteger(precision)), h);
    return R_NilValue;
}

SEXP C_vbnmf_set_host_threads(SEXP nthreads) {
    if (vbnmf_set_host_threads(Rf_asInteger(nthreads)) != 0) Rf_error("libvbnmf: bad thread count");
    return R_NilValue;
}

/* ---- cells sharded over several GPUs: one R process per GPU (the processes the reference would
 * start through Rmpi, R/bayesian.R:263), each holding a contiguous range of the columns --------- */
static void comm_finalizer(SEXP ptr) {
    vbnmf_comm *c = (vbnmf_comm *)R_ExternalPtrAddr(ptr);
    if (c) vbnmf_comm_destroy(c);
    R_ClearExternalPtr(ptr);
}

/* raw(128): the ncclUniqueId made on rank 0, to be broadcast by the host side (e.g. Rmpi::mpi.bcast) */
SEXP C_vbnmf_nccl_unique_id(void) {
    SEXP out = PROTECT(Rf_allocVector(RAWSXP, 128));
    if (vbnmf_nccl_unique_id(RAW(out)) != 0) Rf_error("libvbnmf: %s", vbnmf_last_error(NULL));
    UNPROTECT(1);
    return out;
}

SEXP C_vbnmf_comm_create(SEXP nranks, SEXP rank, SEXP uid, SEXP device) {
    vbnmf_comm *c = NULL;
    if (XLENGTH(uid) != 128) Rf_error("libvbnmf: the unique id must be raw(128)");
    if (vbnmf_comm_create(&c, Rf_asInteger(nranks), Rf_asInteger(rank), RAW(uid),
                          Rf_asInteger(device)) != 0)
        Rf_error("libvbnmf: %s", vbnmf_last_error(NULL));
    SEXP ptr = PROTECT(R_MakeExternalPtr(c, R_NilValue, R_NilValue));
    R_RegisterCFinalizerEx(ptr, comm_finalizer, TRUE);
    UNPROTECT(1);
    return ptr;
}

SEXP C_vbnmf_comm_destroy(SEXP ptr) {
    comm_finalizer(ptr);
    return R_NilValue;
}

/* the handle holds the columns of ONE shard; collective over the ranks of the communicator */
SEXP C_vbnmf_attach_comm(SEXP ptr, SEXP comm) {
    vbnmf_handle *h = get_handle(ptr);
    vbnmf_comm *c = (vbnmf_comm *)R_ExternalPtrAddr(comm);
    if (!c) Rf_error("libvbnmf: communicator has been released");
    chk(vbnmf_attach_comm(h, c), h);
    return R_NilValue;
}

static const R_CallMethodDef CallEntries[] = {
    {"C_vbnmf_create", (DL_FUNC)&C_vbnmf_create, 5},
    {"C_vbnmf_destroy", (DL_FUNC)&C_vbnmf_destroy, 1},
    {"C_vbnmf_set_state", (DL_FUNC)&C_vbnmf_set_state, 5},
    {"C_vbnmf_init_random", (DL_FUNC)&C_vbnmf_init_random, 4},
    {"C_vbnmf_init_svd2", (DL_FUNC)&C_vbnmf_init_svd2, 4},
    {"C_vbnmf_init_svd", (DL_FUNC)&C_vbnmf_init_svd, 3},
    {"C_vbnmf_step", (DL_FUNC)&C_vbnmf_step, 3},
    {"C_vbnmf_run", (DL_FUNC)&C_vbnmf_run, 8},
    {"C_vbnmf_get_state", (DL_FUNC)&C_vbnmf_get_state, 1},
    {"C_vbnmf_uniform_columns", (DL_FUNC)&C_vbnmf_uniform_columns, 2},
    {"C_vbnmf_cluster_id", (DL_FUNC)&C_vbnmf_cluster_id, 1},
    {"C_mlnmf_run", (DL_FUNC)&C_mlnmf_run, 5},
    {"C_vbnmf_set_precision", (DL_FUNC)&C_vbnmf_set_precision, 2},
    {"C_vbnmf_set_host_threads", (DL_FUNC)&C_vbnmf_set_host_threads, 1},
    {"C_vbnmf_nccl_unique_id", (DL_FUNC)&C_vbnmf_nccl_unique_id, 0},
    {"C_vbnmf_comm_create", (DL_FUNC)&C_vbnmf_comm_create, 4},
    {"C_vbnmf_comm_destroy", (DL_FUNC)&C_vbnmf_comm_destroy, 1},
    {"C_vbnmf_attach_comm", (DL_FUNC)&C_vbnmf_attach_comm, 2},
    {NULL, NULL, 0}};

/* mirrors R_init_ccfindR, src/RcppExports.cpp:29-32 */
void R_init_ccfindRgpu(DllInfo *dll) {
    R_registerRoutines(dll, NULL, CallEntries, NULL, NULL);
    R_useDynamicSymbols(dll, FALSE);
}
