# Drop-in for the hot loop of ccfindR::vb_factorize.  R is not installed where this repository is
# built and tested: the C half (src/vbnmf_shim.c) is compiled and executed there against a stand-in
# R runtime (tests/rstub, tests/test_rshim.py), which also checks every .Call below against the
# registered entry points and their arities; this R file itself is source only.
#
# vb_iterate_gpu() is ccfindR's vb_iterate (R/bayesian.R:303-390) with the
# `for(it in seq_len(bundle$Itmax))` loop (:337-352: vbnmf_update + hyper_update + convergence
# test) replaced by ONE .Call on a device-resident handle.  Everything outside that loop is the
# reference's code path: ccfindR:::vb_init, the uniform-column rule, the per-run bookkeeping and
# vb_factorize's best-run selection.  One deliberate omission: the `connectivity` bookkeeping of
# :328-331,353-357 builds an ncol*(ncol-1)/2 vector whose only use is the `dispersion = ` field of
# the verbose print; it is not computed here (it cannot be allocated beyond ~30,000 cells), so the
# verbose line is always the `connectivity=FALSE` form of :363-365.

vbnmf_handle <- function(mat, device = 0L) {
  mat <- methods::as(mat, "CsparseMatrix")          # dgCMatrix: @p, @i, @x, @Dim (no as.matrix())
  .Call(C_vbnmf_create, mat@p, mat@i, as.numeric(mat@x), mat@Dim, as.integer(device))
}

# One NCCL communicator per R process (= per GPU).  `uid` is raw(128): made by rank 0 with
# vbnmf_comm(nranks, 0L, NULL, device) -> attr(, "uid") and distributed by the host side, e.g.
# Rmpi::mpi.bcast (the reference already depends on Rmpi for its restarts, R/bayesian.R:263).
vbnmf_comm <- function(nranks, rank, uid = NULL, device = rank) {
  if (is.null(uid)) uid <- .Call(C_vbnmf_nccl_unique_id)
  comm <- .Call(C_vbnmf_comm_create, as.integer(nranks), as.integer(rank), uid, as.integer(device))
  attr(comm, "uid") <- uid
  comm
}

# Contiguous column ranges with (nearly) equal numbers of nonzeros: boundaries b[1..nranks+1]
# (0-based, half open) from the column pointers of a dgCMatrix.
vbnmf_shard_columns <- function(mat, nranks) {
  p <- methods::as(mat, "CsparseMatrix")@p
  nnz <- p[length(p)]
  b <- vapply(seq_len(nranks - 1), function(k) which.min(abs(p - nnz * k / nranks)) - 1L, 1L)
  c(0L, b, ncol(mat))
}

vb_iterate_gpu <- function(irun, bundle) {
  nrow <- dim(bundle$mat)[1]; ncol <- dim(bundle$mat)[2]
  nrank <- length(bundle$ranks)
  rdat <- rep(-Inf, nrank)
  wdat <- hdat <- dwdat <- dhdat <- hyperp <- list()
  nunif <- rep(0, nrank)
  h <- if (is.null(bundle$handle)) vbnmf_handle(bundle$mat, bundle$device) else bundle$handle
  if (!is.null(bundle$precision)) .Call(C_vbnmf_set_precision, h, as.integer(bundle$precision))
  if (bundle$verbose >= 2) if (bundle$nrun > 1) cat('Run ', irun, '\n', sep = '')
  for (irank in seq_len(nrank)) {
    rank <- bundle$ranks[[irank]]
    if (rank > min(nrow, ncol)) stop('Rank exceeded min(nrow,ncol)')
    hyper <- list(aw = bundle$gamma.a[1], ah = bundle$gamma.a[length(bundle$gamma.a)],
                  bw = bundle$gamma.b[1], bh = bundle$gamma.b[length(bundle$gamma.b)])
    device.init <- isTRUE(bundle$device.init) && bundle$initializer %in% c('random', 'svd2', 'svd')
    if (device.init) {
      # vb_init drawn / computed on the GPU: no nrow x rank / rank x ncol matrices cross the bus
      # ('svd' orients each pair of singular vectors k >= 1 first, include/vbnmf.h)
      seed <- as.numeric(bundle$seed + irun)
      if (bundle$initializer == 'random')
        .Call(C_vbnmf_init_random, h, as.integer(rank),
              c(hyper$aw, hyper$bw, hyper$ah, hyper$bh), seed)
      else if (bundle$initializer == 'svd2')
        .Call(C_vbnmf_init_svd2, h, as.integer(rank),
              c(hyper$aw, hyper$bw, hyper$ah, hyper$bh), seed)
      else
        .Call(C_vbnmf_init_svd, h, as.integer(rank), seed)
    } else {
      wh <- ccfindR:::vb_init(nrow, ncol, bundle$mat, rank, hyper = hyper,
                              initializer = bundle$initializer)
      .Call(C_vbnmf_set_state, h, wh$lw, wh$lh, wh$ew, wh$eh)
    }
    res <- .Call(C_vbnmf_run, h, c(hyper$aw, hyper$bw, hyper$ah, hyper$bh),
                 as.integer(bundle$Itmax), bundle$Tol, as.logical(bundle$hyper.update),
                 as.integer(bundle$hyper.update.n0), as.integer(bundle$hyper.update.dn),
                 bundle$fudge)
    hyper <- list(aw = res$hyper[1], bw = res$hyper[2], ah = res$hyper[3], bh = res$hyper[4])
    lk0 <- res$lml; it <- res$niter
    if (bundle$verbose >= 3)
      for (i in seq_len(it)) cat(i, ', log(evidence) = ', res$lkh_trace[i], '\n', sep = '')
    if (bundle$verbose >= 2)
      cat('Rank = ', rank, ': Nsteps =', it, ', log(evidence) =', lk0, ', hyper = (', hyper$aw, ',',
          hyper$bw, ',', hyper$ah, ',', hyper$bh, ')\n', sep = '')
    contains.unif <- .Call(C_vbnmf_uniform_columns, h, bundle$Tol)
    if (sum(contains.unif) > 0) {
      warning('Rank ', rank, ' row/column ', paste(which(contains.unif), collapse = ','), ' constant.')
      if (bundle$unif.stop) {
        warning('Rank scan stopped for rank >= ', rank)
        if (irank == 1) stop('Rerun with lower ranks')
        break
      }
    }
    st <- .Call(C_vbnmf_get_state, h)
    rdat[irank] <- lk0
    wdat[[irank]] <- st$ew; hdat[[irank]] <- st$eh
    dwdat[[irank]] <- sqrt(st$dw); dhdat[[irank]] <- sqrt(st$dh)
    hyperp[[irank]] <- hyper
  }
  list(rdat = rdat, wdat = wdat, hdat = hdat, hyperp = hyperp, nunif = nunif,
       dwdat = dwdat, dhdat = dhdat)
}

# vb_factorize (R/bayesian.R:229-301) with the GPU worker: same arguments and checks, same
# best-run selection and slot filling.  `comm` (from vbnmf_comm) + `cols` (this process's column
# range from vbnmf_shard_columns): the object holds ONE shard of the cells, the factorization is
# collective over the processes, and coeff / dcoeff are this shard's columns.
vb_factorize_gpu <- function(object, ranks = 2, nrun = 1, verbose = 2, initializer = 'random',
                             Itmax = 10000, hyper.update = rep(TRUE, 4), gamma.a = 1, gamma.b = 1,
                             Tol = 1e-5, hyper.update.n0 = 10, hyper.update.dn = 1, fudge = NULL,
                             unif.stop = TRUE, device = 0L, precision = 0L, comm = NULL,
                             device.init = FALSE, seed = 1) {
  if (is.null(fudge)) fudge <- .Machine$double.eps
  mat <- SingleCellExperiment::counts(object)
  if (initializer %in% c('svd', 'svd2') & nrun > 1) stop('SVD initializer does not require nrun > 1')
  if (is.null(comm) && sum(Matrix::rowSums(mat) == 0) > 0) stop('Input matrix contains empty rows')
  if (sum(Matrix::colSums(mat) == 0) > 0) stop('Input matrix contains empty columns')
  ranks <- ranks[ranks <= ncol(mat)]
  nrank <- length(ranks)
  handle <- vbnmf_handle(mat, device)               # X goes to the GPU once for all runs and ranks
  if (!is.null(comm)) .Call(C_vbnmf_attach_comm, handle, comm)   # (empty genes are tested globally)
  bundle <- list(mat = mat, ranks = ranks, verbose = verbose, gamma.a = gamma.a, gamma.b = gamma.b,
                 initializer = initializer, Itmax = Itmax, fudge = fudge, hyper.update = hyper.update,
                 hyper.update.n0 = hyper.update.n0, hyper.update.dn = hyper.update.dn, Tol = Tol,
                 unif.stop = unif.stop, nrun = nrun, handle = handle, device = device,
                 precision = precision, device.init = device.init, seed = seed)
  vb <- lapply(seq_len(nrun), FUN = vb_iterate_gpu, bundle)
  .Call(C_vbnmf_destroy, handle)
  basis <- dbasis <- coeff <- dcoeff <- vector('list', nrank)
  rdat <- awdat <- bwdat <- ahdat <- bhdat <- nunif <- c()
  ranks2 <- c()
  for (k in seq_len(nrank)) {                       # R/bayesian.R:268-291, unchanged
    rmax <- -Inf
    for (i in seq_len(nrun)) if (vb[[i]]$rdat[k] > rmax) { imax <- i; rmax <- vb[[i]]$rdat[k] }
    if (rmax == -Inf) next
    ranks2 <- c(ranks2, ranks[k]); rdat <- c(rdat, rmax)
    basis[[k]] <- vb[[imax]]$wdat[[k]]; coeff[[k]] <- vb[[imax]]$hdat[[k]]
    dbasis[[k]] <- vb[[imax]]$dwdat[[k]]; dcoeff[[k]] <- vb[[imax]]$dhdat[[k]]
    awdat <- c(awdat, vb[[imax]]$hyperp[[k]]$aw); bwdat <- c(bwdat, vb[[imax]]$hyperp[[k]]$bw)
    ahdat <- c(ahdat, vb[[imax]]$hyperp[[k]]$ah); bhdat <- c(bhdat, vb[[imax]]$hyperp[[k]]$bh)
    nunif <- c(nunif, vb[[imax]]$nunif[k])
    rownames(basis[[k]]) <- rownames(dbasis[[k]]) <- rownames(mat)
    colnames(coeff[[k]]) <- colnames(dcoeff[[k]]) <- colnames(mat)
  }
  object@ranks <- ranks2
  object@basis <- basis; object@dbasis <- dbasis
  object@coeff <- coeff; object@dcoeff <- dcoeff
  object@measure <- data.frame(rank = ranks2, lml = rdat, aw = awdat, bw = bwdat, ah = ahdat,
                               bh = bhdat, nunif = nunif)
  object
}
