// NEW routine (added to the registration table, nothing existing changes arity): rcpp_parallel_WMU_markers
// for a sparse dgCMatrix, without densifying it.  R passes the matrix's slots as they are:
//   rcpp_parallel_WMU_markers_sparse(M@p, M@i, M@x, nrow(M), cluster, printOutput)
// and gets what rcpp_parallel_WMU_markers(as.matrix(M), cluster, printOutput) returns, bit for bit, while
// only the stored values cross to the GPU (gficf_cuda_wmu_markers_csc, include/gficf_cuda.h).  After adding
// this file run Rcpp::compileAttributes() so that src/RcppExports.cpp / R/RcppExports.R gain
// `_gficf_rcpp_parallel_WMU_markers_sparse`.
//
// cluster: one 1-based id per column of M (a factor's codes work as they are); the clusters are
// 1..max(cluster) and each needs at least one cell.  Result: nrow x 2K, columns 2c-1 and 2c are cluster c's
// p-value and log2 fold change.
#include <Rcpp.h>

#include <vector>

#include "gficf_cuda.h"

// [[Rcpp::export]]
Rcpp::NumericMatrix rcpp_parallel_WMU_markers_sparse(Rcpp::IntegerVector p, Rcpp::IntegerVector i, Rcpp::NumericVector x,
                                                     int nrow, Rcpp::IntegerVector cluster, bool printOutput) {
  if (printOutput) Rprintf("Running Parallell WM-U test...\n");
  const R_xlen_t ncol = (R_xlen_t)p.size() - 1;
  if (ncol < 0) Rcpp::stop("p must hold ncol(M) + 1 column pointers");
  if ((R_xlen_t)cluster.size() != ncol) Rcpp::stop("cluster must hold one id per column (cell) of M");
  const R_xlen_t nnz = (R_xlen_t)p[ncol];
  if (nnz < 0 || (R_xlen_t)i.size() < nnz || (R_xlen_t)x.size() < nnz) Rcpp::stop("i and x must hold p[ncol + 1] values");
  std::vector<int32_t> ids(cluster.size());
  int k = 0;
  for (R_xlen_t j = 0; j < (R_xlen_t)cluster.size(); ++j) {
    const int c = cluster[j];
    if (c < 1) Rcpp::stop("cluster ids must be positive integers (found %d at cell %d)", c, (int)j + 1);  // NA too
    ids[j] = c - 1;
    if (c > k) k = c;
  }
  Rcpp::NumericMatrix rmat(nrow, 2 * k);
  char msg[512] = {0};
  const int rc = gficf_cuda_wmu_markers_csc(&p[0], nnz ? &i[0] : nullptr, nnz ? &x[0] : nullptr, (int64_t)nrow,
                                            (int64_t)ncol, ids.data(), (int32_t)k, rmat.begin(), msg, sizeof msg);
  if (rc != GFICF_OK) Rcpp::stop("gficf CUDA Mann-Whitney markers failed (%d): %s", rc, msg);
  if (printOutput) Rprintf("Done!!\n");
  return rmat;
}
