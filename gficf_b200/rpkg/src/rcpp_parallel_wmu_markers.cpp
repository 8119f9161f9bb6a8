// NEW routine (added to the registration table, nothing existing changes arity): the loop of
// findClusterMarkers (R/deGenes.R:44-54) in one call.  For every cluster c it returns what
// rcpp_parallel_WMU_test(mat[, cluster == c], mat[, cluster != c], printOutput) returns, bit for bit,
// while the matrix is uploaded and every gene sorted once instead of once per cluster
// (gficf_cuda_wmu_markers, include/gficf_cuda.h).  After adding this file run
// Rcpp::compileAttributes() so that src/RcppExports.cpp / R/RcppExports.R gain
// `_gficf_rcpp_parallel_WMU_markers`.
//
// cluster: one 1-based id per column of mat (a factor's codes work as they are); the clusters are
// 1..max(cluster) and each needs at least one cell.  Result: n_genes x 2K, columns 2c-1 and 2c are
// cluster c's p-value and log2 fold change.
#include <Rcpp.h>

#include <vector>

#include "gficf_cuda.h"

// [[Rcpp::export]]
Rcpp::NumericMatrix rcpp_parallel_WMU_markers(Rcpp::NumericMatrix mat, Rcpp::IntegerVector cluster, bool printOutput) {
  if (printOutput) Rprintf("Running Parallell WM-U test...\n");
  if ((R_xlen_t)cluster.size() != (R_xlen_t)mat.ncol()) Rcpp::stop("cluster must hold one id per column (cell) of mat");
  std::vector<int32_t> ids(cluster.size());
  int k = 0;
  for (R_xlen_t i = 0; i < (R_xlen_t)cluster.size(); ++i) {
    const int c = cluster[i];
    if (c < 1) Rcpp::stop("cluster ids must be positive integers (found %d at cell %d)", c, (int)i + 1);  // NA too
    ids[i] = c - 1;
    if (c > k) k = c;
  }
  Rcpp::NumericMatrix rmat(mat.nrow(), 2 * k);
  char msg[512] = {0};
  const int rc = gficf_cuda_wmu_markers(mat.begin(), (int64_t)mat.nrow(), (int64_t)mat.ncol(), ids.data(), (int32_t)k,
                                        rmat.begin(), msg, sizeof msg);
  if (rc != GFICF_OK) Rcpp::stop("gficf CUDA Mann-Whitney markers failed (%d): %s", rc, msg);
  if (printOutput) Rprintf("Done!!\n");
  return rmat;
}
