// tests/rpkg_markers_sparse_entry.cpp -- TEST HARNESS.  A C entry point around the drop-in
// gficf_b200/rpkg/src/rcpp_parallel_wmu_markers_sparse.cpp, compiled against the stand-in R runtime of
// oracle/rshim/ plus the IntegerVector below and linked with the product library; built by
// tests/test_gpu_wmu_markers_sparse.py.
#include <Rcpp.h>

#include <cstring>

namespace Rcpp {
// What the export uses of Rcpp's IntegerVector (an R integer vector, wrapped without a copy).
class IntegerVector {
 public:
  IntegerVector(int* p, R_xlen_t n) : p_(p), n_(n) {}
  R_xlen_t size() const { return n_; }
  int& operator[](R_xlen_t i) { return p_[i]; }

 private:
  int* p_;
  R_xlen_t n_;
};
}  // namespace Rcpp

#include "rcpp_parallel_wmu_markers_sparse.cpp"

static std::vector<char> g_sink;

extern "C" {

// rcpp_parallel_WMU_markers_sparse(M@p, M@i, M@x, nrow, cluster, printOutput) with 1-based ids; out has
// nrow x 2k doubles.  Returns 0, or 1 with the R error text.
int rpkg_wmu_markers_sparse(const int* p, const int* i, const double* x, int nnz, int nrow, int ncol, const int* cluster,
                            int k, double* out, int print_output, char* err, int errlen, char* printed, int printedlen) {
  g_sink.clear();
  rshim::printf_sink() = &g_sink;
  int rc = 0;
  try {
    Rcpp::NumericVector xv(x, x + nnz);  // an R double vector (the stand-in runtime owns a copy)
    Rcpp::NumericMatrix res = rcpp_parallel_WMU_markers_sparse(
        Rcpp::IntegerVector(const_cast<int*>(p), ncol + 1), Rcpp::IntegerVector(const_cast<int*>(i), nnz), xv, nrow,
        Rcpp::IntegerVector(const_cast<int*>(cluster), ncol), print_output != 0);
    if (res.nrow() != nrow || res.ncol() != 2 * k) Rcpp::stop("result is %d x %d", res.nrow(), res.ncol());
    std::memcpy(out, res.begin(), sizeof(double) * 2 * (size_t)nrow * (size_t)k);
  } catch (const std::exception& e) {
    snprintf(err, errlen, "%s", e.what());
    rc = 1;
  }
  rshim::printf_sink() = nullptr;
  int m = (int)g_sink.size() < printedlen - 1 ? (int)g_sink.size() : printedlen - 1;
  if (printed && printedlen > 0) {
    std::memcpy(printed, g_sink.data(), m);
    printed[m] = 0;
  }
  return rc;
}
}
