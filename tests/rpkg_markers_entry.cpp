// tests/rpkg_markers_entry.cpp -- TEST HARNESS.  A C entry point around the drop-in
// gficf_b200/rpkg/src/rcpp_parallel_wmu_markers.cpp, compiled against the stand-in R runtime of
// oracle/rshim/ plus the IntegerVector below and linked with the product library; built by
// tests/test_gpu_wmu_markers.py.
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

#include "rcpp_parallel_wmu_markers.cpp"

static std::vector<char> g_sink;

extern "C" {

// rcpp_parallel_WMU_markers(mat, cluster, printOutput) with 1-based ids; out has genes x 2k doubles.
// Returns 0, or 1 with the R error text.
int rpkg_wmu_markers(const double* mat, int genes, int cells, const int* cluster, int k, double* out,
                     int print_output, char* err, int errlen, char* printed, int printedlen) {
  g_sink.clear();
  rshim::printf_sink() = &g_sink;
  int rc = 0;
  try {
    Rcpp::NumericMatrix m = Rcpp::NumericMatrix::wrap_external(const_cast<double*>(mat), genes, cells);
    Rcpp::NumericMatrix res =
        rcpp_parallel_WMU_markers(m, Rcpp::IntegerVector(const_cast<int*>(cluster), cells), print_output != 0);
    if (res.nrow() != genes || res.ncol() != 2 * k) Rcpp::stop("result is %d x %d", res.nrow(), res.ncol());
    std::memcpy(out, res.begin(), sizeof(double) * 2 * (size_t)genes * (size_t)k);
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
