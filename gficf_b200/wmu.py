"""Mann-Whitney U per gene on the GPU (SURVEY section 8f, "next" row 4): the host-side mirror of the
reference's R-visible function for that path.

Reference interface mirrored here:
  rcpp_parallel_WMU_test(matX, matY, printOutput)   R/RcppExports.R:20-22 ->
      src/rcpp_parallel_mann_whitney.cpp:106-127 (worker :12-103, helpers src/mann_whitney.cpp:17-131),
  called once per cluster by findClusterMarkers (R/deGenes.R:44-54) with matX = the cluster's cells,
  matY = all other cells (genes are rows).
"""
from __future__ import annotations

import ctypes as C
import sys

import numpy as np

from . import _lib

_BANNER = "Running Parallell WM-U test...\n"  # rcpp_parallel_mann_whitney.cpp:110
_BANNER_DONE = "Done!!\n"  # :124


def rcpp_parallel_WMU_test(matX, matY, printOutput: bool = False) -> np.ndarray:
    """Drop-in for the reference export: (n_genes x n1), (n_genes x n2) -> n_genes x 2 float64
    (Fortran order): column 0 the two-sided p-value (normal approximation, tie and continuity
    corrections), column 1 log2(mean(x + 1) / mean(y + 1))."""
    x = np.asfortranarray(np.asarray(matX), dtype=np.float64)
    y = np.asfortranarray(np.asarray(matY), dtype=np.float64)
    if x.ndim != 2 or y.ndim != 2:
        raise TypeError("numeric matrices (2-D) are required")
    if x.shape[0] != y.shape[0]:
        raise ValueError("matX and matY must have the same number of rows (genes)")
    if printOutput:
        sys.stdout.write(_BANNER)
    g = x.shape[0]
    out = np.empty((g, 2), dtype=np.float64, order="F")
    err = C.create_string_buffer(512)
    rc = _lib.lib().gficf_cuda_wmu_test(x.ctypes.data, y.ctypes.data, g, x.shape[1], y.shape[1], out.ctypes.data,
                                        err, 512)
    _lib.check(rc, err)
    if printOutput:
        sys.stdout.write(_BANNER_DONE)
    return out


def _cluster_ids(cluster, n_cells):
    """The markers calls' cluster ids as contiguous int32 and n_clusters = max id + 1."""
    cl = np.asarray(cluster)
    if cl.ndim != 1 or cl.shape[0] != n_cells:
        raise ValueError("cluster must hold one id per column (cell) of mat")
    if cl.size and not np.issubdtype(cl.dtype, np.integer):
        raise TypeError("cluster ids must be integers")
    if cl.size and (cl.min() < 0 or cl.max() >= 2 ** 31 - 1):
        raise ValueError("cluster ids must be 0-based and below 2^31 - 1")
    ids = np.ascontiguousarray(cl, dtype=np.int32)
    return ids, (int(ids.max()) + 1 if ids.size else 0)


def rcpp_parallel_WMU_markers(mat, cluster, printOutput: bool = False) -> np.ndarray:
    """Every cluster's one-vs-rest test in one call: a genes x cells matrix and one 0-based cluster id
    per cell -> (n_genes, 2, n_clusters) float64 (Fortran order).  out[:, :, c] equals, bit for bit,
    rcpp_parallel_WMU_test(mat[:, cluster == c], mat[:, cluster != c]); n_clusters = max id + 1, and
    every id in [0, n_clusters) must have cells."""
    m = np.asfortranarray(np.asarray(mat), dtype=np.float64)
    if m.ndim != 2:
        raise TypeError("a numeric matrix (2-D) is required")
    ids, k = _cluster_ids(cluster, m.shape[1])
    if printOutput:
        sys.stdout.write(_BANNER)
    g = m.shape[0]
    out = np.empty((g, 2, k), dtype=np.float64, order="F")
    err = C.create_string_buffer(512)
    rc = _lib.lib().gficf_cuda_wmu_markers(m.ctypes.data, g, m.shape[1], ids.ctypes.data, k, out.ctypes.data, err, 512)
    _lib.check(rc, err)
    if printOutput:
        sys.stdout.write(_BANNER_DONE)
    return out


def _int32_index(a, what):
    a = np.asarray(a)
    if not np.issubdtype(a.dtype, np.integer):
        raise TypeError("%s must be an integer array" % what)
    if a.dtype != np.int32 and a.size and (a.min() < -2 ** 31 or a.max() >= 2 ** 31):
        raise ValueError("%s does not fit in int32 (the dgCMatrix slots are R integers)" % what)
    return np.ascontiguousarray(a, dtype=np.int32)


def rcpp_parallel_WMU_markers_sparse(mat, cluster, printOutput: bool = False) -> np.ndarray:
    """rcpp_parallel_WMU_markers for a scipy.sparse CSC matrix or array (genes x cells; R's dgCMatrix has
    the same slots).  Only the stored values are uploaded and read; the result equals, bit for bit,
    rcpp_parallel_WMU_markers(mat.toarray(), cluster).  Stored zeros are zeros.  Other sparse formats and
    dense arrays raise TypeError (convert with .tocsc() first); index arrays that do not fit in int32 raise
    ValueError."""
    import scipy.sparse as sp

    if not sp.issparse(mat) or mat.format != "csc":
        raise TypeError("a scipy.sparse CSC matrix (genes x cells) is required")
    g, n = mat.shape
    colptr = _int32_index(mat.indptr, "indptr")
    row = _int32_index(mat.indices, "indices")
    x = np.ascontiguousarray(mat.data, dtype=np.float64)
    if colptr.size != n + 1 or row.size < colptr[-1] or x.size < colptr[-1]:
        raise ValueError("indptr / indices / data do not describe a %d x %d matrix" % (g, n))
    ids, k = _cluster_ids(cluster, n)
    if printOutput:
        sys.stdout.write(_BANNER)
    out = np.empty((g, 2, k), dtype=np.float64, order="F")
    err = C.create_string_buffer(512)
    rc = _lib.lib().gficf_cuda_wmu_markers_csc(colptr.ctypes.data, row.ctypes.data, x.ctypes.data, g, n,
                                               ids.ctypes.data, k, out.ctypes.data, err, 512)
    _lib.check(rc, err)
    if printOutput:
        sys.stdout.write(_BANNER_DONE)
    return out
