"""GPU (-m gpu): the markers call on a compressed-column matrix (gficf_cuda_wmu_markers_csc) against the dense
call (gficf_cuda_wmu_markers) on the densified matrix, bit for bit, and against the oracle on subsets; the
malformed-matrix errors raised on the device; and the R export
(gficf_b200/rpkg/src/rcpp_parallel_wmu_markers_sparse.cpp) through the stand-in R runtime."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp

from oracle.binding import WmuOracle
from tests.sum_order_cases import sensitive_genes
from tests.test_gpu_wmu_markers import CAP, labels
from tests.test_wmu_markers_sparse_emu import edge_rows, malformed_cases, to_csc
from tests.test_wmu_oracle import sc_matrix

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def csc(m, rng=None, stored_zeros=0.0):
    colptr, row, x, dense = to_csc(m, rng, stored_zeros)
    return sp.csc_matrix((x, row, colptr), shape=dense.shape), dense


def check(cuda, m, cl, rng=None, stored_zeros=0.05, clusters=None, oracle_genes=None):
    k = int(cl.max()) + 1
    mat, dense = csc(m, rng, stored_zeros)
    got = cuda.rcpp_parallel_WMU_markers_sparse(mat, cl)
    assert got.shape == (m.shape[0], 2, k) and got.flags.f_contiguous
    want = cuda.rcpp_parallel_WMU_markers(dense, cl)
    assert np.array_equal(got.view(np.int64), want.view(np.int64))
    sub = slice(None) if oracle_genes is None else slice(0, oracle_genes)
    orc = WmuOracle()
    for c in range(k) if clusters is None else clusters:
        x, y = np.asfortranarray(dense[sub][:, cl == c]), np.asfortranarray(dense[sub][:, cl != c])
        assert np.array_equal(got[sub, :, c], orc.wmu(x, y), equal_nan=True), c
    return got


def test_sparse_markers_match_dense_call(cuda):
    rng = np.random.default_rng(17)
    genes, cells, k = 17, 30_000, 12
    cl = labels(rng, cells, k)
    m = edge_rows(rng, sc_matrix(rng, genes, cells, integer=True), cl)
    m[:, [0, cells // 3, cells - 1]] = 0.0                   # empty columns
    check(cuda, m, cl, rng)


def test_sparse_markers_many_genes_and_staged_upload(cuda):
    """2500 genes: more genes than resident CTAs, and stored values above the 8 MiB small-copy threshold."""
    rng = np.random.default_rng(25)
    genes, cells, k = 2500, 6000, 7
    cl = labels(rng, cells, k)
    check(cuda, sc_matrix(rng, genes, cells, density=0.3), cl, rng, oracle_genes=64)


def test_sparse_markers_large_n_ordered_tie_sum(cuda):
    """N >= 208064: the tie term is the reference's sequential double sum in sorted order."""
    rng = np.random.default_rng(26)
    genes, cells, k = 4, 210_000, 3
    cl = labels(rng, cells, k)
    m = np.floor(rng.gamma(2.0, 2.0, size=(genes, cells))) * (rng.random((genes, cells)) < 0.2)
    m[3, :] = -m[3, :]
    check(cuda, m, cl, rng)


def test_sparse_markers_order_sensitive_genes(cuda):
    n = 300_000
    rng = np.random.default_rng(3)
    cl = rng.integers(0, 5, n).astype(np.int32)
    m, _ = sensitive_genes(4, n, cl == 1, ("shifted", "plain", "negative", "dense"))
    check(cuda, m, cl, rng, stored_zeros=0.01)


def test_sparse_markers_cluster_cap(cuda):
    rng = np.random.default_rng(27)
    genes, cells = 3, 3 * CAP
    cl = labels(rng, cells, CAP)
    m = sc_matrix(rng, genes, cells, density=0.5)
    picked = [0, 1, CAP // 2, CAP - 1] + list(rng.choice(CAP, size=12, replace=False))
    check(cuda, m, cl, rng, clusters=picked)
    cl[7] = CAP                                              # one cluster more than the cap
    with pytest.raises(cuda.GficfCudaError) as e:
        cuda.rcpp_parallel_WMU_markers_sparse(csc(m)[0], cl)
    assert e.value.code == 5


def test_sparse_markers_malformed_rows_on_device(cuda):
    """Row ids are checked by the device pass that reads them: GFICF_E_ARG, and the next call works."""
    cl = np.array([0, 1, 0, 1], dtype=np.int32)
    for name, colptr, row in malformed_cases():
        mat = sp.csc_matrix((5, 4))
        mat.indptr, mat.indices, mat.data = colptr, row, np.arange(1.0, row.size + 1.0)
        with pytest.raises(cuda.GficfCudaError) as e:
            cuda.rcpp_parallel_WMU_markers_sparse(mat, cl)
        assert e.value.code == 1 and "row id" in e.value.message, name
    rng = np.random.default_rng(30)
    m = sc_matrix(rng, 40, 900)
    check(cuda, m, labels(rng, 900, 4), rng)
    tm = cuda.last_timings()
    assert tm["h2d_ms"] > 0 and tm["jaccard_ms"] > 0 and tm["wall_ms"] >= tm["h2d_ms"]


@pytest.fixture(scope="module")
def rharness(tmp_path_factory):
    import gficf_b200

    so = str(tmp_path_factory.mktemp("rpkg") / "librpkg_markers_sparse.so")
    lib = gficf_b200.library_path()
    cmd = ["g++", "-O2", "-std=c++11", "-fPIC", "-shared", "-Wall", "-Werror",
           "-I" + os.path.join(ROOT, "oracle", "rshim"), "-I" + os.path.join(ROOT, "include"),
           "-I" + os.path.join(ROOT, "gficf_b200", "rpkg", "src"),
           os.path.join(ROOT, "tests", "rpkg_markers_sparse_entry.cpp"), lib, "-Wl,-rpath," + os.path.dirname(lib),
           "-o", so]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    L = C.CDLL(so)
    L.rpkg_wmu_markers_sparse.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p,
                                          C.c_int, C.c_void_p, C.c_int, C.c_char_p, C.c_int, C.c_char_p, C.c_int]
    L.rpkg_wmu_markers_sparse.restype = C.c_int
    return L


def r_markers_sparse(L, mat, cl1, k, print_output):
    p, i = mat.indptr.astype(np.int32), mat.indices.astype(np.int32)
    x = np.ascontiguousarray(mat.data, dtype=np.float64)
    ids = np.ascontiguousarray(cl1, dtype=np.int32)
    out = np.empty((mat.shape[0], 2 * k), dtype=np.float64, order="F")
    err, printed = C.create_string_buffer(1024), C.create_string_buffer(1024)
    rc = L.rpkg_wmu_markers_sparse(p.ctypes.data, i.ctypes.data, x.ctypes.data, int(p[-1]), mat.shape[0], mat.shape[1],
                                   ids.ctypes.data, k, out.ctypes.data, int(print_output), err, 1024, printed, 1024)
    if rc != 0:
        raise RuntimeError(err.value.decode())
    return out, printed.value.decode()


def test_r_export_through_stand_in_runtime(cuda, rharness):
    rng = np.random.default_rng(29)
    genes, cells, k = 40, 1200, 5
    cl = labels(rng, cells, k)
    mat, dense = csc(sc_matrix(rng, genes, cells), rng, 0.05)
    res, text = r_markers_sparse(rharness, mat, cl + 1, k, True)
    assert text == "Running Parallell WM-U test...\nDone!!\n"
    want = cuda.rcpp_parallel_WMU_markers(dense, cl)
    for c in range(k):  # columns 2c-1, 2c (1-based) are cluster c's (p-value, log2FC)
        assert np.array_equal(res[:, 2 * c:2 * c + 2], want[:, :, c], equal_nan=True)
        x, y = np.asfortranarray(dense[:, cl == c]), np.asfortranarray(dense[:, cl != c])
        assert np.array_equal(res[:, 2 * c:2 * c + 2], WmuOracle().wmu(x, y), equal_nan=True)
    assert r_markers_sparse(rharness, mat, cl + 1, k, False)[1] == ""
    bad = cl + 1
    bad[3] = 0
    with pytest.raises(RuntimeError) as e:
        r_markers_sparse(rharness, mat, bad, k, False)
    assert "positive" in str(e.value)
    with pytest.raises(RuntimeError) as e:
        r_markers_sparse(rharness, mat, np.where(cl == 1, 3, cl + 1), k, False)  # cluster 2 has no cells
    assert "failed (1)" in str(e.value)
    broken = mat.copy()
    broken.indices = broken.indices.copy()
    broken.indices[broken.indptr[5]] = genes                 # a row id past nrow
    with pytest.raises(RuntimeError) as e:
        r_markers_sparse(rharness, broken, cl + 1, k, False)
    assert "failed (1)" in str(e.value)
