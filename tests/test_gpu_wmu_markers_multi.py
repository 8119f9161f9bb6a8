"""GPU (-m gpu, two devices or more): the sparse markers call with the genes split over D devices
(gficf_cuda_wmu_markers_csc_devices) against the single-device call (gficf_cuda_wmu_markers_csc), bit for bit,
for D = 2 .. min(8, visible); its errors and the state it leaves; and the R export
(gficf_b200/rpkg/src/rcpp_parallel_wmu_markers_sparse_gpus.cpp) through the stand-in R runtime."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest
import scipy.sparse as sp

from tests.sum_order_cases import sensitive_genes
from tests.test_gpu_wmu_markers import CAP, labels
from tests.test_wmu_markers_sparse_emu import edge_rows, malformed_cases, to_csc
from tests.test_wmu_oracle import sc_matrix

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def ndev(cuda):
    n = cuda.lib().gficf_cuda_device_count()
    if n < 2:
        pytest.skip("needs >= 2 GPUs")
    return n


def device_counts(ndev):
    return list(range(2, min(8, ndev) + 1))


def csc(m, rng=None, stored_zeros=0.0):
    colptr, row, x, dense = to_csc(m, rng, stored_zeros)
    return sp.csc_matrix((x, row, colptr), shape=dense.shape)


def check(cuda, ndev, mat, cl):
    want = cuda.rcpp_parallel_WMU_markers_sparse(mat, cl)
    for D in device_counts(ndev):
        got = cuda.rcpp_parallel_WMU_markers_sparse(mat, cl, n_devices=D)
        assert got.shape == want.shape and got.flags.f_contiguous
        assert np.array_equal(got.view(np.int64), want.view(np.int64)), D
        if min(D, mat.shape[0]) > 1 and mat.nnz > 0:
            assert cuda.last_timings()["allgather_ms"] > 0, D          # the exchange ran
    return want


def random_csc(rng, genes, cells, density):
    """Poisson counts over library sizes, generated in CSC form column by column (geometric gaps between the
    stored rows), never dense; the values repeat, so genes have many tie groups."""
    width = int(genes * density + 8 * np.sqrt(genes * density) + 64)
    lib = rng.uniform(0.5, 2.0, size=cells)
    indptr, rows, xs = np.zeros(cells + 1, dtype=np.int64), [], []
    for j0 in range(0, cells, 4000):
        j1 = min(cells, j0 + 4000)
        r = np.cumsum(rng.geometric(density, size=(j1 - j0, width)), axis=1) - 1
        keep = r < genes
        cnt = keep.sum(axis=1)
        rows.append(r[keep].astype(np.int32))
        xs.append((1 + rng.poisson(0.5, size=int(cnt.sum()))) * 200.0 / np.repeat(lib[j0:j1], cnt))
        indptr[j0 + 1:j1 + 1] = cnt
    return sp.csc_matrix((np.concatenate(xs), np.concatenate(rows), np.cumsum(indptr).astype(np.int32)),
                         shape=(genes, cells))


def test_r03_shaped_matrix(cuda, ndev):
    """2000 genes x 100 000 cells, 20 clusters, about 14 % stored."""
    rng = np.random.default_rng(41)
    mat = random_csc(rng, 2000, 100_000, 0.14)
    check(cuda, ndev, mat, labels(rng, 100_000, 20))


def test_unequal_columns_empty_slabs_and_few_genes(cuda, ndev):
    rng = np.random.default_rng(42)
    genes, cells, k = 40, 20_000, 9
    cl = labels(rng, cells, k)
    m = edge_rows(rng, sc_matrix(rng, genes, cells, density=0.02), cl)
    m[:, rng.choice(cells, size=30, replace=False)] = rng.random((genes, 30)) + 0.25   # a few nearly full columns
    m[:, 1000:4000] = 0.0
    m[[1, 4, 13, 20, 21, 30, 39]] = 0.0                                                 # empty genes
    check(cuda, ndev, csc(m, rng, 0.05), cl)
    slabs = np.zeros((12, cells))                                                       # values in three columns
    slabs[:, [5, 6, 17_000]] = rng.random((12, 3)) + 0.5
    check(cuda, ndev, csc(slabs), cl)
    check(cuda, ndev, csc(np.zeros((12, cells))), cl)                                   # nothing stored
    few = sc_matrix(rng, 3, cells, density=0.3)                                         # n_genes < D
    check(cuda, ndev, csc(few, rng, 0.05), cl)
    check(cuda, ndev, csc(sc_matrix(rng, 10, 5, density=0.6)), np.array([0, 1, 2, 0, 1], np.int32))  # cells < D


def test_order_sensitive_tie_sums(cuda, ndev):
    """N = 300 000 >= 208 064: the tie term is the sequential sum in sorted order, on genes where another order
    gives another p-value (tests/sum_order_cases.py)."""
    n = 300_000
    rng = np.random.default_rng(3)
    cl = rng.integers(0, 5, n).astype(np.int32)
    m, _ = sensitive_genes(4, n, cl == 1, ("shifted", "plain", "negative", "dense"))
    check(cuda, ndev, csc(m, rng, 0.01), cl)


def test_cluster_cap(cuda, ndev):
    rng = np.random.default_rng(43)
    cells = 3 * CAP
    cl = labels(rng, cells, CAP)
    check(cuda, ndev, csc(sc_matrix(rng, 16, cells, density=0.5)), cl)


def test_malformed_row_id_then_a_valid_call(cuda, ndev):
    cl = np.array([0, 1, 0, 1], dtype=np.int32)
    for name, colptr, row in malformed_cases():
        mat = sp.csc_matrix((5, 4))
        mat.indptr, mat.indices, mat.data = colptr, row, np.arange(1.0, row.size + 1.0)
        with pytest.raises(cuda.GficfCudaError) as e:
            cuda.rcpp_parallel_WMU_markers_sparse(mat, cl, n_devices=2)
        assert e.value.code == 1 and "row id" in e.value.message, name
    rng = np.random.default_rng(44)
    mat = random_csc(rng, 300, 30_000, 0.1)
    good = random_csc(rng, 300, 30_000, 0.1)
    cl = labels(rng, 30_000, 6)
    bad = mat.copy()
    bad.indices = bad.indices.copy()
    bad.indices[bad.indptr[-2]] = 300                                                   # in the last column only
    with pytest.raises(cuda.GficfCudaError) as e:
        cuda.rcpp_parallel_WMU_markers_sparse(bad, cl, n_devices=min(8, ndev))
    assert e.value.code == 1
    check(cuda, ndev, good, cl)


def test_device_count_arguments(cuda, ndev):
    rng = np.random.default_rng(45)
    mat = random_csc(rng, 200, 20_000, 0.1)
    cl = labels(rng, 20_000, 5)
    with pytest.raises(cuda.GficfCudaError) as e:
        cuda.rcpp_parallel_WMU_markers_sparse(mat, cl, n_devices=ndev + 1)
    assert e.value.code == 1 and "visible" in e.value.message
    want = cuda.rcpp_parallel_WMU_markers_sparse(mat, cl)
    before = cuda.lib().gficf_cuda_get_devices()
    try:
        for D in (1, 2):
            cuda.set_devices(D)
            got = cuda.rcpp_parallel_WMU_markers_sparse(mat, cl, n_devices=0)               # the configured count
            assert np.array_equal(got.view(np.int64), want.view(np.int64))
            assert (cuda.last_timings()["allgather_ms"] > 0) == (D > 1), D
    finally:
        cuda.set_devices(before)


def test_callers_device_stays_current(cuda, ndev):
    import torch

    rng = np.random.default_rng(46)
    mat = random_csc(rng, 100, 10_000, 0.1)
    cl = labels(rng, 10_000, 4)
    torch.cuda.set_device(1)
    try:
        cuda.rcpp_parallel_WMU_markers_sparse(mat, cl, n_devices=2)
        assert torch.cuda.current_device() == 1
        bad = mat.copy()
        bad.indices = bad.indices.copy()
        bad.indices[0] = -1
        with pytest.raises(cuda.GficfCudaError):
            cuda.rcpp_parallel_WMU_markers_sparse(bad, cl, n_devices=2)
        assert torch.cuda.current_device() == 1
    finally:
        torch.cuda.set_device(0)


@pytest.fixture(scope="module")
def rharness(tmp_path_factory):
    import gficf_b200

    so = str(tmp_path_factory.mktemp("rpkg") / "librpkg_markers_sparse_gpus.so")
    lib = gficf_b200.library_path()
    cmd = ["g++", "-O2", "-std=c++11", "-fPIC", "-shared", "-Wall", "-Werror",
           "-I" + os.path.join(ROOT, "oracle", "rshim"), "-I" + os.path.join(ROOT, "include"),
           "-I" + os.path.join(ROOT, "gficf_b200", "rpkg", "src"),
           os.path.join(ROOT, "tests", "rpkg_markers_sparse_gpus_entry.cpp"), lib,
           "-Wl,-rpath," + os.path.dirname(lib), "-o", so]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    L = C.CDLL(so)
    L.rpkg_wmu_markers_sparse_gpus.argtypes = [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int,
                                               C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_char_p, C.c_int,
                                               C.c_char_p, C.c_int]
    L.rpkg_wmu_markers_sparse_gpus.restype = C.c_int
    return L


def r_markers_sparse_gpus(L, mat, cl1, k, n_gpu, print_output):
    p, i = mat.indptr.astype(np.int32), mat.indices.astype(np.int32)
    x = np.ascontiguousarray(mat.data, dtype=np.float64)
    ids = np.ascontiguousarray(cl1, dtype=np.int32)
    out = np.empty((mat.shape[0], 2 * k), dtype=np.float64, order="F")
    err, printed = C.create_string_buffer(1024), C.create_string_buffer(1024)
    rc = L.rpkg_wmu_markers_sparse_gpus(p.ctypes.data, i.ctypes.data, x.ctypes.data, int(p[-1]), mat.shape[0],
                                        mat.shape[1], ids.ctypes.data, k, n_gpu, out.ctypes.data, int(print_output),
                                        err, 1024, printed, 1024)
    if rc != 0:
        raise RuntimeError(err.value.decode())
    return out, printed.value.decode()


def test_r_export_through_stand_in_runtime(cuda, ndev, rharness):
    rng = np.random.default_rng(47)
    genes, cells, k = 40, 1200, 5
    cl = labels(rng, cells, k)
    mat = csc(sc_matrix(rng, genes, cells), rng, 0.05)
    want = cuda.rcpp_parallel_WMU_markers_sparse(mat, cl)
    for n_gpu in device_counts(ndev):
        res, text = r_markers_sparse_gpus(rharness, mat, cl + 1, k, n_gpu, True)
        assert text == "Running Parallell WM-U test...\nDone!!\n"
        for c in range(k):  # columns 2c-1, 2c (1-based) are cluster c's (p-value, log2FC)
            assert np.array_equal(res[:, 2 * c:2 * c + 2].view(np.int64), want[:, :, c].view(np.int64)), (n_gpu, c)
    assert r_markers_sparse_gpus(rharness, mat, cl + 1, k, 2, False)[1] == ""
    bad = cl + 1
    bad[3] = 0
    with pytest.raises(RuntimeError) as e:
        r_markers_sparse_gpus(rharness, mat, bad, k, 2, False)
    assert "positive" in str(e.value)
    with pytest.raises(RuntimeError) as e:
        r_markers_sparse_gpus(rharness, mat, np.where(cl == 1, 3, cl + 1), k, 2, False)  # cluster 2 has no cells
    assert "failed (1)" in str(e.value)
    broken = mat.copy()
    broken.indices = broken.indices.copy()
    broken.indices[broken.indptr[-2]] = genes                   # a row id past nrow, in the last slab
    with pytest.raises(RuntimeError) as e:
        r_markers_sparse_gpus(rharness, broken, cl + 1, k, 2, False)
    assert "failed (1)" in str(e.value)
    with pytest.raises(RuntimeError) as e:
        r_markers_sparse_gpus(rharness, mat, cl + 1, k, ndev + 1, False)
    assert "failed (1)" in str(e.value)
