"""GPU (-m gpu): every cluster's one-vs-rest Mann-Whitney test in one call (gficf_cuda_wmu_markers) against
the oracle (oracle/wmu_oracle.c) and against the library's own per-cluster call (gficf_cuda_wmu_test) on
the same slices, bit for bit; and the R export (gficf_b200/rpkg/src/rcpp_parallel_wmu_markers.cpp)
through the stand-in R runtime."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle.binding import WmuOracle
from tests.test_wmu_oracle import sc_matrix

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CAP = 8192  # include/gficf_cuda.h


def labels(rng, cells, k):
    """Interleaved ids with unequal cluster sizes; every id has cells."""
    w = rng.random(k) + 0.2
    cl = rng.choice(k, size=cells, p=w / w.sum()).astype(np.int32)
    cl[rng.choice(cells, size=k, replace=False)] = np.arange(k, dtype=np.int32)
    return cl


def check(cuda, m, cl, clusters=None, oracle=True):
    k = int(cl.max()) + 1
    got = cuda.rcpp_parallel_WMU_markers(m, cl)
    assert got.shape == (m.shape[0], 2, k) and got.flags.f_contiguous
    orc = WmuOracle()
    for c in range(k) if clusters is None else clusters:
        x, y = np.asfortranarray(m[:, cl == c]), np.asfortranarray(m[:, cl != c])
        assert np.array_equal(got[:, :, c], cuda.rcpp_parallel_WMU_test(x, y), equal_nan=True), c
        if oracle:
            assert np.array_equal(got[:, :, c], orc.wmu(x, y), equal_nan=True), c
    return got


def test_markers_match_per_cluster_calls(cuda):
    rng = np.random.default_rng(17)
    genes, cells, k = 17, 30_000, 12
    cl = labels(rng, cells, k)
    m = sc_matrix(rng, genes, cells, integer=True)
    m[0, :] = 3.0                                            # p = 1 everywhere
    m[1, :] = 0.0
    m[2, :] = -m[2, :]                                       # negative values
    m[3, ::2] = -0.0                                         # -0.0 ties with +0.0
    m[4, :] = np.where(cl == 5, 0.0, rng.random(cells) + 1.0)  # cluster 5 completely separated
    m[5, :] = rng.normal(size=cells)
    got = check(cuda, np.asfortranarray(m), cl)
    assert np.all(got[0, 0, :] == 1.0)


def test_markers_many_genes_and_staged_upload(cuda):
    """More genes than resident CTAs and a matrix above the 8 MiB small-copy threshold."""
    rng = np.random.default_rng(25)
    genes, cells, k = 2500, 2600, 7                          # 52 MB of pageable doubles
    cl = labels(rng, cells, k)
    check(cuda, sc_matrix(rng, genes, cells), cl)


def test_markers_large_n_ordered_tie_sum(cuda):
    """N >= 208064: the tie term is the reference's sequential double sum in sorted order."""
    rng = np.random.default_rng(26)
    genes, cells, k = 4, 210_000, 3
    cl = labels(rng, cells, k)
    m = np.floor(rng.gamma(2.0, 2.0, size=(genes, cells))) * (rng.random((genes, cells)) < 0.2)
    m[3, :] = -m[3, :]
    check(cuda, np.asfortranarray(m), cl)


def test_markers_cluster_cap(cuda):
    rng = np.random.default_rng(27)
    genes, cells = 3, 3 * CAP
    cl = labels(rng, cells, CAP)
    m = sc_matrix(rng, genes, cells, density=0.5)
    picked = [0, 1, CAP // 2, CAP - 1] + list(rng.choice(CAP, size=12, replace=False))
    check(cuda, m, cl, clusters=picked)
    cl[7] = CAP                                              # one cluster more than the cap
    with pytest.raises(cuda.GficfCudaError) as e:
        cuda.rcpp_parallel_WMU_markers(m, cl)
    assert e.value.code == 5


def test_markers_timings_and_errors(cuda):
    rng = np.random.default_rng(28)
    m = sc_matrix(rng, 40, 900)
    cl = labels(rng, 900, 4)
    cuda.rcpp_parallel_WMU_markers(m, cl)
    tm = cuda.last_timings()
    assert tm["h2d_ms"] > 0 and tm["jaccard_ms"] > 0 and tm["wall_ms"] >= tm["h2d_ms"]
    with pytest.raises(cuda.GficfCudaError) as e:
        cuda.rcpp_parallel_WMU_markers(m, np.where(cl == 2, 3, cl))  # id 2 has no cells
    assert e.value.code == 1
    assert cuda.rcpp_parallel_WMU_markers(np.ones((0, 6)), np.array([0, 1, 0, 1, 0, 1])).shape == (0, 2, 2)


@pytest.fixture(scope="module")
def rharness(tmp_path_factory):
    import gficf_b200

    so = str(tmp_path_factory.mktemp("rpkg") / "librpkg_markers.so")
    lib = gficf_b200.library_path()
    cmd = ["g++", "-O2", "-std=c++11", "-fPIC", "-shared", "-Wall", "-Werror",
           "-I" + os.path.join(ROOT, "oracle", "rshim"), "-I" + os.path.join(ROOT, "include"),
           "-I" + os.path.join(ROOT, "gficf_b200", "rpkg", "src"), os.path.join(ROOT, "tests", "rpkg_markers_entry.cpp"),
           lib, "-Wl,-rpath," + os.path.dirname(lib), "-o", so]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr[-3000:]
    L = C.CDLL(so)
    L.rpkg_wmu_markers.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_char_p,
                                   C.c_int, C.c_char_p, C.c_int]
    L.rpkg_wmu_markers.restype = C.c_int
    return L


def r_markers(L, m, cl1, k, print_output):
    m = np.asfortranarray(m, dtype=np.float64)
    ids = np.ascontiguousarray(cl1, dtype=np.int32)
    out = np.empty((m.shape[0], 2 * k), dtype=np.float64, order="F")
    err, printed = C.create_string_buffer(1024), C.create_string_buffer(1024)
    rc = L.rpkg_wmu_markers(m.ctypes.data, m.shape[0], m.shape[1], ids.ctypes.data, k, out.ctypes.data,
                            int(print_output), err, 1024, printed, 1024)
    if rc != 0:
        raise RuntimeError(err.value.decode())
    return out, printed.value.decode()


def test_r_export_through_stand_in_runtime(cuda, rharness):
    rng = np.random.default_rng(29)
    genes, cells, k = 40, 1200, 5
    cl = labels(rng, cells, k)
    m = sc_matrix(rng, genes, cells)
    res, text = r_markers(rharness, m, cl + 1, k, True)
    assert text == "Running Parallell WM-U test...\nDone!!\n"
    want = cuda.rcpp_parallel_WMU_markers(m, cl)
    for c in range(k):  # columns 2c-1, 2c (1-based) are cluster c's (p-value, log2FC)
        assert np.array_equal(res[:, 2 * c:2 * c + 2], want[:, :, c], equal_nan=True)
        x, y = np.asfortranarray(m[:, cl == c]), np.asfortranarray(m[:, cl != c])
        assert np.array_equal(res[:, 2 * c:2 * c + 2], WmuOracle().wmu(x, y), equal_nan=True)
    assert r_markers(rharness, m, cl + 1, k, False)[1] == ""
    bad = cl + 1
    bad[3] = 0
    with pytest.raises(RuntimeError) as e:
        r_markers(rharness, m, bad, k, False)
    assert "positive" in str(e.value)
    with pytest.raises(RuntimeError) as e:
        r_markers(rharness, m, np.where(cl == 1, 3, cl + 1), k, False)  # cluster 2 has no cells
    assert "failed (1)" in str(e.value)
