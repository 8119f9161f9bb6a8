"""CPU: gficf_cuda_wmu_markers_csc, the markers call on a compressed-column (dgCMatrix) matrix, run on the CUDA
emulation (tests/cuda_emu/wmu_markers_sparse_emu.cpp) from the transpose to the host finish, bit for bit
against the emulated dense markers kernels on the densified matrix and against the oracle per cluster.  Also:
the ones-run replay of the means chains against a brute-force loop, the ordered tie term at N = 300 000, the
malformed-matrix checks (host side through the real library, device side on the emulation and under
AddressSanitizer), and the argument errors of the C ABI and of the Python mirror, none of which needs a GPU.
tests/test_gpu_wmu_markers_sparse.py runs the call on the B200.  About 60 s on one CPU core."""
import ctypes as C
import os
import shutil
import subprocess
import sys

import numpy as np
import pytest
import scipy.sparse as sp

import gficf_b200
from oracle.binding import WmuOracle
from tests.sum_order_cases import assert_discriminates, sensitive_genes
from tests.test_wmu_markers_emu import check_blocks, emu_markers, special_rows
from tests.test_wmu_oracle import sc_matrix

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)


def build_emu(so, source, asan=False):
    cmd = ["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-DGFICF_CUDA_EMU", "-I" + os.path.join(ROOT, "tests", "cuda_emu"),
           "-I" + os.path.join(ROOT, "gficf_b200", "csrc"), "-I" + os.path.join(ROOT, "include"), "-shared", "-fPIC",
           "-Wall", "-Wno-unknown-pragmas", "-Werror", os.path.join(ROOT, "tests", "cuda_emu", source),
           os.path.join(ROOT, "gficf_b200", "csrc", "host_stats.cpp"), "-o", so]
    if asan:
        cmd[1:1] = ["-g", "-fsanitize=address", "-fno-omit-frame-pointer", "-DGFICF_NET_ASAN"]
    out = subprocess.run(cmd, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr


def load_sparse_emu(so):
    L = C.CDLL(so)
    L.emu_ones_run.argtypes = [C.c_double, C.c_longlong]
    L.emu_ones_run.restype = C.c_double
    L.emu_wmu_markers_csc.argtypes = [_ip, _ip, _dp, C.c_longlong, C.c_longlong, _ip, C.c_int, _dp, C.c_int, C.c_int]
    L.emu_wmu_markers_csc.restype = C.c_uint
    return L


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emu") / "libwmu_markers_sparse_emu.so")
    build_emu(so, "wmu_markers_sparse_emu.cpp")
    return load_sparse_emu(so)


@pytest.fixture(scope="module")
def dense_emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emu") / "libwmu_markers_emu.so")
    build_emu(so, "wmu_markers_emu.cpp")
    L = C.CDLL(so)
    L.emu_wmu_markers.argtypes = [_dp, C.c_longlong, C.c_longlong, _ip, C.c_int, _dp, C.c_int]
    L.emu_wmu_markers.restype = None
    return L


def to_csc(m, rng=None, stored_zeros=0.0):
    """The CSC slots of m (every non-zero stored), plus a fraction of its zeros stored explicitly, half of
    them as -0.0.  Returns (colptr, row, x, dense): dense is m with those -0.0 written in."""
    m = np.array(m, dtype=np.float64, order="F")
    mask = m != 0
    if stored_zeros:
        extra = (~mask) & (rng.random(m.shape) < stored_zeros)
        m[extra & (rng.random(m.shape) < 0.5)] = -0.0
        mask |= extra
    cols, rows = np.nonzero(mask.T)                     # column-major order, rows ascending in a column
    colptr = np.concatenate([[0], np.cumsum(mask.sum(axis=0))]).astype(np.int32)
    return colptr, rows.astype(np.int32), np.ascontiguousarray(m[rows, cols]), m


def emu_sparse(L, colptr, row, x, genes, cl, k, grid=3, ctas=2):
    cells = colptr.size - 1
    cl = np.ascontiguousarray(cl, dtype=np.int32)
    out = np.full((genes, 2, k), -7.0, order="F")
    flags = L.emu_wmu_markers_csc(colptr.ctypes.data_as(_ip), row.ctypes.data_as(_ip), x.ctypes.data_as(_dp), genes,
                                  cells, cl.ctypes.data_as(_ip), k, out.ctypes.data_as(_dp), grid, ctas)
    return out, flags


def check_sparse(L, dense_L, m, cl, k, grid=3, ctas=2, stored_zeros=0.1, seed=0):
    colptr, row, x, m = to_csc(m, np.random.default_rng(seed), stored_zeros)
    got, flags = emu_sparse(L, colptr, row, x, m.shape[0], cl, k, grid, ctas)
    assert flags == 0
    want = emu_markers(dense_L, m, cl, k, grid)
    assert np.array_equal(got.view(np.int64), want.view(np.int64))
    check_blocks(got, m, cl, k)
    return got


def edge_rows(rng, m, cl):
    """special_rows plus the rows a sparse matrix makes special, written over the next genes."""
    m = special_rows(rng, m, cl)
    cells = m.shape[1]
    m[7, :] = 0.0                                                       # no stored value (with no stored zeros)
    m[8, :] = rng.random(cells) + 0.5                                   # every cell stored
    m[9, :] = np.where(rng.random(cells) < 0.3, -rng.random(cells) * 5 - 1.0, 0.0)  # below -1: chains go negative
    m[10, :] = np.where(rng.random(cells) < 0.2, rng.choice([1e16, 3e16, 1e17, 2 ** 53 - 1.0], cells), 0.0)  # past 2^53
    m[11, :] = np.where(rng.random(cells) < 0.3, 5e-324 * rng.integers(1, 9, cells), 0.0)  # subnormals
    m[12, :] = np.where(rng.random(cells) < 0.1, -(2.0 ** 53) - 2.0, 0.0)  # chains that start below -2^53
    return m


@pytest.mark.parametrize("genes,cells,k,integer,grid,ctas", [
    (16, 300, 2, False, 3, 1),
    (24, 1500, 9, False, 5, 3),
    (14, 800, 30, True, 1, 2),     # many tie groups, one CTA for every gene
    (13, 2500, 40, True, 7, 4),    # two CTAs of the means kernel per gene
])
def test_emulated_sparse_markers_match_dense_and_oracle(emu, dense_emu, genes, cells, k, integer, grid, ctas):
    rng = np.random.default_rng(genes * 31 + k)
    cl = rng.integers(0, k, size=cells).astype(np.int32)
    cl[:k] = np.arange(k)
    rng.shuffle(cl)
    m = edge_rows(rng, sc_matrix(rng, genes, cells, integer=integer), cl)
    m[:, [0, 1, cells // 2, cells - 1]] = 0.0                           # empty columns: start, middle, end
    check_sparse(emu, dense_emu, m, cl, k, grid, ctas, seed=k)


def test_emulated_sparse_markers_one_cell_clusters(emu, dense_emu):
    rng = np.random.default_rng(5)
    cells = 400
    cl = rng.integers(2, 5, size=cells).astype(np.int32)
    cl[137], cl[0] = 0, 1                                               # two clusters of one cell each
    m = edge_rows(rng, sc_matrix(rng, 14, cells), cl)
    check_sparse(emu, dense_emu, m, cl, 5, grid=4)
    cl = np.ones(cells, dtype=np.int32)
    cl[399] = 0                                                          # one cell against n - 1
    check_sparse(emu, dense_emu, m, cl, 2, grid=2, stored_zeros=0.5)


def test_emulated_sparse_markers_without_stored_values(emu, dense_emu):
    """An all-zero matrix, stored as nothing and as explicit zeros only."""
    cl = np.array([0, 1, 2, 0, 1, 2, 0], dtype=np.int32)
    m = np.zeros((3, 7))
    check_sparse(emu, dense_emu, m, cl, 3, stored_zeros=0.0)
    check_sparse(emu, dense_emu, m, cl, 3, stored_zeros=0.6, seed=2)


def brute_ones(s, m):
    for _ in range(m):
        s = s + 1.0
    return s


def test_ones_run_replay_matches_the_loop(emu):
    rng = np.random.default_rng(9)
    starts = [0.0, -0.0, 5e-324, 2.5e-310, 0.3, 0.7, 1.0, 1.5, 2.0 - 2 ** -52, 1023.999, 2.0 ** 30 - 0.5,
              2.0 ** 53 - 1, 2.0 ** 53, 2.0 ** 53 + 2, 2.0 ** 52 + 0.5, -0.3, -1.0, -2.5, -(2.0 ** 53) - 2,
              -(2.0 ** 53), -(2.0 ** 60), 1e300, -1e300, 1e16, 3e16 + 4] + list(rng.normal(0, 1e3, 200)) + \
        list(rng.random(100) * 2.0 ** rng.integers(-30, 60, 100)) + list(-rng.random(100) * 2.0 ** rng.integers(-30, 60, 100))
    for s in starts:
        for m in (0, 1, 2, 3, 1000, 70_001):
            got, want = emu.emu_ones_run(s, m), brute_ones(s, m)
            assert np.float64(got).view(np.int64) == np.float64(want).view(np.int64), (s, m, got, want)


def test_emulated_sparse_markers_ordered_tie_sum(emu, dense_emu):
    """N = 300 000 >= 208 064: the tie term is the reference's sequential double sum in sorted order, on genes
    where another order gives another p-value (tests/sum_order_cases.py)."""
    n = 300_000
    rng = np.random.default_rng(3)
    cl = rng.integers(0, 3, n).astype(np.int32)
    cl[rng.integers(0, n)] = 3
    m, against = sensitive_genes(2, n, cl == 1, ("shifted", "negative"))
    orc = WmuOracle()
    for v, a in zip(m, against):
        assert_discriminates(v, [cl == c for c in range(4)], orc, a)
    colptr, row, x, m = to_csc(m)
    got, flags = emu_sparse(emu, colptr, row, x, m.shape[0], cl, 4, grid=2)
    assert flags == 0
    check_blocks(got, m, cl, 4)


def malformed_cases():
    """(name, colptr, row) of a valid 5 x 4 matrix with one defect each that only the device pass sees."""
    colptr = np.array([0, 2, 2, 5, 6], dtype=np.int32)
    row = np.array([0, 3, 1, 2, 4, 0], dtype=np.int32)
    cases = []
    for name, pos, val in (("row id negative", 1, -1), ("row id = n_genes", 4, 5), ("row id far out", 0, 1 << 30),
                           ("duplicate row id", 3, 1), ("decreasing row ids", 4, 0)):
        r = row.copy()
        r[pos] = val
        cases.append((name, colptr, r))
    return cases


def test_emulated_malformed_rows_raise_the_flag(emu):
    cl = np.array([0, 1, 0, 1], dtype=np.int32)
    x = np.arange(1.0, 7.0)
    for name, colptr, row in malformed_cases():
        out, flags = emu_sparse(emu, colptr, row, x, 5, cl, 2)
        assert flags == 1, name
        assert (out == -7.0).all(), name
    out, flags = emu_sparse(emu, np.array([0, 2, 2, 5, 6], np.int32), np.array([0, 3, 1, 2, 4, 0], np.int32), x, 5, cl, 2)
    assert flags == 0 and not (out == -7.0).any()


def test_emulated_sparse_pipeline_under_address_sanitizer(tmp_path):
    """The transpose and both kernels on valid and malformed input, built with -fsanitize=address, every
    scratch piece fenced by a poisoned red zone and the inputs in exactly-sized heap arrays: an index that
    leaves its array is reported.  Runs in a child process (the sanitizer runtime has to be loaded first)."""
    libasan = subprocess.run(["g++", "-print-file-name=libasan.so"], capture_output=True, text=True).stdout.strip()
    if not shutil.which("g++") or not os.path.isabs(libasan) or not os.path.exists(libasan):
        pytest.skip("no AddressSanitizer runtime next to g++")
    so = str(tmp_path / "libwmu_markers_sparse_emu_asan.so")
    build_emu(so, "wmu_markers_sparse_emu.cpp", asan=True)
    env = dict(os.environ, LD_PRELOAD=libasan, ASAN_OPTIONS="detect_leaks=0:abort_on_error=0:exitcode=23",
               PYTHONPATH=ROOT)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "cuda_emu", "asan_markers_sparse_run.py"), so],
                         capture_output=True, text=True, env=env, timeout=900)
    assert "ERROR: AddressSanitizer" not in out.stderr, out.stderr[-4000:]
    assert out.returncode == 0, (out.stdout[-2000:], out.stderr[-2000:])
    assert "asan run ok" in out.stdout


def _abi(colptr, row, x, genes, cl, k, cells=None):
    L = gficf_b200.lib()
    err = C.create_string_buffer(256)
    out = np.empty(64)  # every call here fails or returns before the output is written
    p = lambda a: None if a is None else a.ctypes.data  # noqa: E731
    cells = (colptr.size - 1 if colptr is not None else 0) if cells is None else cells
    rc = L.gficf_cuda_wmu_markers_csc(p(colptr), p(row), p(x), genes, cells, p(cl), k, out.ctypes.data, err, 256)
    return rc, err.value.decode()


def test_sparse_markers_argument_errors_without_gpu():
    """Checked on the host before any device is touched: the same codes with or without a GPU."""
    colptr = np.array([0, 2, 2, 5, 6], dtype=np.int32)
    row = np.array([0, 3, 1, 2, 4, 0], dtype=np.int32)
    x = np.arange(1.0, 7.0)
    cl = np.array([0, 1, 0, 1], dtype=np.int32)
    rc, msg = _abi(np.array([1, 2, 2, 5, 6], dtype=np.int32), row, x, 5, cl, 2)    # colptr[0] != 0
    assert rc == 1 and "colptr[0]" in msg
    rc, msg = _abi(np.array([0, 2, 1, 5, 6], dtype=np.int32), row, x, 5, cl, 2)    # colptr decreasing
    assert rc == 1 and "decreases" in msg
    assert _abi(np.array([0, -1, 2, 5, 6], dtype=np.int32), row, x, 5, cl, 2)[0] == 1
    assert _abi(colptr, row, x, -1, cl, 2)[0] == 1                                   # negative size
    assert _abi(colptr, row, x, 5, cl, 2, cells=-1)[0] == 1
    assert _abi(None, row, x, 5, cl, 2, cells=4)[0] == 1                             # null pointers
    assert _abi(colptr, None, x, 5, cl, 2)[0] == 1
    assert _abi(colptr, row, None, 5, cl, 2)[0] == 1
    assert _abi(colptr, row, x, 5, None, 2)[0] == 1
    assert _abi(colptr, row, x, 5, np.zeros(4, np.int32), 1)[0] == 1               # fewer than two clusters
    rc, msg = _abi(colptr, row, x, 5, np.array([0, 1, 2, 1], np.int32), 2)          # id outside [0, n_clusters)
    assert rc == 1 and "outside" in msg
    rc, msg = _abi(colptr, row, x, 5, np.array([0, 2, 0, 2], np.int32), 3)          # cluster 1 has no cells
    assert rc == 1 and "no cells" in msg
    assert _abi(colptr, row, x, 5, cl, 8193)[0] == 5                                 # above the cluster cap
    assert _abi(colptr, row, x, 5, cl, 2, cells=1 << 31)[0] == 5                     # 2^31 cells
    assert _abi(colptr, row, x, 1 << 31, cl, 2)[0] == 5                              # 2^31 genes
    assert _abi(colptr, row, x, 0, cl, 2)[0] == 0                                    # no genes: nothing to do


def test_sparse_markers_mirror_argument_errors():
    m = sp.csc_matrix(np.eye(4, 6))
    f = gficf_b200.rcpp_parallel_WMU_markers_sparse
    with pytest.raises(TypeError):
        f(m.toarray(), np.array([0, 1, 0, 1, 0, 1]))                             # dense
    with pytest.raises(TypeError):
        f(m.tocsr(), np.array([0, 1, 0, 1, 0, 1]))                               # another sparse format
    with pytest.raises(TypeError):
        f(sp.coo_matrix(m), np.array([0, 1, 0, 1, 0, 1]))
    with pytest.raises(ValueError):
        f(m, np.array([0, 1, 0, 1, 0]))                                          # one id per cell
    with pytest.raises(TypeError):
        f(m, np.array([0.0, 1, 0, 1, 0, 1]))
    with pytest.raises(ValueError):
        f(m, np.array([0, 1, 0, -1, 0, 1]))
    big = m.copy()
    big.indices = big.indices.astype(np.int64)
    big.indices[0] = 1 << 33                                                     # does not fit in int32
    with pytest.raises(ValueError):
        f(big, np.array([0, 1, 0, 1, 0, 1]))
    bad = m.copy()
    bad.indptr = bad.indptr.astype(np.int32)
    bad.indptr[0] = 1                                                            # reaches the library's check
    with pytest.raises(gficf_b200.GficfCudaError) as e:
        f(bad, np.array([0, 1, 0, 1, 0, 1]))
    assert e.value.code == 1
    with pytest.raises(gficf_b200.GficfCudaError) as e:
        f(m, np.array([0, 2, 0, 2, 0, 2]))                                        # cluster 1 is empty
    assert e.value.code == 1
    assert f(sp.csc_matrix((0, 6)), np.array([0, 1, 0, 1, 0, 1])).shape == (0, 2, 2)
    if hasattr(sp, "csc_array"):                                                 # the array form is accepted too
        with pytest.raises(gficf_b200.GficfCudaError) as e:
            f(sp.csc_array(m), np.array([0, 2, 0, 2, 0, 2]))
        assert e.value.code == 1
