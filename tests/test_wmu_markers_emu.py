"""CPU: the one-vs-rest kernels of gficf_cuda_wmu_markers (gficf_b200/csrc/wmu_kernels.cuh) run on the
CUDA emulation (tests/cuda_emu) with the host half of the call: every cluster's block against the oracle
run on that cluster's split.  Also the argument checks of the C ABI and the Python mirror, which need no
GPU.  tests/test_gpu_wmu_markers.py runs the same on the B200."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import gficf_b200
from oracle.binding import WmuOracle
from tests.test_wmu_oracle import sc_matrix

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emu") / "libwmu_markers_emu.so")
    cmd = ["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-DGFICF_CUDA_EMU", "-I" + os.path.join(ROOT, "tests", "cuda_emu"),
           "-I" + os.path.join(ROOT, "gficf_b200", "csrc"), "-shared", "-fPIC", "-Wall", "-Wno-unknown-pragmas", "-Werror",
           os.path.join(ROOT, "tests", "cuda_emu", "wmu_markers_emu.cpp"),
           os.path.join(ROOT, "gficf_b200", "csrc", "host_stats.cpp"), "-o", so]
    out = subprocess.run(cmd, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    L = C.CDLL(so)
    L.emu_wmu_markers.argtypes = [_dp, C.c_longlong, C.c_longlong, _ip, C.c_int, _dp, C.c_int]
    L.emu_wmu_markers.restype = None
    return L


def emu_markers(L, m, cl, k, grid):
    m = np.asfortranarray(m, dtype=np.float64)
    cl = np.ascontiguousarray(cl, dtype=np.int32)
    out = np.empty((m.shape[0], 2, k), dtype=np.float64, order="F")
    L.emu_wmu_markers(m.ctypes.data_as(_dp), m.shape[0], m.shape[1], cl.ctypes.data_as(_ip), k, out.ctypes.data_as(_dp),
                      grid)
    return out


def special_rows(rng, m, cl):
    """Rows the reference treats specially, written over the first genes."""
    cells = m.shape[1]
    m[0, :] = 3.0                                    # one tie group: p = 1 for every cluster
    m[1, :] = 0.0
    m[2, :] = -m[2, :]                               # negative values
    m[3, ::2] = -0.0                                 # -0.0 ties with +0.0
    m[4, :] = np.where(cl == 0, 0.0, rng.random(cells) + 1.0)  # cluster 0 completely separated
    m[5, :] = rng.normal(size=cells)                 # dense, all distinct
    m[6, :] = np.where(rng.random(cells) < 0.5, -2.0, 0.0)     # negative ties before the zeros
    return m


def check_blocks(got, m, cl, k):
    assert got.shape == (m.shape[0], 2, k)
    orc = WmuOracle()
    for c in range(k):
        want = orc.wmu(np.asfortranarray(m[:, cl == c]), np.asfortranarray(m[:, cl != c]), nthreads=2)
        assert np.array_equal(got[:, :, c], want, equal_nan=True), c


@pytest.mark.parametrize("genes,cells,k,integer,grid", [
    (20, 300, 2, False, 3),      # two clusters
    (24, 1500, 9, False, 5),     # interleaved labels, more genes than CTAs
    (12, 800, 30, True, 1),      # many tie groups, one CTA for every gene
    (9, 2500, 4, True, 7),
])
def test_emulated_markers_match_oracle(emu, genes, cells, k, integer, grid):
    rng = np.random.default_rng(genes * 31 + k)
    cl = rng.integers(0, k, size=cells).astype(np.int32)
    cl[:k] = np.arange(k)                            # every id has cells
    rng.shuffle(cl)
    m = special_rows(rng, sc_matrix(rng, genes, cells, integer=integer), cl)
    check_blocks(emu_markers(emu, m, cl, k, grid), m, cl, k)


def test_emulated_markers_cluster_of_one_cell(emu):
    """A cluster of one cell and one of n - 1 cells (the same split, seen from both sides), and a
    three-way split with a singleton."""
    rng = np.random.default_rng(5)
    cells = 400
    m = special_rows(rng, sc_matrix(rng, 10, cells), np.zeros(cells))
    cl = np.ones(cells, dtype=np.int32)
    cl[137] = 0
    check_blocks(emu_markers(emu, m, cl, 2, 4), m, cl, 2)
    cl = rng.integers(1, 3, size=cells).astype(np.int32)
    cl[0] = 0
    check_blocks(emu_markers(emu, m, cl, 3, 2), m, cl, 3)


def _abi(m, cl, k, genes=None, cells=None, out=None):
    L = gficf_b200.lib()
    err = C.create_string_buffer(256)
    if out is None:
        out = np.empty((m.shape[0], 2, max(k, 1)), order="F")
    rc = L.gficf_cuda_wmu_markers(None if m is None else m.ctypes.data, m.shape[0] if genes is None else genes,
                                  m.shape[1] if cells is None else cells, None if cl is None else cl.ctypes.data, k,
                                  out.ctypes.data, err, 256)
    return rc, err.value.decode()


def test_markers_argument_errors_without_gpu():
    """Checked before any device is touched: the same codes with or without a GPU."""
    m = np.asfortranarray(np.ones((4, 6)))
    cl = np.array([0, 1, 2, 0, 1, 2], dtype=np.int32)
    assert _abi(m, cl, 3, genes=-1)[0] == 1
    assert _abi(m, cl, 3, cells=-1)[0] == 1
    assert _abi(None, cl, 3, genes=4, cells=6, out=np.empty((4, 2, 3), order="F"))[0] == 1
    assert _abi(m, None, 3)[0] == 1
    assert _abi(m, np.zeros(6, dtype=np.int32), 1)[0] == 1             # fewer than two clusters
    rc, msg = _abi(m, np.array([0, 1, 3, 0, 1, 2], dtype=np.int32), 3)  # id outside [0, n_clusters)
    assert rc == 1 and "outside" in msg
    assert _abi(m, np.array([0, 1, -1, 0, 1, 2], dtype=np.int32), 3)[0] == 1
    rc, msg = _abi(m, np.array([0, 1, 0, 0, 1, 1], dtype=np.int32), 3)  # cluster 2 has no cells
    assert rc == 1 and "no cells" in msg
    assert _abi(m, cl, 8193)[0] == 5                                   # above the cluster cap
    assert _abi(m, cl, 3, cells=1 << 31)[0] == 5                       # 2^31 cells
    assert _abi(np.ones((0, 6), order="F"), cl, 3)[0] == 0             # no genes: nothing to do


def test_markers_mirror_argument_errors():
    m = np.ones((4, 6))
    with pytest.raises(ValueError):
        gficf_b200.rcpp_parallel_WMU_markers(m, np.array([0, 1, 0, 1, 0]))
    with pytest.raises(TypeError):
        gficf_b200.rcpp_parallel_WMU_markers(m, np.array([0.0, 1, 0, 1, 0, 1]))
    with pytest.raises(ValueError):
        gficf_b200.rcpp_parallel_WMU_markers(m, np.array([0, 1, 0, -1, 0, 1]))
    with pytest.raises(TypeError):
        gficf_b200.rcpp_parallel_WMU_markers(np.ones(6), np.array([0, 1, 0, 1, 0, 1]))
    with pytest.raises(gficf_b200.GficfCudaError) as e:
        gficf_b200.rcpp_parallel_WMU_markers(m, np.array([0, 2, 0, 2, 0, 2]))  # cluster 1 is empty
    assert e.value.code == 1
