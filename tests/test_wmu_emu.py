"""CPU: the Mann-Whitney kernels (gficf_b200/csrc/wmu_kernels.cuh) run on the CUDA emulation
(tests/cuda_emu) against the oracle and the golden vectors of the reference's own sources -- the
no-GPU check of what tests/test_gpu_wmu.py runs on the B200."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle.binding import WmuOracle
from tests.test_wmu_oracle import WMU_GOLDEN, sc_matrix

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_dp = C.POINTER(C.c_double)


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emu") / "libwmu_emu.so")
    cmd = ["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-DGFICF_CUDA_EMU", "-I" + os.path.join(ROOT, "tests", "cuda_emu"),
           "-I" + os.path.join(ROOT, "gficf_b200", "csrc"), "-I" + os.path.join(ROOT, "include"), "-shared", "-fPIC", "-Wall", "-Wno-unknown-pragmas", "-Werror",
           os.path.join(ROOT, "tests", "cuda_emu", "wmu_emu.cpp"), os.path.join(ROOT, "gficf_b200", "csrc", "host_stats.cpp"),
           "-o", so]
    out = subprocess.run(cmd, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    L = C.CDLL(so)
    L.emu_wmu_test.argtypes = [_dp, _dp, C.c_longlong, C.c_longlong, C.c_longlong, _dp, C.c_int]
    L.emu_wmu_test.restype = None
    return L


def emu_wmu(L, x, y, grid=3):
    x, y = np.asfortranarray(x, dtype=np.float64), np.asfortranarray(y, dtype=np.float64)
    g = x.shape[0]
    out = np.empty((g, 2), dtype=np.float64, order="F")
    L.emu_wmu_test(x.ctypes.data_as(_dp), y.ctypes.data_as(_dp), g, x.shape[1], y.shape[1], out.ctypes.data_as(_dp), grid)
    return out


@pytest.mark.parametrize("path", WMU_GOLDEN, ids=[os.path.basename(p)[:-4] for p in WMU_GOLDEN])
def test_emulated_wmu_matches_golden(emu, path):
    g = np.load(path)
    assert np.array_equal(emu_wmu(emu, g["x"], g["y"]), g["out"], equal_nan=True)


@pytest.mark.parametrize("genes,n1,n2,integer", [(40, 30, 200, False), (25, 1, 50, False), (33, 64, 64, True),
                                                  (6, 300, 900, False), (12, 7, 5, True)])
def test_emulated_wmu_matches_oracle(emu, genes, n1, n2, integer):
    rng = np.random.default_rng(genes + n1)
    m = sc_matrix(rng, genes, n1 + n2, integer=integer)
    m[0, :] = 3.0           # one tie group: p = 1
    m[1, :] = 0.0
    m[2, :n1] = 0.0         # complete separation
    m[2, n1:] = rng.random(n2) + 1.0
    m[3, :] = -m[3, :]      # negative values
    m[4, ::2] = -0.0        # -0.0 ties with +0.0
    m[5, :] = rng.normal(size=n1 + n2)  # dense, all distinct
    x, y = m[:, :n1], m[:, n1:]
    want = WmuOracle().wmu(x, y, nthreads=2)
    assert np.array_equal(emu_wmu(emu, x, y, grid=int(rng.integers(1, 5))), want, equal_nan=True)
