"""CPU: the kernels of the Jaccard path itself (gficf_b200/csrc/jaccard_kernels.cuh) run on the CUDA
emulation (tests/cuda_emu) against the oracle and the golden vectors: layout pre-pass, the
k <= 32 / <= 128 / <= 1024 count kernels (fused, counts, mutual-bit and tagged/grouped outputs),
the exact kernel, expand and compaction.  The no-GPU check of what tests/test_gpu_parity.py runs on the
B200; the five inline-PTX helpers of the header have plain C++ bodies in this build."""
import ctypes as C
import glob
import os
import subprocess

import numpy as np
import pytest

from tests.conftest import random_knn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_dp, _bp, _ll = C.POINTER(C.c_double), C.POINTER(C.c_ubyte), C.POINTER(C.c_longlong)
GOLDEN = sorted(p for p in glob.glob(os.path.join(ROOT, "tests", "golden", "*.npz"))
                if not os.path.basename(p).startswith(("wmu_", "net_")))


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emu") / "libjaccard_emu.so")
    cmd = ["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-DGFICF_CUDA_EMU", "-I" + os.path.join(ROOT, "tests", "cuda_emu"),
           "-I" + os.path.join(ROOT, "gficf_b200", "csrc"), "-shared", "-fPIC", "-Wall", "-Wno-unknown-pragmas", "-Werror",
           os.path.join(ROOT, "tests", "cuda_emu", "jaccard_emu.cpp"), "-o", so]
    out = subprocess.run(cmd, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    L = C.CDLL(so)
    L.emu_jaccard.argtypes = [_dp, C.c_longlong, C.c_int, C.c_int, _dp, _bp, _ll, C.c_int]
    L.emu_jaccard.restype = C.c_uint
    return L


def run(L, idx, mode, grid=3):
    idx = np.asfortranarray(idx, dtype=np.float64)
    n, k = idx.shape
    out = np.full((n * k, 3), -7.0, order="F")
    counts = np.full(n * k + 16, 0xEE, np.uint8)
    nw = np.full(1, -1, np.int64)
    flags = L.emu_jaccard(idx.ctypes.data_as(_dp), n, k, mode, out.ctypes.data_as(_dp), counts.ctypes.data_as(_bp),
                          nw.ctypes.data_as(_ll), grid)
    return out, counts[:n * k].reshape(n, k), int(nw[0]), flags


@pytest.mark.parametrize("path", GOLDEN, ids=[os.path.basename(p)[:-4] for p in GOLDEN])
def test_emulated_kernels_match_golden(emu, path):
    g = np.load(path)
    idx = g["idx"]
    n, k = idx.shape
    distinct = all(len(set(r.tolist())) == k for r in idx)
    out, _, _, flags = run(emu, idx, 0)
    if distinct and k <= 1024:
        assert flags == 0 and np.array_equal(out, g["parallel"])  # the fused kernel
        out, _, _, flags = run(emu, idx, 1)
        assert flags == 0 and np.array_equal(out, g["parallel"])  # counts + expand
    else:
        assert flags & (2 | 4) or flags == 0x80000000  # repeated ids: the fast kernels say so, the exact path answers
    out, _, _, _ = run(emu, idx, 3)
    assert np.array_equal(out, g["parallel"])  # exact kernel, multiset semantics
    out, _, nw, _ = run(emu, idx, 2)
    assert np.array_equal(out, g["serial"])  # exact kernel with set semantics + compaction + zero tail
    assert nw == int((g["serial"][:, 2] > 0).sum())


@pytest.mark.parametrize("n,k", [(300, 1), (257, 4), (400, 7), (500, 15), (230, 16), (333, 27), (400, 30), (200, 32),
                                  (150, 33), (120, 64), (130, 100), (160, 128), (152, 150)])
def test_emulated_fast_kernels_match_oracle(emu, oracle, n, k):
    rng = np.random.default_rng(n + k)
    idx = random_knn(rng, n, k)
    want = oracle.parallel(idx)
    for mode in ((0, 1) if k <= 128 else (0,)):  # the CTA-per-row kernel is slow to emulate
        out, _, _, flags = run(emu, idx, mode, grid=int(rng.integers(1, 4)))
        assert flags == 0, (mode, flags)
        assert np.array_equal(out, want), mode
    if k <= 127:  # counts with the mutual bit (what the graph build reads)
        a = (idx - 1).astype(np.int64)
        sets = [set(r.tolist()) for r in a]
        _, um, _, flags = run(emu, idx, 4)
        assert flags == 0
        u = (want[:, 2] * (2 * k) / (1 + want[:, 2])).round().astype(np.int64).reshape(n, k)  # w = u/(2k-u); slot i*k+j
        mutual = np.array([[i in sets[t] for t in a[i]] for i in range(n)])
        assert np.array_equal(um & 0x7F, u) and np.array_equal((um & 0x80) != 0, mutual)
    if k <= 32:  # parity-tagged counts, rows sent in groups of 8 (the multi-GPU gather's peer kernel)
        _, ut, _, flags = run(emu, idx, 5)
        assert flags == 0 and np.array_equal(ut, u | 0x80)
    if k <= 127:  # both halves of the streaming gather: tagged counts, then the expand that reads (polls) them
        for mode in (6, 7) if k <= 32 else (6,):
            out, ut, _, flags = run(emu, idx, mode, grid=6)  # 6 emulated SMs: 2 CTAs per segment
            assert flags == 0 and np.array_equal(ut, u | 0x80) and np.array_equal(out, want), mode


def test_emulated_layout_flags_bad_ids(emu):
    rng = np.random.default_rng(1)
    idx = random_knn(rng, 100, 10)
    for bad in (0.0, 101.0, 3.5, np.nan, -2.0):
        a = idx.copy()
        a[17, 3] = bad
        assert run(emu, a, 0)[3] & 1, bad
