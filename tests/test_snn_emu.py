"""CPU: the graph-build kernels (gficf_b200/csrc/snn_kernels.cuh) run on the CUDA emulation
(tests/cuda_emu) against the reference's steps restated in oracle/louvain.py -- the no-GPU check of
what tests/test_gpu_snn.py runs on the B200 (vertex numbering incl. target-only / absent cells,
lower-triangle CSC, summed mutual weights, all column-sort variants)."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import gficf_b200
from gficf_b200 import synth
from oracle import louvain

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_ll, _ip, _dp, _bp = C.POINTER(C.c_longlong), C.POINTER(C.c_int), C.POINTER(C.c_double), C.POINTER(C.c_ubyte)


@pytest.fixture(scope="module")
def emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emu") / "libsnn_emu.so")
    cmd = ["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-DGFICF_CUDA_EMU", "-I" + os.path.join(ROOT, "tests", "cuda_emu"),
           "-I" + os.path.join(ROOT, "gficf_b200", "csrc"), "-I" + os.path.join(ROOT, "include"), "-shared", "-fPIC", "-Wall", "-Wno-unknown-pragmas", "-Werror",
           os.path.join(ROOT, "tests", "cuda_emu", "snn_emu.cpp"), "-o", so]
    out = subprocess.run(cmd, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    L = C.CDLL(so)
    L.emu_snn_lower.argtypes = [_ip, C.c_longlong, C.c_int, C.c_int, _bp, _ll, _ip, _dp, _ip, _ll, _ll, C.c_int, C.c_int]
    L.emu_snn_lower.restype = C.c_uint
    return L


def counts_with_mutual_bit(idx):
    """What the count kernel leaves for the graph build: u(i, j) in bits 0-6, bit 7 = i is in N(idx[i, j])."""
    n, k = idx.shape
    sets = [set(r.tolist()) for r in idx]
    um = np.zeros((n, k), np.uint8)
    for i in range(n):
        for j, t in enumerate(idx[i].tolist()):
            um[i, j] = len(sets[i] & sets[t]) | (0x80 if i in sets[t] else 0)
    return um


def emu_lower(L, idx, max_ctas=2, sort_ctas=2, um=None):
    n, k = idx.shape
    kp = int(gficf_b200.lib().gficf_cuda_row_stride(k))
    padded = np.full((n, kp), -2, np.int32)
    padded[:, :k] = idx
    if um is None:
        um = counts_with_mutual_bit(idx)
    colptr = np.zeros(n + 1, np.int64)
    row, w, vcell = np.zeros(n * k, np.int32), np.zeros(n * k), np.zeros(n, np.int32)
    nv, nnz = C.c_longlong(0), C.c_longlong(0)
    p = lambda a, t: a.ctypes.data_as(t)  # noqa: E731
    flags = L.emu_snn_lower(p(padded, _ip), n, k, kp, p(um, _bp), p(colptr, _ll), p(row, _ip), p(w, _dp), p(vcell, _ip),
                            C.byref(nv), C.byref(nnz), max_ctas, sort_ctas)
    return colptr[:nv.value + 1], row[:nnz.value], w[:nnz.value], vcell[:nv.value], flags


def check(L, oracle, idx0, um=None):
    idx = idx0.numpy() if hasattr(idx0, "numpy") else idx0
    names, cols, rows_ref, data_ref = louvain.lower_triangle_edges(oracle.parallel(synth.to_r_matrix(idx0)))
    colptr, rows, w, vcell, flags = emu_lower(L, idx, um=um)
    assert flags & ~16 == 0
    assert np.array_equal(vcell, names.astype(np.int64))  # igraph's vertex numbering
    assert np.array_equal(np.repeat(np.arange(names.size), np.diff(colptr)), cols)
    assert np.array_equal(rows, rows_ref) and np.array_equal(w, data_ref)  # bit-exact sums
    return flags, colptr


@pytest.mark.parametrize("n,k,family", [(600, 15, "planted"), (400, 30, "planted"), (300, 7, "planted"),
                                         (500, 5, "uniform"), (2500, 4, "uniform"), (300, 40, "planted")])
def test_emulated_lower_triangle_matches_reference_steps(emu, oracle, n, k, family):
    import torch  # noqa: F401  (synth returns torch tensors)

    flags, _ = check(emu, oracle, synth.knn_index(n, k, family=family, scramble=True))
    if family == "uniform":
        assert flags & 16  # cells without an edge of their own: the vertex numbering differs from the cell numbering


def test_emulated_hub_columns_take_the_big_sorts(emu, oracle):
    """Columns beyond 32 and 512 entries: warp rank sort and the shared-memory bitonic sort of
    snn_sort_big_kernel (dynamic shared memory in the emulation)."""
    import torch

    n, k = 1500, 8
    rng = np.random.default_rng(4)
    idx = synth.knn_index(n, k, family="planted", scramble=False).numpy().copy()
    for hub, fans in ((0, 900), (1, 120)):
        for r in rng.choice(np.arange(10, n), fans, replace=False):
            if hub not in idx[r]:
                idx[r, rng.integers(0, k)] = hub
    idx[:, 0] = np.where((idx[:, 1:] == 5).any(axis=1) | (np.arange(n) == 5), idx[:, 0], 5)  # a shared neighbour: u > 0
    if any(len(set(r.tolist())) < k for r in idx):
        pytest.skip("the construction produced a repeated id")
    _, colptr = check(emu, oracle, torch.from_numpy(idx))
    assert np.diff(colptr).max() > 512


@pytest.fixture(scope="module")
def jaccard_emu(tmp_path_factory):
    from tests.test_jaccard_slabs_emu import _build

    return _build(str(tmp_path_factory.mktemp("emu") / "libjaccard_emu.so"), [])


@pytest.mark.parametrize("n,k", [(300, 7), (400, 30), (200, 64)])
def test_emulated_graph_with_self_ids_from_the_count_kernel(emu, jaccard_emu, oracle, n, k):
    """Duplicate cells are common in real data, so a cell can be in its own list after neigh[, -1]: rows
    that list themselves (a self loop with u = k) mixed with rows that do not.  The
    mutual-bit counts come from the emulated count kernel (mode 4), as on the device."""
    from tests.test_jaccard_slabs_emu import run_slab, self_ids

    rng = np.random.default_rng(n + k)
    r = self_ids(rng, k, n)
    keep = rng.random(n) < 0.5  # half the rows drop their self id again
    a = (r - 1).astype(np.int64)
    for i in np.flatnonzero(keep):
        j = int(np.flatnonzero(a[i] == i)[0])
        free = np.setdiff1d(np.arange(n), np.append(a[i], i))
        a[i, j] = rng.choice(free)
    idx = a.astype(np.int32)
    _, um, _, flags = run_slab(jaccard_emu, idx + 1.0, 4, 0, n, grid=3)
    assert flags == 0
    assert np.array_equal(um, counts_with_mutual_bit(idx))
    import torch

    check(emu, oracle, torch.from_numpy(idx), um=um.astype(np.uint8))
