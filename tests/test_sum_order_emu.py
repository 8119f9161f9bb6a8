"""CPU: the two sums that must follow the reference's order, on inputs where the order changes the
result (tests/sum_order_cases.py), through the CUDA emulation (tests/cuda_emu):

* the Mann-Whitney tie term above N = 208 064 (wmu_tie_groups in wmu_kernels.cuh), through both rank
  kernels, against the oracle -- on genes where an integer sum or a "zero group first" sum would give
  another p-value;
* the exact replay of std::accumulate (net_seq_sum) past the largest window, on ties-heavy input, and
  on runs of leading zeros, whose cost is pinned by the number of launches.

tests/test_gpu_sum_order.py runs the same inputs on the B200."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle.binding import WmuOracle
from tests.network_cases import seq_sum
from tests.sum_order_cases import (SEQ_MAX_BLOCKS, assert_discriminates, capped_crossings, jaccard_weights,
                                   order_sensitive_gene, sensitive_genes, tie_weights, window_schedule,
                                   with_long_binade)
from tests.test_network_emu import _emu_seq, compile_emu, load_emu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_dp, _ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)


def _build_wmu(so, source):
    cmd = ["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-DGFICF_CUDA_EMU", "-I" + os.path.join(ROOT, "tests", "cuda_emu"),
           "-I" + os.path.join(ROOT, "gficf_b200", "csrc"), "-I" + os.path.join(ROOT, "include"), "-shared", "-fPIC", "-Wall", "-Wno-unknown-pragmas", "-Werror",
           os.path.join(ROOT, "tests", "cuda_emu", source), os.path.join(ROOT, "gficf_b200", "csrc", "host_stats.cpp"),
           "-o", so]
    out = subprocess.run(cmd, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    return C.CDLL(so)


@pytest.fixture(scope="module")
def wmu_emu(tmp_path_factory):
    L = _build_wmu(str(tmp_path_factory.mktemp("emu") / "libwmu_emu.so"), "wmu_emu.cpp")
    L.emu_wmu_test.argtypes = [_dp, _dp, C.c_longlong, C.c_longlong, C.c_longlong, _dp, C.c_int]
    L.emu_wmu_test.restype = None
    return L


@pytest.fixture(scope="module")
def markers_emu(tmp_path_factory):
    L = _build_wmu(str(tmp_path_factory.mktemp("emu") / "libwmu_markers_emu.so"), "wmu_markers_emu.cpp")
    L.emu_wmu_markers.argtypes = [_dp, C.c_longlong, C.c_longlong, _ip, C.c_int, _dp, C.c_int]
    L.emu_wmu_markers.restype = None
    return L


@pytest.fixture(scope="module")
def net_emu(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emu") / "libnetwork_emu.so")
    compile_emu(so)
    L = load_emu(so)
    L.emu_launch_count.restype = C.c_longlong
    return L


N = 300_000   # the smallest order-sensitive gene needs N^3 > 2^54 (N > 262 144)
N1 = 40_000   # the two-group test: cells [0, N1) against the rest


def boundary_gene(seed, n):
    """A large zero group at N = 208 063 (integer tie term) and N = 208 064 (ordered tie term): checks
    the switch between the two, not the order (below 2^53 every order gives the same sum)."""
    return np.asfortranarray(order_sensitive_gene(np.random.default_rng(seed), n, 200_000)[None, :])


def emu_wmu(L, m, n1, grid):
    x, y = np.asfortranarray(m[:, :n1]), np.asfortranarray(m[:, n1:])
    out = np.empty((m.shape[0], 2), order="F")
    L.emu_wmu_test(x.ctypes.data_as(_dp), y.ctypes.data_as(_dp), m.shape[0], n1, m.shape[1] - n1,
                   out.ctypes.data_as(_dp), grid)
    return out, WmuOracle().wmu(x, y)


def test_emulated_wmu_ordered_tie_sum(wmu_emu):
    first = np.arange(N) < N1
    m, against = sensitive_genes(1, N, first, ("shifted", "negative", "dense"))
    orc = WmuOracle()
    for v, a in zip(m, against):
        assert_discriminates(v, [first], orc, a)
    got, want = emu_wmu(wmu_emu, m, N1, grid=3)
    assert np.array_equal(got, want, equal_nan=True)


@pytest.mark.parametrize("n", [208_063, 208_064])
def test_emulated_wmu_tie_sum_branch_switch(wmu_emu, n):
    m = boundary_gene(n, n)
    got, want = emu_wmu(wmu_emu, m, 30_000, grid=2)
    assert np.array_equal(got, want, equal_nan=True)


def markers_labels(seed, n):
    """Three interleaved clusters and a cluster of one cell."""
    rng = np.random.default_rng(seed)
    cl = rng.integers(0, 3, n).astype(np.int32)
    cl[rng.integers(0, n)] = 3
    return cl


def emu_markers_check(L, m, cl, grid, against=None):
    k = int(cl.max()) + 1
    out = np.empty((m.shape[0], 2, k), order="F")
    L.emu_wmu_markers(m.ctypes.data_as(_dp), m.shape[0], m.shape[1], cl.ctypes.data_as(_ip), k,
                      out.ctypes.data_as(_dp), grid)
    orc = WmuOracle()
    if against is not None:
        for v, a in zip(m, against):
            assert_discriminates(v, [cl == c for c in range(k)], orc, a)
    for c in range(k):
        want = orc.wmu(np.asfortranarray(m[:, cl == c]), np.asfortranarray(m[:, cl != c]))
        assert np.array_equal(out[:, :, c], want, equal_nan=True), c


def test_emulated_markers_ordered_tie_sum(markers_emu):
    cl = markers_labels(2, N)
    m, against = sensitive_genes(2, N, cl == 1, ("shifted", "negative"))
    emu_markers_check(markers_emu, m, cl, 2, against)


@pytest.mark.parametrize("n", [208_063, 208_064])
def test_emulated_markers_tie_sum_branch_switch(markers_emu, n):
    emu_markers_check(markers_emu, boundary_gene(n + 1, n), markers_labels(n, n), 3)


# ---- the exact sum ---------------------------------------------------------------------------------

@pytest.mark.parametrize("family,n,s0,ctas", [("jaccard", 6_000_000, 0.0, 3), ("ties", 4_700_000, 0.0, 2),
                                               ("ties", 4_700_000, 7.25, 4)])
def test_emulated_seq_sum_past_the_window_cap(net_emu, family, n, s0, ctas):
    """Past the largest window of the replay: 6M SNN weights run capped windows to the end; the tie-heavy
    family behind one large element meets a binade crossing inside a capped window."""
    rng = np.random.default_rng(1)
    x = jaccard_weights(rng, n) if family == "jaccard" else with_long_binade(tie_weights(rng, n))
    assert any(b == SEQ_MAX_BLOCKS for _, b, _ in window_schedule(x, s0))
    if family == "ties":
        assert capped_crossings(x, s0)
    got, flags = _emu_seq(net_emu, x, s0, ctas=ctas)
    assert flags == 0
    assert got == seq_sum(x, s0), (got, seq_sum(x, s0))


def test_emulated_seq_sum_leading_zeros(net_emu):
    """A masked sum whose first entries are all masked out: the zeros are consumed a window at a time
    (a few dozen launches), not one element per step -- and the bits are the loop's."""
    rng = np.random.default_rng(4)
    tail = rng.random(300)
    # (x, s0, launch bound): a few dozen launches however long the run of zeros; inside the subnormal
    # binade every non-zero element is an addition of its own, whatever precedes it
    cases = [(np.concatenate([np.zeros(z), tail]), 0.0, 64) for z in (0, 1, 4095, 4096, 4097, 200_000)]
    cases += [
        (np.zeros(50_000), 0.0, 64),                                                   # all zeros
        (np.concatenate([np.zeros(100_000), tail]), 3.5, 64),                          # s0 > 0
        (np.zeros(0), 3.0, 64),                                                        # empty
        (np.zeros(3000), -0.0, 64),                                                    # -0.0 + 0.0 is +0.0
        (np.concatenate([np.zeros(10_000), [5e-324, 1e-310, 2.5e-308], rng.random(50) * 1e-300]), 0.0, None),
        (np.concatenate([np.zeros(10_000), 2.0 ** -1074 * rng.integers(1, 9, 200)]), 0.0, None),
    ]
    for x, s0, bound in cases:
        before = net_emu.emu_launch_count()
        got, flags = _emu_seq(net_emu, x, s0, ctas=3)
        launches = net_emu.emu_launch_count() - before
        assert flags == 0
        assert got == seq_sum(x, s0) and np.signbit(got) == np.signbit(seq_sum(x, s0)), (x.size, s0, got)
        assert bound is None or launches <= bound, (x.size, s0, launches)
    # a negative value inside the run of zeros is still flagged
    x = np.zeros(20_000)
    x[15_000] = -1.0
    assert _emu_seq(net_emu, x)[1] & 32
