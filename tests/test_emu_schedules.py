"""CPU: every kernel family of the CUDA emulation (tests/cuda_emu) under permuted schedules.

The emulation runs one fibre per CUDA thread.  By default the runnable fibres of a round run in
ascending threadIdx.x and the CTAs of a launch in ascending blockIdx, so a missing barrier where a
lower thread writes and a higher one reads, results that depend on the order of atomics (the cursors
of snn_edges_kernel<true>, the compaction order of wmu_load, the atomicCAS probes of the large-k
Jaccard kernel, the atomicMin of snn_targets_kernel<0>), "whichever writer survives" slot stores, and
a CTA that reads what a lower-numbered CTA of the same launch wrote can never fail there.
`emu_set_schedule` (cuda_emu.h) runs the same launches in descending order or in a seeded random
permutation redrawn every round.  Here each family runs representative shapes under descending and
two random seeds and must give the bits of the ascending run, which must equal the family's oracle.

Also: the schedules themselves (the order threads and CTAs actually run in, the same run for the same
seed, dynamic shared memory poisoned per CTA), the aborts that must survive them (divergent
__syncthreads, partial masks, collectives after lanes exit), and a barrier removed from a product
kernel that passes in ascending order and fails under the permuted schedules."""
import contextlib
import ctypes as C
import os
import re
import shutil
import subprocess
import sys
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMU = os.path.join(ROOT, "tests", "cuda_emu")
CSRC = os.path.join(ROOT, "gficf_b200", "csrc")
ASCENDING, DESCENDING, RANDOM = 0, 1, 2
SCHEDULES = [(DESCENDING, 0), (RANDOM, 0x5EED), (RANDOM, 20261021)]
_dp, _ip = C.POINTER(C.c_double), C.POINTER(C.c_int32)


@contextlib.contextmanager
def schedule(libs, mode, seed=0):
    """Run the block under `mode` / `seed`, then go back to the default ascending order."""
    for L in libs:
        L.emu_set_schedule(mode, C.c_ulonglong(seed))
    try:
        yield
    finally:
        for L in libs:
            L.emu_set_schedule(ASCENDING, C.c_ulonglong(0))


def bits(x):
    """A comparable form of a result: arrays by dtype, shape and bytes, floats by their bit pattern."""
    if isinstance(x, np.ndarray):
        return ("a", x.dtype.str, x.shape, x.tobytes())
    if isinstance(x, (float, np.floating)):
        return ("f", np.float64(x).tobytes())
    if isinstance(x, dict):
        return ("d", tuple((k, bits(v)) for k, v in sorted(x.items())))
    if isinstance(x, (tuple, list)):
        return ("t", tuple(bits(v) for v in x))
    return ("o", x)


def across_schedules(libs, run):
    """run() in ascending order, then under each permuted schedule: every result must be the ascending
    one bit for bit.  Returns the ascending result, for the oracle."""
    want = run()
    for mode, seed in SCHEDULES:
        with schedule(libs, mode, seed):
            got = run()
        assert bits(got) == bits(want), ("schedule", mode, seed)
    return want


# ---------------------------------------------------------------- harnesses
def _compile(so, source, extra=(), host_stats=False):
    cmd = ["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-DGFICF_CUDA_EMU", *extra, "-I" + EMU, "-I" + CSRC,
           "-I" + os.path.join(ROOT, "include"), "-shared", "-fPIC", "-Wall", "-Wno-unknown-pragmas", "-Werror", source]
    if host_stats:
        cmd.append(os.path.join(CSRC, "host_stats.cpp"))
    out = subprocess.run(cmd + ["-o", so], capture_output=True, text=True)
    assert out.returncode == 0, out.stderr


HARNESSES = ("jaccard_emu", "snn_emu", "network_emu", "wmu_emu", "wmu_markers_emu", "wmu_markers_sparse_emu")


@pytest.fixture(scope="module")
def libs(tmp_path_factory):
    """The six harnesses, plus the Jaccard one with GFICF_MAX_TRIES=1, built side by side.  That one runs a few
    small slabs only and is built at -O0, which takes a third of the time."""
    from tests.test_jaccard_slabs_emu import _build as build_jaccard
    from tests.test_network_emu import load_emu
    from tests.test_snn_emu import _ll, _bp
    from tests.test_wmu_markers_sparse_emu import load_sparse_emu

    d = tmp_path_factory.mktemp("emu_schedules")

    def plain(name):
        so = str(d / f"lib{name}.so")
        _compile(so, os.path.join(EMU, name + ".cpp"), host_stats=name.startswith("wmu"))
        return C.CDLL(so)

    with ThreadPoolExecutor(7) as ex:
        jac = ex.submit(build_jaccard, str(d / "libjaccard_emu.so"), [])
        jac1 = ex.submit(build_jaccard, str(d / "libjaccard_emu_1try.so"), ["-DGFICF_MAX_TRIES=1", "-O0"])
        rest = {name: ex.submit(plain, name) for name in HARNESSES[1:]}
        out = {"jaccard_emu": jac.result(), "jaccard_1try": jac1.result(), **{k: f.result() for k, f in rest.items()}}
    out["network_emu"] = load_emu(out["network_emu"]._name)
    out["wmu_markers_sparse_emu"] = load_sparse_emu(out["wmu_markers_sparse_emu"]._name)
    L = out["snn_emu"]
    L.emu_snn_lower.argtypes = [_ip, C.c_longlong, C.c_int, C.c_int, _bp, _ll, _ip, _dp, _ip, _ll, _ll, C.c_int, C.c_int]
    L.emu_snn_lower.restype = C.c_uint
    out["wmu_emu"].emu_wmu_test.argtypes = [_dp, _dp, C.c_longlong, C.c_longlong, C.c_longlong, _dp, C.c_int]
    out["wmu_emu"].emu_wmu_test.restype = None
    out["wmu_markers_emu"].emu_wmu_markers.argtypes = [_dp, C.c_longlong, C.c_longlong, _ip, C.c_int, _dp, C.c_int]
    out["wmu_markers_emu"].emu_wmu_markers.restype = None
    for lib in out.values():
        lib.emu_set_schedule.argtypes = [C.c_int, C.c_ulonglong]
        lib.emu_set_schedule.restype = None
    return out


def test_every_harness_exports_the_setter(libs):
    for name in HARNESSES:
        assert hasattr(libs[name], "emu_set_schedule"), name


# ---------------------------------------------------------------- Jaccard
def _jaccard(libs, idx, mode, lo, hi, grid=3, lib="jaccard_emu"):
    from tests.test_jaccard_slabs_emu import run_slab

    L = libs[lib]
    return across_schedules([L], lambda: run_slab(L, idx, mode, lo, hi, grid=grid, offset=lo % 3))


@pytest.mark.parametrize("k", [3, 7, 10, 30])
def test_jaccard_small_k_kernel(libs, oracle, k):
    """The k <= 32 kernel at KP 4, 8, 16 (pad pieces skipped) and 32: fused (OUT 0), mutual bit (OUT 2) and
    grouped tagged counts (OUT 3) on a slab long enough for whole rounds of 8-row groups at grid 2."""
    from tests.conftest import random_knn
    from tests.test_jaccard_slabs_emu import mutual_of, u_of

    rng = np.random.default_rng(40 + k)
    idx = random_knn(rng, 150, k)
    lo, hi = 1, 150
    par = oracle.parallel_rows(idx, lo, hi)
    u = u_of(par, k)
    out, _, _, flags = _jaccard(libs, idx, 0, lo, hi, grid=2)
    assert flags == 0 and np.array_equal(out, par)
    _, cnt, _, flags = _jaccard(libs, idx, 4, lo, hi, grid=3)
    assert flags == 0 and np.array_equal(cnt & 0x7F, u) and np.array_equal((cnt & 0x80) != 0, mutual_of(idx, lo, hi))
    _, cnt, _, flags = _jaccard(libs, idx, 5, lo, hi, grid=2)
    assert flags == 0 and np.array_equal(cnt, u | 0x80)


@pytest.mark.parametrize("k", [33, 64, 128])
def test_jaccard_wide_k_kernel(libs, oracle, k):
    """The k <= 128 kernel (CTA table, warp 0 builds it): counts + expand, fused, and the mutual bit."""
    from tests.conftest import random_knn
    from tests.test_jaccard_slabs_emu import u_of

    rng = np.random.default_rng(k)
    idx = random_knn(rng, k + 20, k)
    lo, hi = 3, 3 + (10 if k < 128 else 5)
    par = oracle.parallel_rows(idx, lo, hi)
    for mode in (1, 0, 4) if k <= 127 else (1, 0):
        out, cnt, _, flags = _jaccard(libs, idx, mode, lo, hi, grid=3)
        assert flags == 0, (mode, flags)
        if mode in (0, 1):
            assert np.array_equal(out, par), mode
        if mode != 0:
            assert np.array_equal(cnt & 0x7F, u_of(par, k)), mode


@pytest.mark.parametrize("k", [200, 1024])
def test_jaccard_large_k_kernel(libs, oracle, k):
    """The CTA-per-row kernel: its table is filled with atomicCAS, so the slot each id lands in depends on
    the order of the inserts; the counts must not."""
    from tests.conftest import random_knn
    from tests.test_jaccard_slabs_emu import u_of

    rng = np.random.default_rng(k)
    idx = random_knn(rng, k + 6, k)
    lo, hi = 2, 4
    par = oracle.parallel_rows(idx, lo, hi)
    out, cnt, _, flags = _jaccard(libs, idx, 1, lo, hi, grid=2)
    assert flags == 0 and np.array_equal(out, par) and np.array_equal(cnt, u_of(par, k))
    if k <= 255:
        out, _, _, flags = _jaccard(libs, idx, 0, lo, hi, grid=2)
        assert flags == 0 and np.array_equal(out, par)


@pytest.mark.parametrize("k,p,q", [(5, 0, 4), (30, 17, 3), (40, 1, 33), (200, 64, 199)])
def test_jaccard_repeated_id(libs, oracle, k, p, q):
    """A row that lists an id twice: several lanes store to one slot of the k <= 32 / k <= 128 tables (any
    store may survive), and two CAS inserts meet in the large-k table.  Flag 2 in every order; the exact
    kernel gives the oracle."""
    from tests.conftest import random_knn

    rng = np.random.default_rng(k + p)
    idx = random_knn(rng, k + 12, k)
    r = 6
    idx[r, q] = idx[r, p]
    _, _, _, flags = _jaccard(libs, idx, 1, r - 1, r + 2, grid=2)
    assert flags == 2
    if k <= 128:
        out, _, _, _ = _jaccard(libs, idx, 3, r - 1, r + 2, grid=2)
        assert np.array_equal(out, oracle.parallel_rows(idx, r - 1, r + 2))


@pytest.mark.parametrize("k", [12, 46])
def test_jaccard_forced_hash_failure(libs, oracle, k):
    """GFICF_MAX_TRIES=1: flag 4 exactly when the slab holds a row whose ids collide under the first
    multiplier, and the counts of every other row right and the same in every order.  The counts of a
    failed row are discarded (the exact path answers for the slab); they come from a table in which
    colliding lanes stored to one slot, and which store survived depends on the schedule -- so they may
    differ between schedules, and at these seeds they do, which shows the permuted orders reach the
    "whichever writer survives" stores of both kernels."""
    from tests.conftest import random_knn
    from tests.test_jaccard_slabs_emu import _collides_at_first_multiplier, _log_ts, run_slab, u_of

    L = libs["jaccard_1try"]
    rng = np.random.default_rng(900 + k)
    idx = random_knn(rng, 3000, k)
    coll = _collides_at_first_multiplier(idx, _log_ts(L, k))
    h = int(np.flatnonzero(coll[10:])[0]) + 10
    clean = int(np.flatnonzero(~coll)[0])
    failed_rows_differ = False
    for lo, hi in ((h - 4, h + 4), (clean, clean + 1)):
        ok = ~coll[lo:hi]
        u = u_of(oracle.parallel_rows(idx, lo, hi), k)
        _, want, _, flags = run_slab(L, idx, 1, lo, hi, grid=2)
        assert flags == (4 if coll[lo:hi].any() else 0), (lo, hi, flags)
        assert np.array_equal(want[ok], u[ok])
        for mode, seed in SCHEDULES:
            with schedule([L], mode, seed):
                _, cnt, _, got_flags = run_slab(L, idx, 1, lo, hi, grid=2)
            assert got_flags == flags and np.array_equal(cnt[ok], want[ok]), (mode, seed, lo, hi)
            failed_rows_differ |= not np.array_equal(cnt[~ok], want[~ok])
    assert failed_rows_differ


@pytest.mark.parametrize("k", [7, 40])
def test_jaccard_exact_kernel_and_compaction(libs, oracle, k):
    """Repeated ids: the exact kernel (multiset) + expand, and (set semantics) + the compaction, whose
    chunk offsets come from a one-CTA scan."""
    from tests.conftest import random_knn
    from tests.test_jaccard_slabs_emu import serial_slab

    rng = np.random.default_rng(k)
    idx = random_knn(rng, k + 30, k, distinct=False)
    n = idx.shape[0]
    lo, hi = 1, n if k <= 32 else 13
    out, _, _, _ = _jaccard(libs, idx, 3, lo, hi, grid=3)
    assert np.array_equal(out, oracle.parallel_rows(idx, lo, hi))
    out, _, nw, _ = _jaccard(libs, idx, 2, lo, hi, grid=3)
    want, m = serial_slab(oracle.serial(idx), lo, hi, k)
    assert nw == m and np.array_equal(out, want)


@pytest.mark.parametrize("k,mode", [(30, 7), (30, 6), (64, 6)])
def test_jaccard_streaming_expand(libs, oracle, k, mode):
    """Tagged counts (row stores or 8-row groups), then expand_stream_kernel over three segments on a 2 x 3
    grid (6 emulated SMs shared by the 3 segments): the 2-D CTA order is permuted too."""
    from tests.conftest import random_knn
    from tests.test_jaccard_slabs_emu import u_of

    rng = np.random.default_rng(k + mode)
    idx = random_knn(rng, k + 40, k)
    lo, hi = 7, k + 40
    par = oracle.parallel_rows(idx, lo, hi)
    out, cnt, _, flags = _jaccard(libs, idx, mode, lo, hi, grid=6)
    assert flags == 0 and np.array_equal(cnt, u_of(par, k) | 0x80) and np.array_equal(out, par)


# ---------------------------------------------------------------- SNN graph build
def _snn(libs, oracle, idx):
    from tests.test_snn_emu import check, emu_lower

    L = libs["snn_emu"]
    across_schedules([L], lambda: emu_lower(L, idx.numpy()))
    return check(L, oracle, idx)


def test_snn_uniform_graph_with_target_only_vertices(libs, oracle):
    """Cells that only appear as targets get their vertex id from the atomicMin of snn_targets_kernel<0>;
    column entries are placed by the atomicAdd cursors of snn_edges_kernel<true>, then sorted."""
    from gficf_b200 import synth

    flags, _ = _snn(libs, oracle, synth.knn_index(500, 5, family="uniform", scramble=True))
    assert flags & 16


def test_snn_hub_columns(libs, oracle):
    """Columns past 32 and 512 entries: the warp rank sort and the shared-memory bitonic sort."""
    import torch

    from gficf_b200 import synth

    n, k = 1000, 8
    rng = np.random.default_rng(4)
    idx = synth.knn_index(n, k, family="planted", scramble=False).numpy().copy()
    for hub, fans in ((0, 700), (1, 100)):
        for r in rng.choice(np.arange(10, n), fans, replace=False):
            if hub not in idx[r]:
                idx[r, rng.integers(0, k)] = hub
    idx[:, 0] = np.where((idx[:, 1:] == 5).any(axis=1) | (np.arange(n) == 5), idx[:, 0], 5)
    assert all(len(set(r.tolist())) == k for r in idx)
    _, colptr = _snn(libs, oracle, torch.from_numpy(idx))
    deg = np.diff(colptr)
    assert deg.max() > 512 and ((deg > 32) & (deg <= 512)).any()


# ---------------------------------------------------------------- network
@pytest.mark.parametrize("nv,m,nc,seed", [(60, 300, 7, 2), (250, 2000, 25, 4)])
def test_network_build_quality_reduce(libs, nv, m, nc, seed):
    from oracle.binding import NetworkOracle
    from tests.network_cases import assert_same_network, random_lower
    from tests.test_network_emu import emu_build, emu_quality, emu_reduce

    L = libs["network_emu"]
    rng = np.random.default_rng(seed)
    n1, n2, w = random_lower(rng, nv, m)
    nv = int(max(n1.max(), n2.max())) + 1
    O = NetworkOracle()
    want = O.network(n1, n2, w)
    got, flags = across_schedules([L], lambda: emu_build(L, n1, n2, w, nv))
    assert flags == 0
    assert_same_network(got, want)
    cl = rng.integers(0, nc, nv).astype(np.int32)
    cl[rng.permutation(nv)[:nc]] = np.arange(nc)
    res = 0.8 / (2 * want["total_w"])
    q, cw, flags = across_schedules([L], lambda: emu_quality(L, got, cl, nc, res))
    q_want, cw_want = O.quality(want, cl, res)
    assert flags == 0 and q == q_want and np.array_equal(cw, cw_want)
    red, flags = across_schedules([L], lambda: emu_reduce(L, got, cl, nc))
    assert flags == 0
    assert_same_network(red, O.reduce(want, cl))


def test_network_sequential_sum_past_one_window(libs):
    """The exact replay of std::accumulate over a few windows (kSeqBlock = 4096 elements each): block sums
    of several CTAs, then the walk to the first binade crossing."""
    from tests.network_cases import seq_sum
    from tests.sum_order_cases import SEQ_BLOCK, jaccard_weights, window_schedule
    from tests.test_network_emu import _emu_seq

    L = libs["network_emu"]
    rng = np.random.default_rng(12)
    x = np.concatenate([np.zeros(5000), jaccard_weights(rng, 5 * SEQ_BLOCK + 17)])
    assert max(b for _, b, _ in window_schedule(x)) >= 2
    got, flags = across_schedules([L], lambda: _emu_seq(L, x, 0.0, ctas=3))
    assert flags == 0 and got == seq_sum(x)


# ---------------------------------------------------------------- Mann-Whitney
def test_wmu_single_split(libs):
    """Negative values, +-0, ties and a dense gene: wmu_load compacts the non-zero values through an
    atomicAdd per warp, so their order before the sort follows the schedule."""
    from oracle.binding import WmuOracle
    from tests.test_wmu_emu import emu_wmu
    from tests.test_wmu_oracle import sc_matrix

    L = libs["wmu_emu"]
    rng = np.random.default_rng(8)
    n1, n2 = 300, 700
    m = sc_matrix(rng, 8, n1 + n2, integer=True)
    m[1, :] = 0.0
    m[2, :] = -m[2, :]
    m[3, ::2] = -0.0
    m[4, :] = rng.normal(size=n1 + n2)
    m[5, :] = np.where(rng.random(n1 + n2) < 0.5, -2.0, m[5, :])
    x, y = m[:, :n1], m[:, n1:]
    got = across_schedules([L], lambda: emu_wmu(L, x, y, grid=3))
    assert np.array_equal(got, WmuOracle().wmu(np.asfortranarray(x), np.asfortranarray(y), nthreads=2), equal_nan=True)


@pytest.mark.parametrize("k", [2, 30])
def test_wmu_markers_dense_and_sparse(libs, k):
    """Every cluster's block from the dense markers kernels and from the sparse pipeline (radix-sort
    transpose with atomic histograms, then the rank and means kernels), each against the oracle."""
    from tests.test_wmu_markers_emu import check_blocks, emu_markers
    from tests.test_wmu_markers_sparse_emu import edge_rows, emu_sparse, to_csc
    from tests.test_wmu_oracle import sc_matrix

    dense, sparse = libs["wmu_markers_emu"], libs["wmu_markers_sparse_emu"]
    rng = np.random.default_rng(k)
    cells = 600
    cl = rng.integers(0, k, cells).astype(np.int32)
    cl[:k] = np.arange(k)
    rng.shuffle(cl)
    colptr, row, x, m = to_csc(edge_rows(rng, sc_matrix(rng, 14, cells, integer=k > 2), cl), rng, 0.1)
    got = across_schedules([dense], lambda: emu_markers(dense, m, cl, k, 3))
    check_blocks(got, m, cl, k)
    gs, flags = across_schedules([sparse], lambda: emu_sparse(sparse, colptr, row, x, m.shape[0], cl, k, grid=3, ctas=3))
    assert flags == 0 and np.array_equal(gs.view(np.int64), got.view(np.int64))


def test_wmu_ordered_tie_term(libs):
    """N = 208 064: the tie term is the reference's sequential double sum, its 4 032 non-trivial groups
    compacted in sorted order through a block scan (one gene)."""
    from oracle.binding import WmuOracle
    from tests.sum_order_cases import order_sensitive_gene
    from tests.test_wmu_emu import emu_wmu

    L = libs["wmu_emu"]
    n, n1 = 208_064, 30_000
    m = np.asfortranarray(order_sensitive_gene(np.random.default_rng(5), n, 200_000)[None, :])
    got = across_schedules([L], lambda: emu_wmu(L, m[:, :n1], m[:, n1:], grid=1))
    assert np.array_equal(got, WmuOracle().wmu(np.asfortranarray(m[:, :n1]), np.asfortranarray(m[:, n1:])), equal_nan=True)


# ---------------------------------------------------------------- the schedules themselves
TOYS = r"""
#include "cuda_emu.h"

extern "C" {
// the order in which the threads of CTA (0, 0) take a ticket before and after a __syncthreads, and the
// order in which the CTAs of a gx x gy grid run
void toy_order(unsigned block, unsigned gx, unsigned gy, unsigned* first, unsigned* second, unsigned* cta) {
  unsigned nt = 0, nc = 0;
  unsigned *pt = &nt, *pc = &nc;
  cuda_emu::launch(gx, block, [=] {
    const bool origin = blockIdx.x == 0 && blockIdx.y == 0;
    if (threadIdx.x == 0) cta[blockIdx.y * gridDim.x + blockIdx.x] = atomicAdd(pc, 1u);
    if (origin) first[threadIdx.x] = atomicAdd(pt, 1u);
    __syncthreads();
    if (origin) second[threadIdx.x] = atomicAdd(pt, 1u) - blockDim.x;
  }, 0, gy);
}

// what each CTA finds in its dynamic shared memory before it writes there
void toy_smem_poison(unsigned grid, unsigned* seen) {
  cuda_emu::launch(grid, 64, [=] {
    unsigned* s = reinterpret_cast<unsigned*>(cuda_emu::dynamic_smem());
    seen[blockIdx.x * 64 + threadIdx.x] = s[threadIdx.x];
    s[threadIdx.x] = blockIdx.x;
  }, 64 * sizeof(unsigned));
}

// must abort: half of every warp waits at __syncthreads, the other half in a warp collective
void toy_divergent_syncthreads() {
  cuda_emu::launch(1, 64, [] {
    if ((threadIdx.x & 31) < 16) __syncthreads();
    else __syncwarp();
  });
}
// must abort: a collective with a partial member mask
void toy_partial_mask() {
  cuda_emu::launch(1, 64, [] { (void)__shfl_sync(0x0000FFFFu, (int)threadIdx.x, 0); });
}
// must abort: lane 3 of every warp has exited when the others reach a collective
void toy_collective_after_exit() {
  cuda_emu::launch(1, 64, [] {
    if ((threadIdx.x & 31) == 3) return;
    (void)__ballot_sync(0xFFFFFFFFu, 1);
  });
}
}
"""


@pytest.fixture(scope="module")
def toys(tmp_path_factory):
    d = tmp_path_factory.mktemp("emu_toys")
    (d / "toys.cpp").write_text(TOYS)
    so = str(d / "libtoys.so")
    _compile(so, str(d / "toys.cpp"))
    L = C.CDLL(so)
    L.emu_set_schedule.argtypes = [C.c_int, C.c_ulonglong]
    u32p = C.POINTER(C.c_uint32)
    L.toy_order.argtypes = [C.c_uint, C.c_uint, C.c_uint, u32p, u32p, u32p]
    L.toy_smem_poison.argtypes = [C.c_uint, u32p]
    return L


def _up(a):
    return a.ctypes.data_as(C.POINTER(C.c_uint32))


def _launch_order(L, block=96, gx=5, gy=3):
    first, second, cta = np.zeros(block, np.uint32), np.zeros(block, np.uint32), np.zeros(gx * gy, np.uint32)
    L.toy_order(block, gx, gy, _up(first), _up(second), _up(cta))
    return first, second, cta


def _order(L, mode, seed):
    with schedule([L], mode, seed):
        return _launch_order(L)


def test_schedule_orders(toys):
    """Ascending and descending are what they say (after a barrier, the last thread to arrive runs on
    first); a random schedule is a permutation redrawn in every round and every launch, the same for the
    same seed, and permutes the CTAs over both x and y of a 2-D grid."""
    first, second, cta = _order(toys, ASCENDING, 0)
    assert np.array_equal(first, np.arange(96)) and np.array_equal(cta, np.arange(15))
    assert second[95] == 0 and np.array_equal(second[:95], np.arange(1, 96))
    first, second, cta = _order(toys, DESCENDING, 0)
    assert np.array_equal(first, np.arange(96)[::-1]) and np.array_equal(cta, np.arange(15)[::-1])
    assert second[0] == 0 and np.array_equal(second[1:], np.arange(95, 0, -1))
    a = _order(toys, RANDOM, 7)
    for x, n in zip(a, (96, 96, 15)):
        assert np.array_equal(np.sort(x), np.arange(n))
    assert all(np.array_equal(x, y) for x, y in zip(a, _order(toys, RANDOM, 7)))  # same seed, same run
    b = _order(toys, RANDOM, 8)
    assert not np.array_equal(a[0], b[0]) and not np.array_equal(a[2], b[2])
    round1, round2 = np.argsort(a[0]), np.argsort(a[1])  # threads in the order they ran
    assert not np.array_equal(round1, np.arange(96)) and not np.array_equal(round1, np.arange(96)[::-1])
    assert not np.array_equal(round2[1:], round1[round1 != round2[0]])  # a new permutation after the barrier
    cells = a[2].reshape(3, 5)  # CTA (x, y) at [y, x]: neither whole rows nor whole columns run together
    assert not all(np.ptp(r) == 4 for r in cells) and not all(np.ptp(c) == 2 for c in cells.T)
    with schedule([toys], RANDOM, 7):  # and a new one for the next launch
        again = [_launch_order(toys) for _ in range(2)]
    assert np.array_equal(again[0][0], a[0]) and not np.array_equal(again[1][0], a[0])


@pytest.mark.parametrize("mode,seed", [(ASCENDING, 0)] + SCHEDULES)
def test_dynamic_shared_memory_is_poisoned_for_every_cta(toys, mode, seed):
    seen = np.zeros(4 * 64, np.uint32)
    with schedule([toys], mode, seed):
        toys.toy_smem_poison(4, _up(seen))
    assert (seen == 0xA5A5A5A5).all()


@pytest.mark.parametrize("toy,message", [("toy_divergent_syncthreads", "deadlock"),
                                         ("toy_partial_mask", "partial member mask"),
                                         ("toy_collective_after_exit", "lanes of the warp have exited")])
def test_aborts_survive_every_schedule(toys, toy, message):
    """Each emulated launch that the hardware would hang on or leave undefined still aborts with its report,
    whichever fibre arrives last.  Run in child processes (the emulation aborts)."""
    for mode, seed in [(ASCENDING, 0)] + SCHEDULES:
        code = (f"import ctypes; L = ctypes.CDLL({toys._name!r}); "
                f"L.emu_set_schedule(ctypes.c_int({mode}), ctypes.c_ulonglong({seed})); L.{toy}()")
        out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=120)
        assert out.returncode != 0 and "cuda_emu: " in out.stderr and message in out.stderr, (mode, seed, out.stderr)


# ---------------------------------------------------------------- a missing barrier
def test_a_removed_barrier_fails_only_under_permuted_schedules(libs, tmp_path):
    """wmu_rank_kernel, px scan: thread kWmuThreads - 1 publishes the running carry (sm.carry) after the
    scan's second barrier, and after the last tile thread 0 reads it into px[M].  Without the __syncthreads
    between the two, thread 0 may read the carry of the tile before.  In ascending order this can never
    show: the highest thread is the last to reach the barrier before, and the last arriver runs on at
    once, so its store always lands first.  In descending order thread 0 is that last arriver and reads
    the stale carry; a random order has some other thread arrive last.  Every group-1 count of the last
    tie group comes from px[M], so the rank sums go wrong on every gene."""
    from oracle.binding import WmuOracle
    from tests.test_wmu_emu import emu_wmu
    from tests.test_wmu_oracle import sc_matrix

    csrc = tmp_path / "csrc"
    shutil.copytree(CSRC, csrc)
    src = (csrc / "wmu_kernels.cuh").read_text()
    mutant, n = re.subn(r"(if \(tid == kWmuThreads - 1\) sm\.carry = before \+ inc;\n)\s*__syncthreads\(\);\n(\s*\}\n"
                        r"\s*if \(tid == 0\) px\[M\] = sm\.carry;)", r"\1\2", src)
    assert n == 1, "the barrier is gone from wmu_kernels.cuh: pick another"
    (csrc / "wmu_kernels.cuh").write_text(mutant)
    so = str(tmp_path / "libwmu_emu_mutant.so")
    cmd = ["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-DGFICF_CUDA_EMU", "-I" + EMU, "-I" + str(csrc),
           "-I" + os.path.join(ROOT, "include"), "-shared", "-fPIC", "-Wall", "-Wno-unknown-pragmas", "-Werror", os.path.join(EMU, "wmu_emu.cpp"),
           str(csrc / "host_stats.cpp"), "-o", so]
    out = subprocess.run(cmd, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    L = C.CDLL(so)
    L.emu_wmu_test.argtypes = [_dp, _dp, C.c_longlong, C.c_longlong, C.c_longlong, _dp, C.c_int]
    L.emu_wmu_test.restype = None
    L.emu_set_schedule.argtypes = [C.c_int, C.c_ulonglong]
    rng = np.random.default_rng(12)
    n1, n2 = 300, 900
    m = sc_matrix(rng, 4, n1 + n2)
    x, y = np.asfortranarray(m[:, :n1]), np.asfortranarray(m[:, n1:])
    want = WmuOracle().wmu(x, y, nthreads=2)
    assert np.array_equal(emu_wmu(L, x, y), want, equal_nan=True)  # the blind spot
    for mode, seed in SCHEDULES:
        with schedule([L], mode, seed):
            assert not np.array_equal(emu_wmu(L, x, y), want, equal_nan=True), (mode, seed)
