"""CPU: the Jaccard kernels (gficf_b200/csrc/jaccard_kernels.cuh) on ROW SLABS [row_lo, row_hi) of the
matrix, run on the CUDA emulation (tests/cuda_emu/jaccard_emu.cpp: emu_jaccard_slab, emu_layout_slab).

Every kernel writes edge (i, j) at (i - row_lo) * k + j; with row_lo = 0 that offset vanishes, so these
tests start slabs at rows 1, 7, 8, 9 and 17 and put guard zones filled with a sentinel around every
output and count buffer.  Also covered: every k from 1 to 128 (and the large-k kernel), a repeated id
at every pair of positions of a row (each kernel detects repeats differently), and the hash-failure
flag, forced by a build with GFICF_MAX_TRIES=1 whose colliding rows are predicted by replaying the
first multiplier here."""
import ctypes as C
import os
import subprocess
from concurrent.futures import ThreadPoolExecutor

import numpy as np
import pytest

import gficf_b200
from tests.conftest import random_knn

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
_dp, _ip, _ll, _vp = C.POINTER(C.c_double), C.POINTER(C.c_int), C.POINTER(C.c_longlong), C.c_void_p
FLAG_BAD, FLAG_DUP, FLAG_HASH = 1, 2, 4
SENT_F64, SENT_U8, SENT_I32 = -7.0, 0xEE, 0x7A7A7A7A
K_MULT0 = 0x9E3779B1  # first multiplier of the k <= 128 kernels' collision-free hash
LOS = (0, 1, 7, 8, 9, 17)


def _build(so, extra):
    cmd = ["g++", "-O1", "-std=c++17", "-ffp-contract=off", "-DGFICF_CUDA_EMU", *extra,
           "-I" + os.path.join(ROOT, "tests", "cuda_emu"), "-I" + os.path.join(ROOT, "gficf_b200", "csrc"), "-shared",
           "-fPIC", "-Wall", "-Wno-unknown-pragmas", "-Werror", os.path.join(ROOT, "tests", "cuda_emu", "jaccard_emu.cpp"),
           "-o", so]
    out = subprocess.run(cmd, capture_output=True, text=True)
    assert out.returncode == 0, out.stderr
    L = C.CDLL(so)
    L.emu_jaccard_slab.argtypes = [_dp, C.c_longlong, C.c_int, C.c_int, C.c_longlong, C.c_longlong, _vp, _vp, _vp, _vp,
                                   _ll, C.c_int]
    L.emu_jaccard_slab.restype = C.c_uint
    L.emu_layout_slab.argtypes = [_vp, C.c_int, C.c_longlong, C.c_int, C.c_longlong, C.c_longlong, _ip, C.c_int]
    L.emu_layout_slab.restype = C.c_uint
    L.emu_jaccard_variant.argtypes = [C.c_int]
    L.emu_jaccard_variant.restype = C.c_int
    return L


@pytest.fixture(scope="module")
def libs(tmp_path_factory):
    """The harness as shipped, and the same harness with GFICF_MAX_TRIES=1 (one multiplier: any row whose
    ids collide under it raises the hash-failure flag).  Built side by side."""
    d = tmp_path_factory.mktemp("emu_slabs")
    with ThreadPoolExecutor(2) as ex:
        a = ex.submit(_build, str(d / "libjaccard_emu.so"), [])
        b = ex.submit(_build, str(d / "libjaccard_emu_1try.so"), ["-DGFICF_MAX_TRIES=1"])
        return a.result(), b.result()


@pytest.fixture(scope="module")
def emu(libs):
    return libs[0]


@pytest.fixture(scope="module")
def emu1(libs):
    return libs[1]


def run_slab(L, idx, mode, lo, hi, grid=3, offset=0):
    """emu_jaccard_slab with guard zones around every buffer.  The guards are n*k + 64 elements wide, so
    that a store at an absolute instead of a slab-relative edge still lands inside one (and is seen
    there).  Returns ((hi-lo)*k x 3 output, (hi-lo) x k counts, n_written, flags)."""
    idx = np.asfortranarray(idx, dtype=np.float64)
    n, k = idx.shape
    e = (hi - lo) * k
    g = n * k + 64
    cb = 2 if k > 255 else 1
    out = np.full((3, g + e + g), SENT_F64)
    counts = np.full((2 * g + e) * cb + offset, SENT_U8, np.uint8)
    c0 = g * cb + offset
    nw = np.full(1, -1, np.int64)
    flags = L.emu_jaccard_slab(idx.ctypes.data_as(_dp), n, k, mode, lo, hi, *(out[c].ctypes.data + 8 * g for c in range(3)),
                               counts.ctypes.data + c0, nw.ctypes.data_as(_ll), grid)
    assert (out[:, :g] == SENT_F64).all() and (out[:, g + e:] == SENT_F64).all(), ("output guard", mode, lo, hi)
    assert (counts[:c0] == SENT_U8).all() and (counts[c0 + e * cb:] == SENT_U8).all(), ("count guard", mode, lo, hi)
    cnt = counts[c0:c0 + e * cb].copy()
    if cb == 2:
        cnt = cnt.view(np.uint16)
    return np.asfortranarray(out[:, g:g + e].T), cnt.reshape(hi - lo, k), int(nw[0]), flags


def u_of(par, k):
    """Intersection counts from the reference's weights: w = u / (2k - u)."""
    return (par[:, 2] * (2 * k) / (1 + par[:, 2])).round().astype(np.int64).reshape(-1, k)


def mutual_of(idx, lo, hi):
    a = (np.asarray(idx) - 1).astype(np.int64)
    sets = [set(r.tolist()) for r in a]
    return np.array([[i in sets[t] for t in a[i]] for i in range(lo, hi)]).reshape(hi - lo, a.shape[1])


def serial_slab(ser, lo, hi, k):
    """The compacted export of rows [lo, hi) alone: the oracle's serial rows of that slab, zero tail."""
    rows = ser[(ser[:, 0] >= lo + 1) & (ser[:, 0] <= hi)]
    want = np.zeros(((hi - lo) * k, 3), order="F")
    want[:rows.shape[0]] = rows
    return want, rows.shape[0]


# ---------------------------------------------------------------- inputs
def high_overlap(rng, k, n_min):
    """n = k + 3 .. k + 40: every row lists most cells, so u comes near k."""
    return random_knn(rng, max(k + int(rng.integers(3, 41)), n_min), k)


def identical_and_disjoint(rng, k, n_min):
    """Rows of block A list A itself (u = k on every edge) next to blocks C and D that list each
    other (u = 0), ids shuffled inside each row; padded with random rows up to n_min."""
    n = max(3 * k + 2, n_min)
    a = np.zeros((n, k), np.int64)
    blocks = (np.arange(k), np.arange(k, 2 * k), np.arange(2 * k, 3 * k))
    for r in range(n):
        if r < k:
            ids = blocks[0]
        elif r < 2 * k:
            ids = blocks[2]
        elif r < 3 * k:
            ids = blocks[1]
        else:
            ids = rng.choice(n, k, replace=False)
        a[r] = rng.permutation(ids)
    return np.asfortranarray(a.astype(np.float64) + 1.0)


def ends_in_every_row(rng, k, n_min):
    """Ids 0 and n - 1 (the first and the last row) in every row."""
    n = max(k + 10, n_min)
    a = np.zeros((n, k), np.int64)
    for r in range(n):
        ids = np.concatenate([rng.choice(np.arange(1, n - 1), k - 2, replace=False), [0, n - 1]])[-k:]
        a[r] = rng.permutation(ids)
    return np.asfortranarray(a.astype(np.float64) + 1.0)


def self_ids(rng, k, n_min):
    """Every row lists itself (duplicate cells keep themselves in neigh[, -1])."""
    n = max(k + 20, n_min)
    a = (random_knn(rng, n, k, with_self=True) - 1).astype(np.int64)
    for r in range(n):
        if r not in a[r]:
            a[r, rng.integers(0, k)] = r
    return np.asfortranarray(a.astype(np.float64) + 1.0)


def low_overlap(rng, k, n_min):
    return random_knn(rng, max(3 * k + 30, n_min), k)


FAMILIES = (high_overlap, low_overlap, identical_and_disjoint, ends_in_every_row, self_ids)


def slab_of(rng, n, which, max_rows=None):
    """Slab `which`: starts at LOS[which % 6] and ends at n (odd `which`) or short of it; at most max_rows
    rows (a slab that would be longer and end at n starts later instead)."""
    lo = LOS[which % len(LOS)]
    cap = max_rows or n
    if which % 2:
        return max(lo, n - cap), n
    span = n - lo
    return lo, lo + min(cap, max(1, span - int(rng.integers(1, max(2, span // 2)))))


# ---------------------------------------------------------------- every k, on slabs
@pytest.mark.parametrize("k", range(1, 129))
def test_every_k_on_slabs(emu, oracle, k):
    """Counts + expand (mode 1) at every k <= 128, the mutual bit (mode 4) for k <= 127, the fused kernel
    (mode 0) for k <= 32 and every third k above; input family, slab start, slab end and the emulated SM
    count vary with k (one SM, a few, and more SMs than the slab gives the persistent kernels work for)."""
    rng = np.random.default_rng(1000 + k)
    fam = FAMILIES[k % len(FAMILIES)]
    idx = fam(rng, k, 24)
    n = idx.shape[0]
    lo, hi = slab_of(rng, n, k, None if k <= 32 else 24 if k <= 64 else 12)  # gathers cost k^2 per row
    grid = (1, 2, 3, 64)[k % 4]
    par = oracle.parallel_rows(idx, lo, hi)
    u = u_of(par, k)
    modes = [1] + ([4] if k <= 127 else []) + ([0] if k <= 32 or k % 3 == 0 else [])
    for mode in modes:
        out, cnt, _, flags = run_slab(emu, idx, mode, lo, hi, grid=grid)
        assert flags == 0, (mode, flags)
        if mode in (0, 1):
            assert np.array_equal(out, par), (mode, lo, hi, grid)
        if mode == 1:
            assert np.array_equal(cnt, u)
        if mode == 4:
            assert np.array_equal(cnt & 0x7F, u) and np.array_equal((cnt & 0x80) != 0, mutual_of(idx, lo, hi))


@pytest.mark.parametrize("k", [129, 200, 255, 256, 257, 511, 1024])
def test_large_k_on_slabs(emu, oracle, k):
    """The CTA-per-row kernel (uint16 counts above 255), fused and counts + expand, on short slabs."""
    rng = np.random.default_rng(k)
    idx = high_overlap(rng, k, 0) if k % 2 else low_overlap(rng, k, 0)
    n = idx.shape[0]
    for lo, hi, grid in ((1, 4, 2), (9, 11, 1), (n - 3, n, 3)):
        par = oracle.parallel_rows(idx, lo, hi)
        for mode in (0, 1):
            out, cnt, _, flags = run_slab(emu, idx, mode, lo, hi, grid=grid)
            assert flags == 0 and np.array_equal(out, par), (mode, lo, hi)
            if mode == 1:
                assert np.array_equal(cnt, u_of(par, k))


@pytest.mark.parametrize("k", [1, 3, 8, 17, 30, 33, 64, 100])
def test_exact_kernel_and_compaction_on_slabs(emu, oracle, k):
    """The exact kernel (multiset, mode 3) + expand and (set semantics, mode 2) + compaction on slabs,
    on input with repeated ids and on clean input."""
    rng = np.random.default_rng(50 + k)
    for idx in (random_knn(rng, k + 30, k, distinct=False), self_ids(rng, k, 30)):
        n = idx.shape[0]
        ser = oracle.serial(idx)
        for which, grid in ((1, 1), (2, 3), (5, 2), (4, 64)):
            lo, hi = slab_of(rng, n, which, 40 if k <= 32 else 12)
            out, _, _, _ = run_slab(emu, idx, 3, lo, hi, grid=grid)
            assert np.array_equal(out, oracle.parallel_rows(idx, lo, hi)), (lo, hi)
            out, _, nw, _ = run_slab(emu, idx, 2, lo, hi, grid=grid)
            want, m = serial_slab(ser, lo, hi, k)
            assert nw == m and np.array_equal(out, want), (lo, hi)


@pytest.mark.parametrize("k", [1, 2, 3, 4, 5, 7, 8, 9, 15, 16, 17, 24, 25, 29, 30, 31, 32])
def test_grouped_counts_on_slabs(emu, oracle, k):
    """Tagged counts in groups of 8 rows (mode 5): slabs longer and shorter than 8 rows x warps (grouped
    part present / absent), starting at odd rows, with the count pointer 0..15 bytes past a 16-byte
    boundary (16-byte, 8-byte and bytewise group stores)."""
    rng = np.random.default_rng(300 + k)
    idx = random_knn(rng, 190, k) if k % 2 else high_overlap(rng, k, 190)
    n = idx.shape[0]
    case = 0
    for grid in (1, 2):
        rows8 = 8 * 7 * grid  # 8 rows per group x warps of the grid
        for lo in LOS:
            for span in (rows8 + 8 * int(rng.integers(0, 3)) + int(rng.integers(0, 8)), rows8 - 1 - int(rng.integers(0, 9))):
                hi = min(n, lo + span)
                u = u_of(oracle.parallel_rows(idx, lo, hi), k)
                offset = case % 16
                case += 1
                _, cnt, _, flags = run_slab(emu, idx, 5, lo, hi, grid=grid, offset=offset)
                assert flags == 0 and np.array_equal(cnt, u | 0x80), (grid, lo, hi, offset)


@pytest.mark.parametrize("k,mode", [(5, 6), (5, 7), (30, 6), (30, 7), (31, 7), (64, 6), (127, 6)])
def test_streaming_gather_on_slabs(emu, oracle, k, mode):
    """Tagged counts of a slab, then the streaming expand over three segments of it (absolute edges)."""
    rng = np.random.default_rng(k + mode)
    idx = random_knn(rng, k + 60, k)
    n = idx.shape[0]
    for lo, hi in ((7, n), (9, n - 5), (17, n - 2)):
        par = oracle.parallel_rows(idx, lo, hi)
        out, cnt, _, flags = run_slab(emu, idx, mode, lo, hi, grid=6, offset=lo % 2)  # 2 CTAs per segment
        assert flags == 0 and np.array_equal(cnt, u_of(par, k) | 0x80) and np.array_equal(out, par), (lo, hi)


# ---------------------------------------------------------------- layout pre-pass on slabs
@pytest.mark.parametrize("k", [1, 4, 5, 16, 30, 33, 100, 128, 300])
def test_layout_of_a_slab_shaped_source(emu, k):
    """layout_colmajor_kernel with ld_rows = hi - lo and ld_row0 = lo (f64 and int32), and pad_i32_kernel,
    convert rows [lo, hi) only; a bad id (NaN, NA_integer_, out of range) inside the slab raises flag 1,
    one outside it does not."""
    rng = np.random.default_rng(k)
    n = k + 150
    a = (random_knn(rng, n, k) - 1).astype(np.int32)  # 0-based
    kp = int(gficf_b200.lib().gficf_cuda_row_stride(k))
    for lo, hi, grid in ((0, n, 3), (1, n, 1), (7, 75, 2), (9, 10, 1), (17, n - 1, 8), (8, n, 64)):
        want = np.full((n, kp), SENT_I32, np.int32)
        want[lo:hi] = -2
        want[lo:hi, :k] = a[lo:hi]
        slab_f64 = np.asfortranarray(a[lo:hi].astype(np.float64) + 1.0)
        slab_i32 = np.asfortranarray(a[lo:hi] + 1)
        dense = np.ascontiguousarray(a)
        for elem, src in ((8, slab_f64), (4, slab_i32), (0, dense)):
            dst = np.full((n, kp), SENT_I32, np.int32)
            flags = emu.emu_layout_slab(src.ctypes.data, elem, n, k, lo, hi, dst.ctypes.data_as(_ip), grid)
            assert flags == 0 and np.array_equal(dst, want), (elem, lo, hi)
        r = int(rng.integers(lo, hi))
        for elem, src, bad in ((8, slab_f64, np.nan), (8, slab_f64, n + 1.0), (4, slab_i32, np.iinfo(np.int32).min),
                               (0, dense, n)):
            s = src.copy(order="A")
            s[r - (lo if elem else 0), k - 1] = bad
            dst = np.full((n, kp), SENT_I32, np.int32)
            assert emu.emu_layout_slab(s.ctypes.data, elem, n, k, lo, hi, dst.ctypes.data_as(_ip), grid) & FLAG_BAD
        if lo > 0:  # pad_i32_kernel reads the absolute rows of its source: a bad id before the slab is not its business
            s = dense.copy()
            s[lo - 1, 0] = -5
            dst = np.full((n, kp), SENT_I32, np.int32)
            assert emu.emu_layout_slab(s.ctypes.data, 0, n, k, lo, hi, dst.ctypes.data_as(_ip), grid) == 0


# ---------------------------------------------------------------- a repeated id at every position
def _dup_pairs(k):
    if k <= 33:
        return [(p, q) for p in range(k) for q in range(p + 1, k)]
    if k <= 128:
        # lane l of the k <= 128 kernel's warp 0 owns positions l, l+32, l+64, l+96 (c = 0..3): pairs in one
        # lane at different c, between lanes at c >= 1, across warps' quarters of the edges, first / last,
        # and at the last positions before the pads
        q4 = k // 4
        cand = [(0, 1), (0, k - 1), (k - 2, k - 1), (31, 32), (0, 32), (1, 33), (32, 64), (33, 97), (64, 96), (40, 100),
                (63, 127), (96, 127), (33, 34), (65, 66), (98, 99), (5, 69), (17, 113), (30, 94), (63, 64), (95, 96),
                (1, 2), (q4 - 1, q4), (q4, 2 * q4), (0, 2 * q4), (2 * q4 + 1, 3 * q4 + 1), (3, k - 2), (k - 33, k - 1),
                (k - 3, k - 2), (32, k - 1)]
    else:
        cand = [(0, 1), (0, k - 1), (k - 2, k - 1), (127, 128), (64, 200), (5, 133)]
    return sorted({(p, q) for p, q in cand if 0 <= p < q < k})


@pytest.mark.parametrize("k", [2, 3, 4, 5, 8, 9, 16, 17, 25, 31, 32, 33, 45, 46, 64, 65, 100, 127, 128, 129, 300])
def test_repeated_id_at_every_position(emu, oracle, k):
    """One matrix per position pair (p, q): exactly one row r gets id[r, q] := id[r, p].  The fast kernel
    on a slab holding r raises flag 2; on a slab next to r it raises nothing; the exact kernel (modes 3
    and 2, every third / sixth pair) gives the oracle on a slab around r."""
    rng = np.random.default_rng(700 + k)
    base = random_knn(rng, k + 12, k)
    n = base.shape[0]
    r = n // 2
    one_row = k > 128  # the CTA-per-row and the exact kernels are slow to emulate at these k
    for i, (p, q) in enumerate(_dup_pairs(k)):
        idx = base.copy()
        idx[r, q] = idx[r, p]
        grid = (1, 3)[i % 2]
        _, _, _, flags = run_slab(emu, idx, 1, r, r + 1, grid=grid)
        assert flags & FLAG_DUP, (p, q)
        if i % 8 == 0:
            _, _, _, flags = run_slab(emu, idx, 1, r + 1, min(n, r + 4), grid=grid)
            assert flags == 0, (p, q)
        if i % 3 == 0:
            lo, hi = (r, r + 1) if one_row else (r - 1, r + 2)
            if not one_row and i % 9 == 3:
                lo, hi = 0, n
            out, _, _, _ = run_slab(emu, idx, 3, lo, hi, grid=grid)
            assert np.array_equal(out, oracle.parallel_rows(idx, lo, hi)), (p, q)
            if i % 6 == 0:
                out, _, nw, _ = run_slab(emu, idx, 2, lo, hi, grid=grid)
                want, m = serial_slab(oracle.serial(idx), lo, hi, k)
                assert nw == m and np.array_equal(out, want), (p, q)
        if k <= 32 and i % 5 == 0:  # the fused and the mutual-bit forms of the same kernel
            for mode in (0, 4):
                assert run_slab(emu, idx, mode, r, r + 1, grid=grid)[3] & FLAG_DUP, (mode, p, q)


# ---------------------------------------------------------------- forced hash failure
def _log_ts(L, k):
    v = int(L.emu_jaccard_variant(k))
    return {4: 6, 8: 6, 16: 7, 32: 9}[v] if v < 1000 else v - 1000


def _collides_at_first_multiplier(idx, log_ts):
    """Rows whose ids share a table slot under kMult0: slot(x) = (x * m mod 2^32) >> (32 - LOG_TS)."""
    a = (np.asarray(idx) - 1).astype(np.uint64)
    slots = ((a * np.uint64(K_MULT0)) & np.uint64(0xFFFFFFFF)) >> np.uint64(32 - log_ts)
    return np.array([len(set(s.tolist())) < a.shape[1] for s in slots])


@pytest.mark.parametrize("k", [3, 5, 8, 12, 16, 20, 30, 32, 33, 45, 46, 64, 65, 100, 128])
def test_hash_failure_flag_and_fallback(emu1, oracle, k):
    """With one multiplier allowed, flag 4 is raised exactly when the slab holds a row whose ids collide
    under kMult0; the counts of every other row stay right, and the exact path gives the oracle."""
    rng = np.random.default_rng(900 + k)
    log_ts = _log_ts(emu1, k)
    # ids drawn from 3000 cells: kMult0 spreads a few hundred consecutive small ids over the table
    # without a single collision, so a small matrix would never fail
    n = 3000
    idx = random_knn(rng, n, k)
    coll = _collides_at_first_multiplier(idx, log_ts)
    assert 0.01 < coll.mean() < 0.99, "input does not discriminate"
    clean, hits = np.flatnonzero(~coll), np.flatnonzero(coll)
    span = 40 if k <= 32 else 10
    slabs = [(7, 7 + span), (int(hits[0]), int(hits[0]) + 1), (int(clean[3]), int(clean[3]) + 1),
             (n - span, n)]
    for lo, hi in slabs:
        par = oracle.parallel_rows(idx, lo, hi)
        for mode in (1, 0):
            out, cnt, _, flags = run_slab(emu1, idx, mode, lo, hi, grid=2)
            assert bool(flags & FLAG_HASH) == bool(coll[lo:hi].any()), (mode, lo, hi, flags)
            assert flags & ~FLAG_HASH == 0
            ok = ~coll[lo:hi]
            if mode == 1:
                assert np.array_equal(cnt[ok], u_of(par, k)[ok])
            else:
                assert np.array_equal(out.reshape(hi - lo, k, 3)[ok], par.reshape(hi - lo, k, 3)[ok])
        out, _, _, _ = run_slab(emu1, idx, 3, lo, hi, grid=2)
        assert np.array_equal(out, par)
    lo = int(hits[0])
    if k <= 127:  # the mutual-bit counts of the graph build raise it too
        assert run_slab(emu1, idx, 4, lo, lo + 1)[3] & FLAG_HASH
    if k <= 32:
        assert run_slab(emu1, idx, 5, lo, lo + 1)[3] & FLAG_HASH


def test_variant_numbering(emu):
    """The kernel each k is dispatched to, numbered like gficf_cuda_last_launch reports it (the GPU test
    tests/test_gpu_jaccard_slabs.py compares these numbers with the product's launches)."""
    want = {1: 4, 4: 4, 5: 8, 8: 8, 9: 16, 16: 16, 17: 32, 32: 32, 33: 1010, 45: 1010, 46: 1011, 64: 1011, 65: 1012,
            128: 1012, 129: 2000, 255: 2000, 256: 2001, 1024: 2001, 1025: 0}
    assert {k: int(emu.emu_jaccard_variant(k)) for k in want} == want
