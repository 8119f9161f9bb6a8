"""CPU: gficf_cuda_wmu_markers_csc_devices, the sparse markers call with the genes split over D devices, run on
the CUDA emulation (tests/cuda_emu/wmu_markers_multi_emu.cpp): the product's plan from wmu_csc_plan.h -- column
slabs, transpose per slab, gene ranges and exchange table, the exchange as copies between per-device buffers,
wmu_regroup_kernel, the rank + means launches of each gene range and the finish into its rows -- bit for bit
against the emulated single-device call for D = 1, 2, 3, 4, 8.  Also the partition functions on their own, a bad
row id that only the last slab holds, and the host-side argument errors of the C entry and the Python mirror.
tests/test_gpu_wmu_markers_multi.py runs the call on several B200s."""
import ctypes as C

import numpy as np
import pytest
import scipy.sparse as sp

import gficf_b200
from tests.test_wmu_markers_sparse_emu import build_emu, edge_rows, emu_sparse, load_sparse_emu, to_csc
from tests.test_wmu_oracle import sc_matrix

_dp = C.POINTER(C.c_double)
_ip = C.POINTER(C.c_int32)
_lp = C.POINTER(C.c_longlong)
DEVICES = (1, 2, 3, 4, 8)


@pytest.fixture(scope="module")
def single(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emu") / "libwmu_markers_sparse_emu.so")
    build_emu(so, "wmu_markers_sparse_emu.cpp")
    return load_sparse_emu(so)


@pytest.fixture(scope="module")
def multi(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emu") / "libwmu_markers_multi_emu.so")
    build_emu(so, "wmu_markers_multi_emu.cpp")
    L = C.CDLL(so)
    L.emu_cell_slabs.argtypes = [_ip, C.c_longlong, C.c_int, _lp]
    L.emu_cell_slabs.restype = None
    L.emu_gene_ranges.argtypes = [_lp, C.c_longlong, C.c_int, _lp]
    L.emu_gene_ranges.restype = None
    L.emu_wmu_markers_csc_devices.argtypes = [_ip, _ip, _dp, C.c_longlong, C.c_longlong, _ip, C.c_int, C.c_int, _dp,
                                              C.c_int, C.c_int]
    L.emu_wmu_markers_csc_devices.restype = C.c_uint
    return L


def cell_slabs(L, colptr, D):
    colptr = np.ascontiguousarray(colptr, dtype=np.int32)
    c = np.empty(D + 1, dtype=np.int64)
    L.emu_cell_slabs(colptr.ctypes.data_as(_ip), colptr.size - 1, D, c.ctypes.data_as(_lp))
    return c


def gene_ranges(L, counts, D):
    G = np.ascontiguousarray(np.concatenate([[0], np.cumsum(counts)]), dtype=np.int64)
    g = np.empty(D + 1, dtype=np.int64)
    L.emu_gene_ranges(G.ctypes.data_as(_lp), counts.size, D, g.ctypes.data_as(_lp))
    return g


def emu_multi(L, colptr, row, x, genes, cl, k, D, grid=3, ctas=2):
    cl = np.ascontiguousarray(cl, dtype=np.int32)
    out = np.full((genes, 2, k), -7.0, order="F")
    flags = L.emu_wmu_markers_csc_devices(colptr.ctypes.data_as(_ip), row.ctypes.data_as(_ip), x.ctypes.data_as(_dp),
                                          genes, colptr.size - 1, cl.ctypes.data_as(_ip), k, D,
                                          out.ctypes.data_as(_dp), grid, ctas)
    return out, flags


def check_devices(single, multi, m, cl, k, stored_zeros=0.1, seed=0, devices=DEVICES, grid=3, ctas=2):
    colptr, row, x, m = to_csc(m, np.random.default_rng(seed), stored_zeros)
    want, flags = emu_sparse(single, colptr, row, x, m.shape[0], cl, k, grid, ctas)
    assert flags == 0
    for D in devices:
        got, flags = emu_multi(multi, colptr, row, x, m.shape[0], cl, k, D, grid, ctas)
        assert flags == 0, D
        assert np.array_equal(got.view(np.int64), want.view(np.int64)), D
    return colptr


def clusters(rng, cells, k):
    cl = rng.integers(0, k, size=cells).astype(np.int32)
    cl[:k] = np.arange(k)
    rng.shuffle(cl)
    return cl


def test_unequal_columns_empty_columns_and_edge_genes(single, multi):
    """Columns of very unequal density (a few nearly full, most nearly empty, runs of empty ones), stored zeros
    and -0.0, and the special genes: no stored value, every cell stored (values in every slab), below -1, past
    2^53, subnormals."""
    rng = np.random.default_rng(11)
    genes, cells, k = 24, 900, 6
    cl = clusters(rng, cells, k)
    m = edge_rows(rng, sc_matrix(rng, genes, cells, density=0.05), cl)
    dense_cols = rng.choice(cells, size=12, replace=False)
    m[:, dense_cols] = rng.random((genes, 12)) + 0.25
    m[:, 100:180] = 0.0
    m[:, [0, cells - 1]] = 0.0
    check_devices(single, multi, m, cl, k, stored_zeros=0.1, seed=1)


def test_empty_genes_at_range_boundaries(single, multi):
    """Every other gene has no stored value, so the gene ranges start and end next to empty genes."""
    rng = np.random.default_rng(12)
    genes, cells, k = 32, 600, 4
    cl = clusters(rng, cells, k)
    m = sc_matrix(rng, genes, cells, density=0.3)
    m[0::2] = 0.0
    colptr = check_devices(single, multi, m, cl, k, stored_zeros=0.0)
    counts = (m != 0).sum(axis=1)
    for D in (2, 3, 4, 8):
        g = gene_ranges(multi, counts, D)
        assert any(counts[b] == 0 or counts[b - 1] == 0 for b in g[1:-1]), D
    assert colptr[-1] == (m != 0).sum()


def test_slabs_without_stored_values(single, multi):
    """All stored values in three columns: most slabs have cells but no value, or no cell at all."""
    rng = np.random.default_rng(13)
    genes, cells, k = 10, 200, 3
    cl = clusters(rng, cells, k)
    m = np.zeros((genes, cells))
    for j in (3, 4, 150):
        m[:, j] = rng.random(genes) + 0.5
    colptr, _, _, _ = to_csc(m)
    c = cell_slabs(multi, colptr, 8)
    assert (np.diff(colptr[c]) == 0).sum() >= 5
    check_devices(single, multi, m, cl, k, stored_zeros=0.0)
    check_devices(single, multi, np.zeros((genes, cells)), cl, k, stored_zeros=0.0)   # nothing stored at all
    check_devices(single, multi, np.zeros((genes, cells)), cl, k, stored_zeros=0.3, seed=4)  # only zeros stored


def test_fewer_genes_or_cells_than_devices(single, multi):
    rng = np.random.default_rng(14)
    cl = clusters(rng, 300, 3)
    check_devices(single, multi, sc_matrix(rng, 3, 300, density=0.4), cl, 3)        # n_genes < D: D = n_genes
    check_devices(single, multi, sc_matrix(rng, 1, 300, density=0.4), cl, 3)        # one gene: one device
    cl = np.array([0, 1, 2, 0, 1], dtype=np.int32)
    check_devices(single, multi, sc_matrix(rng, 12, 5, density=0.6), cl, 3)         # n_cells < D: empty slabs


def test_many_tie_groups_and_grids(single, multi):
    """Integer counts (many ties), one rank-kernel CTA per device, then several; the means kernel with more
    clusters than one CTA covers."""
    rng = np.random.default_rng(15)
    genes, cells, k = 14, 1200, 40
    cl = clusters(rng, cells, k)
    m = edge_rows(rng, sc_matrix(rng, genes, cells, integer=True), cl)
    check_devices(single, multi, m, cl, k, grid=1, ctas=1, devices=(2, 4))
    check_devices(single, multi, m, cl, k, grid=5, ctas=3, devices=(3, 8))


def test_partition_covers_and_balances(multi):
    rng = np.random.default_rng(16)
    for trial in range(300):
        cells = int(rng.integers(0, 60))
        D = int(rng.integers(1, 17))
        cnt = rng.integers(0, 5, cells) * (rng.random(cells) < rng.random())
        if trial % 7 == 0 and cells:
            cnt[rng.integers(0, cells)] = 500                      # one very dense column
        colptr = np.concatenate([[0], np.cumsum(cnt)]).astype(np.int32)
        c = cell_slabs(multi, colptr, D)
        assert c[0] == 0 and c[-1] == cells and (np.diff(c) >= 0).all()
        nnz = int(colptr[-1])
        for r in range(1, D):                                      # slab r starts at the first column at r nnz / D
            assert colptr[c[r]] >= nnz * r // D and (c[r] == 0 or colptr[c[r] - 1] < nnz * r // D)

        genes = int(rng.integers(1, 80))
        D = int(rng.integers(1, min(genes, 16) + 1))
        counts = rng.integers(0, 30, genes) * (rng.random(genes) < rng.random())
        if trial % 5 == 0:
            counts[rng.integers(0, genes)] = 2000                  # one gene with most of the values
        g = gene_ranges(multi, counts, D)
        assert g[0] == 0 and g[-1] == genes and (np.diff(g) >= 1).all()   # every gene once, no range empty
        G = np.concatenate([[0], np.cumsum(counts)])
        big = counts.max(initial=0)
        for d in range(1, D):
            target = G[-1] * d // D
            forced = g[d] == g[d - 1] + 1 or g[d] == genes - (D - d)
            if not forced:                                          # the cut is within one gene of its share
                assert target <= G[g[d]] < target + max(big, 1), (trial, d)


def test_bad_row_id_in_the_last_slab_only(single, multi):
    rng = np.random.default_rng(17)
    genes, cells, k = 9, 80, 3
    cl = clusters(rng, cells, k)
    colptr, row, x, _ = to_csc(sc_matrix(rng, genes, cells, density=0.4))
    for D in (2, 3, 4, 8):
        c = cell_slabs(multi, colptr, D)
        for name, val in (("past n_genes", genes), ("negative", -1), ("repeated", None)):
            r = row.copy()
            if val is None:                                         # second value of the slab's last column with two
                j = c[-2] + np.flatnonzero(np.diff(colptr[c[-2]:]) >= 2)[-1]
                last = colptr[j] + 1
            else:
                last = colptr[-1] - 1
            assert last >= colptr[c[-2]]                            # in the last slab
            r[last] = r[last - 1] if val is None else val
            out, flags = emu_multi(multi, colptr, r, x, genes, cl, k, D)
            assert flags == 1 and (out == -7.0).all(), (D, name)
            assert emu_sparse(single, colptr, r, x, genes, cl, k)[1] == 1
    out, flags = emu_multi(multi, colptr, row, x, genes, cl, k, 4)
    assert flags == 0 and not (out == -7.0).any()


def _abi(colptr, row, x, genes, cl, k, n_devices, cells=None):
    L = gficf_b200.lib()
    err = C.create_string_buffer(256)
    out = np.empty(64)  # every call here fails or returns before the output is written
    p = lambda a: None if a is None else a.ctypes.data  # noqa: E731
    cells = (colptr.size - 1 if colptr is not None else 0) if cells is None else cells
    rc = L.gficf_cuda_wmu_markers_csc_devices(p(colptr), p(row), p(x), genes, cells, p(cl), k, n_devices,
                                              out.ctypes.data, err, 256)
    return rc, err.value.decode()


def test_argument_errors_without_gpu():
    """The host checks of the single-device call, in the same order, before any device is touched."""
    colptr = np.array([0, 2, 2, 5, 6], dtype=np.int32)
    row = np.array([0, 3, 1, 2, 4, 0], dtype=np.int32)
    x = np.arange(1.0, 7.0)
    cl = np.array([0, 1, 0, 1], dtype=np.int32)
    rc, msg = _abi(np.array([1, 2, 2, 5, 6], dtype=np.int32), row, x, 5, cl, 2, 2)
    assert rc == 1 and "colptr[0]" in msg
    rc, msg = _abi(np.array([0, 2, 1, 5, 6], dtype=np.int32), row, x, 5, cl, 2, 2)
    assert rc == 1 and "decreases" in msg
    assert _abi(colptr, row, x, -1, cl, 2, 2)[0] == 1
    assert _abi(None, row, x, 5, cl, 2, 2, cells=4)[0] == 1
    assert _abi(colptr, None, x, 5, cl, 2, 2)[0] == 1
    assert _abi(colptr, row, x, 5, None, 2, 2)[0] == 1
    rc, msg = _abi(colptr, row, x, 5, np.array([0, 2, 0, 2], np.int32), 3, 2)
    assert rc == 1 and "no cells" in msg
    assert _abi(colptr, row, x, 5, cl, 8193, 2)[0] == 5
    assert _abi(colptr, row, x, 1 << 31, cl, 2, 2)[0] == 5
    rc, msg = _abi(colptr, row, x, 5, cl, 2, -1)
    assert rc == 1 and "n_devices" in msg
    assert _abi(colptr, row, x, 0, cl, 2, 2)[0] == 0                  # no genes: nothing to do
    if gficf_b200.lib().gficf_cuda_device_count() == 0:
        assert _abi(colptr, row, x, 5, cl, 2, 2)[0] == 3               # no device, no fallback


def test_mirror_passes_n_devices():
    m = sp.csc_matrix(np.eye(4, 6))
    f = gficf_b200.rcpp_parallel_WMU_markers_sparse
    with pytest.raises(gficf_b200.GficfCudaError) as e:
        f(m, np.array([0, 2, 0, 2, 0, 2]), n_devices=2)                   # cluster 1 is empty
    assert e.value.code == 1
    with pytest.raises(gficf_b200.GficfCudaError) as e:
        f(m, np.array([0, 1, 0, 1, 0, 1]), n_devices=-1)
    assert e.value.code == 1 and "n_devices" in e.value.message
    assert f(sp.csc_matrix((0, 6)), np.array([0, 1, 0, 1, 0, 1]), n_devices=4).shape == (0, 2, 2)
