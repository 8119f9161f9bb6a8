"""GPU (-m gpu): the SNN graph built on the device (gficf_b200.snn) equals what the reference's
R / igraph / C++ steps produce from the edge matrix (oracle/louvain.py restates them), and gives
the same Louvain labels through the reference's ModularityOptimizer."""
import os
import subprocess
import tempfile

import numpy as np
import pytest
import torch

from gficf_b200 import synth
from oracle import louvain
from oracle.binding import MODOPT_BIN

pytestmark = pytest.mark.gpu


def _gpu_triangle(n, k, idx0):
    from gficf_b200 import device as D, snn

    padded, _ = D.pad_rows(idx0.cuda())
    colptr, rows, w, vcell, flags = snn.snn_lower_triangle(padded, n, k, with_vertex_map=True)
    torch.cuda.synchronize()
    return colptr.cpu().numpy(), rows.cpu().numpy(), w.cpu().numpy(), vcell.cpu().numpy(), int(flags[0])


def _same_graph(names, cols, rows_ref, data_ref, colptr, rows, w, vcell):
    assert np.array_equal(vcell, names)  # igraph's vertex numbering: first appearance in c(from, to)
    assert colptr.shape[0] == names.shape[0] + 1
    assert np.array_equal(np.repeat(np.arange(names.shape[0]), np.diff(colptr)), cols)
    assert np.array_equal(rows, rows_ref)
    assert np.array_equal(w, data_ref)  # bit-exact sums


@pytest.mark.parametrize("n,k,family", [(20_000, 15, "planted"), (30_000, 30, "planted"), (5_000, 100, "planted"),
                                         (3_000, 30, "uniform"), (300, 7, "planted"), (2_000, 5, "uniform"),
                                         (50_000, 4, "uniform")])
def test_lower_triangle_matches_reference_steps(cuda, oracle, n, k, family):
    """Incl. the uniform family, where many cells keep no edge of their own: igraph then numbers the
    vertices differently from the cells (target-only vertices last, absent cells not at all)."""
    idx0 = synth.knn_index(n, k, family=family, scramble=True)
    rel = oracle.parallel(synth.to_r_matrix(idx0))
    names, cols, rows_ref, data_ref = louvain.lower_triangle_edges(rel)
    colptr, rows, w, vcell, flags = _gpu_triangle(n, k, idx0)
    assert flags & ~16 == 0
    assert bool(flags & 16) or np.array_equal(names, np.arange(1, n + 1))  # not the identity -> ISOLATED was raised
    _same_graph(names.astype(np.int64), cols, rows_ref, data_ref, colptr, rows, w, vcell)


def test_hub_vertices_take_the_big_column_sorts(cuda, oracle):
    """Columns beyond 32 / 512 / 4096 entries (warp rank sort, shared-memory bitonic, CTA rank sort)."""
    n, k = 12_000, 10
    rng = np.random.default_rng(4)
    idx = synth.knn_index(n, k, family="planted", scramble=False).numpy().copy()
    # cells 0, 1, 2 become hubs: many rows list them (and each other's neighbourhoods overlap)
    for hub, fans in ((0, 6000), (1, 900), (2, 100)):
        rows = rng.choice(np.arange(10, n), fans, replace=False)
        for r in rows:
            if hub not in idx[r]:
                idx[r, rng.integers(0, k)] = hub
    idx[:, 0] = np.where((idx[:, 1:] == 5).any(axis=1) | (np.arange(n) == 5), idx[:, 0], 5)  # a shared neighbour: u > 0
    idx0 = torch.from_numpy(idx)
    rel = oracle.parallel(synth.to_r_matrix(idx0))
    names, cols, rows_ref, data_ref = louvain.lower_triangle_edges(rel)
    colptr, rows, w, vcell, flags = _gpu_triangle(n, k, idx0)
    if flags & 2:
        pytest.skip("the construction produced a repeated id")
    assert np.diff(colptr).max() > 4096
    _same_graph(names.astype(np.int64), cols, rows_ref, data_ref, colptr, rows, w, vcell)


def test_host_buffer_entry(cuda, oracle):
    """gficf_cuda_snn_lower: kNN matrix in host memory -> CSC arrays in host memory, f64 and int32."""
    from gficf_b200 import snn

    for n, k, family in ((40_000, 30, "planted"), (4_000, 6, "uniform")):
        idx0 = synth.knn_index(n, k, family=family, scramble=True)
        r = synth.to_r_matrix(idx0)
        names, cols, rows_ref, data_ref = louvain.lower_triangle_edges(oracle.parallel(r))
        for mat in (r, r.astype(np.int32)):
            g = snn.snn_graph(mat)
            assert g["n_vertices"] == names.shape[0] and g["nnz"] == rows_ref.shape[0]
            _same_graph(names.astype(np.int64), cols, rows_ref, data_ref, g["colptr"], g["row"], g["weight"],
                        g["vertex_cell"])
    bad = synth.to_r_matrix(synth.knn_index(100, 5))
    bad[3, 1] = bad[3, 2]
    with pytest.raises(cuda.GficfCudaError) as e:
        snn.snn_graph(bad)
    assert e.value.code == 5
    with pytest.raises(cuda.GficfCudaError) as e:
        snn.snn_graph(synth.to_r_matrix(synth.knn_index(300, 128)))
    assert e.value.code == 5


def test_self_ids_in_the_graph_build(cuda, oracle):
    """Duplicate cells keep themselves in their neighbour list after neigh[, -1]: rows that list their
    own cell (a self loop with u = k) next to rows that do not, device and host-buffer entries."""
    from gficf_b200 import snn
    from tests.test_jaccard_slabs_emu import self_ids

    n, k = 6_000, 30
    rng = np.random.default_rng(6)
    a = np.ascontiguousarray(self_ids(rng, k, n) - 1, dtype=np.int32)
    for i in np.flatnonzero(rng.random(n) < 0.5):  # half the rows drop their self id again
        j = int(np.flatnonzero(a[i] == i)[0])
        a[i, j] = rng.choice(np.setdiff1d(np.arange(n), np.append(a[i], i)))
    idx0 = torch.from_numpy(a)
    r = synth.to_r_matrix(idx0)
    names, cols, rows_ref, data_ref = louvain.lower_triangle_edges(oracle.parallel(r))
    colptr, rows, w, vcell, flags = _gpu_triangle(n, k, idx0)
    assert flags & ~16 == 0
    _same_graph(names.astype(np.int64), cols, rows_ref, data_ref, colptr, rows, w, vcell)
    g = snn.snn_graph(r)
    _same_graph(names.astype(np.int64), cols, rows_ref, data_ref, g["colptr"], g["row"], g["weight"], g["vertex_cell"])


@pytest.mark.skipif(not os.path.exists(MODOPT_BIN), reason="oracle/_ref/modopt not shipped")
def test_labels_from_device_graph(cuda, oracle):
    n, k = 50_000, 30
    idx0 = synth.knn_index(n, k)
    colptr, rows, w, vcell, flags = _gpu_triangle(n, k, idx0)
    assert flags == 0 and np.array_equal(vcell, np.arange(1, n + 1))
    cols = np.repeat(np.arange(n), np.diff(colptr))
    with tempfile.TemporaryDirectory() as d:
        fin, fout = os.path.join(d, "e.tsv"), os.path.join(d, "l.txt")
        with open(fin, "w") as f:
            for x, y, z in zip(cols.tolist(), rows.tolist(), w.tolist()):
                f.write("%d\t%d\t%.17g\n" % (x, y, z))
        p = louvain.DEFAULTS
        subprocess.run([MODOPT_BIN, fin, fout, str(p["modularity"]), repr(p["resolution"]), str(p["algorithm"]),
                        "1", "10", str(p["seed"]), "0"], check=True, capture_output=True)
        lab_gpu = np.loadtxt(fout, dtype=np.int64)
    rel = oracle.parallel(synth.to_r_matrix(idx0))
    cells, lab_ref = louvain.louvain_labels(rel, n_start=1, n_iter=10)
    assert np.array_equal(cells, np.arange(1, n + 1))
    assert np.array_equal(lab_gpu, lab_ref)


def test_device_graph_is_the_input_of_the_stored_reference_labels(cuda, oracle):
    """Label parity with nothing outside the repository: tests/golden/net_snn_900_k12_louvain.npz holds
    the lower-triangle edge list of this seeded 900 x 12 matrix and the Louvain labels the reference's
    own ModularityOptimizer returned for it (tests/golden/make_golden.py).  The graph built on the
    device is that edge list bit for bit, so the reference's optimiser returns those labels for it, and
    the network of the device graph gives the stored quality value for them."""
    from gficf_b200 import modularity

    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "net_snn_900_k12_louvain.npz"))
    n, k = 900, 12
    idx0 = synth.knn_index(n, k, family="planted", scramble=True)
    names = louvain.lower_triangle_edges(oracle.parallel(synth.to_r_matrix(idx0)))[0]
    colptr, rows, w, vcell, flags = _gpu_triangle(n, k, idx0)
    assert flags & ~16 == 0 and np.array_equal(vcell, names.astype(np.int64))
    assert np.array_equal(np.repeat(np.arange(vcell.size), np.diff(colptr)), g["node1"])
    assert np.array_equal(rows, g["node2"]) and np.array_equal(w, g["w"])
    net = modularity.matrix_to_network(*(torch.from_numpy(x).cuda() for x in (colptr, rows, w)))
    assert net.calc_quality_function(g["cluster"], float(g["resolution"])) == float(g["quality"])


def test_snn_timing_record(cuda):
    """Not a pass/fail gate: prints the device time of the whole step at 1M x 30."""
    from gficf_b200 import device as D, snn

    n, k = 1_000_000, 30
    idx0 = synth.knn_index(n, k, scramble=True, device="cuda")
    padded, _ = D.pad_rows(idx0)
    snn.snn_lower_triangle(padded, n, k)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    colptr, rows, w, flags = snn.snn_lower_triangle(padded, n, k)
    e1.record()
    torch.cuda.synchronize()
    print("SNN 1M x 30: %.2f ms, nnz=%d" % (e0.elapsed_time(e1), rows.numel()))
    assert int(flags[0]) == 0
