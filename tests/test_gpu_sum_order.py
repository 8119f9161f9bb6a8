"""GPU (-m gpu): the sums that must follow the reference's order, on inputs where the order changes
the result (tests/sum_order_cases.py), bit for bit against the oracle:

* the Mann-Whitney tie term above N = 208 064, through gficf_cuda_wmu_test and gficf_cuda_wmu_markers;
* the exact replay of std::accumulate in the network pieces: a total edge weight long and tie-heavy
  enough for capped windows, an intra-cluster sum that starts with a long
  run of masked-out edges, and the self-link total of a reduced network (s0 != 0).

tests/test_sum_order_emu.py runs the same kernels on the CPU emulation."""
import numpy as np
import pytest

from oracle.binding import NetworkOracle, WmuOracle
from tests.network_cases import assert_same_network, random_lower
from tests.sum_order_cases import SEQ_MAX_BLOCKS, assert_discriminates, sensitive_genes, tie_weights, window_schedule
from tests.test_gpu_network import as_dict, full_clustering, gpu_network

pytestmark = pytest.mark.gpu

KINDS = ("shifted", "plain", "negative", "dense")


@pytest.mark.parametrize("n_cells,n1", [(300_000, 40_000), (400_000, 150_000)])
def test_wmu_ordered_tie_sum(cuda, n_cells, n1):
    first = np.arange(n_cells) < n1
    m, against = sensitive_genes(n_cells, n_cells, first, KINDS)
    orc = WmuOracle()
    for v, a in zip(m, against):
        assert_discriminates(v, [first], orc, a)
    x, y = np.asfortranarray(m[:, :n1]), np.asfortranarray(m[:, n1:])
    assert np.array_equal(cuda.rcpp_parallel_WMU_test(x, y), orc.wmu(x, y), equal_nan=True)


@pytest.mark.parametrize("n_cells", [300_000, 400_000])
def test_markers_ordered_tie_sum(cuda, n_cells):
    """Five clusters, one of them a single cell; every block against the oracle and against the
    per-cluster call on the same split."""
    rng = np.random.default_rng(n_cells + 1)
    cl = rng.integers(0, 4, n_cells).astype(np.int32)
    cl[rng.integers(0, n_cells)] = 4
    k = 5
    m, against = sensitive_genes(n_cells + 2, n_cells, cl == 1, KINDS)
    orc = WmuOracle()
    for v, a in zip(m, against):
        assert_discriminates(v, [cl == c for c in range(k)], orc, a)
    got = cuda.rcpp_parallel_WMU_markers(m, cl)
    assert got.shape == (m.shape[0], 2, k)
    for c in range(k):
        x, y = np.asfortranarray(m[:, cl == c]), np.asfortranarray(m[:, cl != c])
        want = orc.wmu(x, y)
        assert np.array_equal(got[:, :, c], want, equal_nan=True), c
        assert np.array_equal(got[:, :, c], cuda.rcpp_parallel_WMU_test(x, y), equal_nan=True), c


@pytest.fixture(scope="module")
def tie_graph():
    """2.6M lower-triangle entries (5.2M directed edges) with tie-heavy positive weights, its oracle
    network, and a device network built from it."""
    rng = np.random.default_rng(31)
    n1, n2, _ = random_lower(rng, 200_000, 2_600_000)
    w = tie_weights(rng, n1.size)
    nv = int(max(n1.max(), n2.max())) + 1
    want = NetworkOracle().network(n1, n2, w)
    return want, gpu_network(n1, n2, w, nv)


def test_network_total_weight_in_capped_windows(cuda, tie_graph):
    want, net = tie_graph
    assert any(b == SEQ_MAX_BLOCKS for _, b, _ in window_schedule(want["edge_w"]))  # getTotalEdgeWeight's sum
    assert_same_network(as_dict(net), want)


def _intra(net, cl):
    """The weights calcQualityFunction adds, in its order: edge weights with 0 for edges that leave the
    cluster."""
    src = np.repeat(np.arange(net["n_nodes"]), np.diff(net["first"]))
    return np.where(cl[src] == cl[net["neighbor"]], net["edge_w"], 0.0)


def test_network_quality_and_reduction_after_leading_zeros(cuda, tie_graph):
    """A clustering whose lowest nodes are singletons: the first ~100k directed edges leave their
    cluster, so the intra-cluster sum of the quality function and the self-link sum of the reduced
    network both start with a long run of zeros.  Then an ordinary clustering, and the next level,
    whose self-link total starts from the parent's non-zero one."""
    want, net = tie_graph
    O = NetworkOracle()
    nv = want["n_nodes"]
    rng = np.random.default_rng(32)
    p = int(np.searchsorted(want["first"], 100_000)) + 1  # nodes [0, p) own the first >= 100k edges
    cl = np.empty(nv, np.int32)
    cl[:p] = np.arange(p)
    cl[p:] = p + full_clustering(rng, nv - p, 300)
    lead = np.flatnonzero(_intra(want, cl))
    assert lead.size and lead[0] >= 100_000
    res = 0.8 / (2 * want["total_w"])
    plain = full_clustering(rng, nv, 500)
    for c in (cl, plain):
        q_want, cw_want = O.quality(want, c, res)
        assert net.calc_quality_function(c, res) == q_want
        assert np.array_equal(net.cluster_weights(c).cpu().numpy(), cw_want)
    red_want = O.reduce(want, cl)
    red = net.create_reduced_network(cl)
    assert_same_network(as_dict(red), red_want)
    assert red_want["self_links"] > 0
    # level 1: quality and reduction of the reduced network, self-link sums from s0 != 0
    nc = int(cl.max()) + 1
    cl2 = full_clustering(rng, nc, 40)
    q2_want, cw2_want = O.quality(red_want, cl2, res)
    assert red.calc_quality_function(cl2, res) == q2_want
    assert np.array_equal(red.cluster_weights(cl2).cpu().numpy(), cw2_want)
    red2_want = O.reduce(red_want, cl2)
    assert_same_network(as_dict(red.create_reduced_network(cl2)), red2_want)
    assert red2_want["self_links"] != red_want["self_links"]
