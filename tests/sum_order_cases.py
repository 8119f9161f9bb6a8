"""Shared inputs of the ordered-sum tests (tests/test_sum_order_emu.py on the CPU emulation,
tests/test_gpu_sum_order.py on the GPU).

Two results of this project are bit-identical to the reference only because a sequential double sum
is replayed in the reference's order:

* the Mann-Whitney tie term sum(t^3 - t), which the reference adds over the tie groups in sorted
  order (rcpp_parallel_mann_whitney.cpp; oracle/wmu_oracle.c:82-83).  Below 2^53 every partial sum is
  an exact integer and any order gives the same double, so a test input must push the total past 2^54,
  where adding a pair's 6 to a multiple of 4 is a rounding tie: `order_sensitive_gene`;
* std::accumulate over the whole graph (network_kernels.cuh, "The reference's whole-graph sums"),
  replayed a window of up to kSeqMaxBlocks x kSeqBlock elements at a time: the families below are long
  enough to reach capped windows and to leave a binade inside one (`window_schedule`).

`tie_terms` says, in numpy, whether an input discriminates at all: the tests assert that the sorted
order gives another p-value than an integer sum or a "zero group first" sum, so an input that stops
telling the orders apart fails instead of passing vacuously."""
import math

import numpy as np

# network_kernels.cuh
SEQ_BLOCK = 4096
SEQ_MAX_BLOCKS = 1024


# ---- Mann-Whitney: genes whose tie term depends on the order of the sum ---------------------------

def order_sensitive_gene(rng, N, n_zero, signs="random", big=None, shift=None):
    """One gene of N cells: n_zero zeros (one tie group) and N - n_zero non-zero values drawn as
    pairs 1, 1, 2, 2, 3, 3, ... -- each pair a tie group of 2 whose term t^3 - t = 6 is a rounding tie
    once the running sum is in [2^54, 2^55) -- with random signs (signs="random") or all negative
    (signs="negative": every group sorts before the zeros).  `big` = (value, count) puts one more
    large group of that value in place of `count` pairs' cells (the dense variant: a large negative
    group that sorts first).  `shift` is a boolean mask of cells whose non-zero values get +0.25,
    which breaks the pairs that straddle it (a group of cells that differs from the rest)."""
    v = np.zeros(N)
    nnz = N - n_zero
    pos = rng.permutation(N)[:nnz]
    vals = np.repeat(np.arange(1, nnz // 2 + 2, dtype=np.float64), 2)[:nnz]
    if signs == "random":
        vals = vals * np.where(rng.random(nnz) < 0.5, -1.0, 1.0)
    else:
        vals = -vals
    if big is not None:
        value, count = big
        vals[:count] = value
    v[pos] = vals
    if shift is not None:
        v[shift & (v != 0)] += 0.25
    return v


def _z(n1, n2, two_r1, nties):
    """z of oracle/wmu_oracle.c:81-87 from the exact rank sum and a tie term, in its operation order."""
    n = n1 + n2
    u1 = (two_r1 - n1 * (n1 + 1)) / 2          # multiples of 1/2 below 2^53: exact
    u2 = ((n * (n + 1) - two_r1) - n2 * (n2 + 1)) / 2
    mu = float((n1 * n2) // 2)
    d1, d2 = float(n1), float(n2)
    sig = math.sqrt((d1 * d2 / 12) * ((d1 + d2 + 1) - nties / ((d1 + d2) * (d1 + d2 - 1))))
    z = u1 - mu if u1 < u2 else u2 - mu
    z = z + 0.5 if z < 0 else z - 0.5
    return z / sig


def tie_terms(v, in_group1):
    """The tie term of gene v summed three ways -- "sorted" (the reference's order), "int" (exact
    integers, rounded once), "zeros_first" (the zero group before the negative groups) -- each carried
    through getSigma and z for the split in_group1 (boolean mask) against the rest.
    Returns {order: (tie_sum, z)}."""
    v = np.asarray(v, dtype=np.float64) + 0.0  # -0.0 ties with +0.0
    vals, inv, counts = np.unique(v, return_inverse=True, return_counts=True)
    # 2 R1 exactly: a group at sorted positions [i, j) has the averaged rank (i + j + 1) / 2 (1-based)
    ends = np.cumsum(counts)
    two_rank = (2 * ends - counts + 1)[inv]
    two_r1 = int(two_rank[np.asarray(in_group1, bool)].sum())
    n1 = int(np.count_nonzero(in_group1))
    n2 = v.size - n1
    big = counts >= 2                          # groups of one add exactly 0
    terms = [((t * t) * t) - t for t in counts[big].astype(np.float64).tolist()]
    gvals = vals[big]
    orders = {"sorted": terms,
              "zeros_first": [t for t, g in zip(terms, gvals) if g == 0] + [t for t, g in zip(terms, gvals) if g != 0]}
    out = {}
    tiny = len(vals) >= v.size                 # no ties at all: the reference skips the term (:82)
    for name, seq in orders.items():
        acc = 0.0
        for t in seq:
            acc = acc + t
        out[name] = 0.0 if tiny else acc
    out["int"] = 0.0 if tiny else float(sum(int(t) ** 3 - int(t) for t in counts[big].tolist()))
    return {k: (s, _z(n1, n2, two_r1, s)) for k, s in out.items()}


def pvalue(z, orc):
    """The reference's getPvalue through the oracle's normal cdf (oracle/gauss_cdf.c)."""
    return orc.lib.gsl_cdf_ugaussian_P(z) * 2 if z < 0 else orc.lib.gsl_cdf_ugaussian_Q(z) * 2


def assert_discriminates(v, splits, orc, against=("int", "zeros_first")):
    """The input tells the orders apart where it matters, in the p-value: for every order named in
    `against`, the sorted order gives another p-value in at least one of the splits (boolean masks of
    group 1).  A split whose z is near 0 may not: the p-value is flat there."""
    t = [tie_terms(v, s) for s in splits]
    p = [{k: pvalue(z, orc) for k, (_, z) in ti.items()} for ti in t]
    assert t[0]["sorted"][0] >= 2.0 ** 54, t[0]
    for k in against:
        assert any(pi["sorted"] != pi[k] for pi in p), (k, t)


# what a gene tells apart from the sorted order: an integer sum rounded once ("int"), the zero group
# added before the negative groups ("zeros_first")
GENE_KINDS = {
    "shifted": ("int", "zeros_first"),   # zero group of 280 001, pairs on both sides, pairs in `group` broken
    "plain": ("int", "zeros_first"),     # zero group of 270 003, pairs on both sides
    "negative": ("zeros_first",),        # every group precedes the zeros: one rounding, like the integer sum
    "dense": ("int",),                   # no zeros (nz = 0), a large negative group first
}


def sensitive_genes(seed, N, group, kinds):
    """A matrix of order-sensitive genes of N cells (N > 262 144, so that a group can pass 2^54), one
    row per kind, and what each row discriminates."""
    rng = np.random.default_rng(seed)
    make = {
        "shifted": lambda: order_sensitive_gene(rng, N, 280_001, shift=group),
        "plain": lambda: order_sensitive_gene(rng, N, 270_003),
        "negative": lambda: order_sensitive_gene(rng, N, 280_001, signs="negative"),
        "dense": lambda: order_sensitive_gene(rng, N, 0, signs="negative", big=(-1e6, 270_000)),
    }
    return np.asfortranarray(np.stack([make[k]() for k in kinds])), [GENE_KINDS[k] for k in kinds]


# ---- the exact sum: long inputs ------------------------------------------------------------------

def jaccard_weights(rng, n, k=30):
    """SNN edge weights u / (2k - u'): about 60 distinct values, correlated rounding."""
    return rng.integers(1, k + 1, n) / (2 * k - rng.integers(1, k + 1, n))


def tie_weights(rng, n):
    """Powers of two times {1, 1.5, 3}, some of them half an ulp of the running sum or 1.5 ulp: most
    additions with a small element are rounding ties.  All positive (valid network weights)."""
    e = rng.choice([-32, -31, -30, -29, -2, -1, 0, 1], n)
    return np.ldexp(rng.choice([1.0, 1.5, 3.0], n), e)


def with_long_binade(x, at=4_500_000):
    """x behind one large element B, chosen so that s = B + x[0] + ... stays in one binade for the first
    `at` elements of x and leaves it right after.  The replay's windows follow the binades of the running
    sum, which on a stationary input double in length, so a crossing inside a capped window would
    otherwise take about 10M elements; here the windows grow to the cap inside B's binade (from 2 blocks
    after B: 2 + 4 + ... + 512 blocks) and the next one holds the crossing."""
    x = np.asarray(x, dtype=np.float64)
    s_at = float(np.sum(x[:at]))
    top = 2.0 ** (math.ceil(math.log2(s_at)) + 1)  # B = top - s_at lies in [top / 2, top)
    return np.concatenate([[top - s_at], x])


def window_schedule(x, s0=0.0):
    """The windows net_seq_sum walks for x (network_kernels.cuh, seq_advance_kernel): a list of
    (t0, blocks, crossing) with `crossing` the index of the element that leaves the running sum's binade
    inside the window, or None.  A step that finds no crossing moves to the window's end and doubles the
    window (up to SEQ_MAX_BLOCKS); one that does continues behind the crossing element with twice the
    blocks it consumed."""
    x = np.asarray(x, dtype=np.float64)
    part = np.cumsum(np.concatenate([[s0], x]))              # part[t] = s before element t
    exp = np.frexp(part)[1]
    exp[part == 0] = -2000                                     # s == 0: every non-zero element leaves it
    cross = np.flatnonzero(exp[1:] != exp[:-1])              # element t changes the binade
    steps, t0, blocks, n = [], 0, 1, x.size
    while t0 < n:
        end = min(t0 + blocks * SEQ_BLOCK, n)
        k = np.searchsorted(cross, t0)
        if k < cross.size and cross[k] < end:
            i = int(cross[k])
            steps.append((t0, blocks, i))
            blocks = min(2 * ((i + 1 - t0) // SEQ_BLOCK + 1), SEQ_MAX_BLOCKS)
            t0 = i + 1
        else:
            steps.append((t0, blocks, None))
            blocks = min(2 * blocks, SEQ_MAX_BLOCKS)
            t0 = end
    return steps


def capped_crossings(x, s0=0.0):
    """Crossings that the replay meets inside a window of SEQ_MAX_BLOCKS blocks."""
    return [c for _, b, c in window_schedule(x, s0) if b == SEQ_MAX_BLOCKS and c is not None]
