"""GPU (-m gpu), needs >= 2 devices (skipped on a 1-GPU box; run with `gpurun --gpus 2`):
row sharding inside ONE process through the C ABI (n_devices = 2, 4, ...: NCCL all-gather of the
index slabs, every GPU returns its own edge slab) and one process per GPU over torch.distributed
(gficf_b200.sharding)."""
import os
import subprocess
import sys

import numpy as np
import pytest

from gficf_b200 import synth
from tests.conftest import random_knn

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ndev(cuda):
    return cuda.lib().gficf_cuda_device_count()


@pytest.mark.parametrize("n,k", [(100_000, 30), (10_001, 15), (3_000, 100), (7, 3)])
def test_in_process_row_sharding(cuda, oracle, n, k):
    nd = _ndev(cuda)
    if nd < 2:
        pytest.skip("needs >= 2 GPUs")
    r = synth.to_r_matrix(synth.knn_index(n, k, scramble=True)) if n > k + 1 else \
        random_knn(np.random.default_rng(0), n, k, with_self=True)
    want = oracle.parallel(r)
    for d in sorted({2, nd}):
        got = cuda.rcpp_parallel_jaccard_coef(r, False, d)
        assert np.array_equal(got, want), "n_devices=%d" % d
    # repeated ids on a slab other than the first: the exact path must run on every device
    r2 = r.copy()
    r2[n - 1, 0] = r2[n - 1, k - 1]
    assert np.array_equal(cuda.rcpp_parallel_jaccard_coef(r2, False, 2), oracle.parallel(r2))
    # invalid id on the last slab
    r3 = r.copy()
    r3[n - 1, 0] = n + 5
    with pytest.raises(cuda.GficfCudaError):
        cuda.rcpp_parallel_jaccard_coef(r3, False, 2)


def test_set_devices_default(cuda, oracle):
    if _ndev(cuda) < 2:
        pytest.skip("needs >= 2 GPUs")
    r = synth.to_r_matrix(synth.knn_index(50_000, 30))
    cuda.set_devices(2)
    try:
        got = cuda.rcpp_parallel_jaccard_coef(r)  # n_devices=0 -> the configured default
    finally:
        cuda.set_devices(1)
    assert np.array_equal(got, oracle.parallel(r))


def test_single_device_calls_leave_the_callers_device_current(cuda):
    """The host-buffer graph-build and Mann-Whitney calls run on device 0; the caller's current device is
    current again when they return, also when they fail (a malformed row id is found on the device)."""
    if _ndev(cuda) < 2:
        pytest.skip("needs >= 2 GPUs")
    import scipy.sparse as sp
    import torch

    from gficf_b200 import snn
    from tests.test_wmu_markers_sparse_emu import malformed_cases

    torch.cuda.set_device(1)
    try:
        _, colptr, row = malformed_cases()[1]
        bad = sp.csc_matrix((5, 4))
        bad.indptr, bad.indices, bad.data = colptr, row, np.arange(1.0, row.size + 1.0)
        with pytest.raises(cuda.GficfCudaError) as e:
            cuda.rcpp_parallel_WMU_markers_sparse(bad, np.array([0, 1, 0, 1], dtype=np.int32))
        assert e.value.code == 1 and "row id" in e.value.message
        assert torch.cuda.current_device() == 1
        rng = np.random.default_rng(5)
        m = np.asfortranarray(np.floor(rng.gamma(1.0, 2.0, size=(20, 300))))
        cl = (np.arange(300) % 4).astype(np.int32)
        calls = (lambda: cuda.rcpp_parallel_WMU_test(m[:, :100], m[:, 100:]),
                 lambda: cuda.rcpp_parallel_WMU_markers(m, cl),
                 lambda: cuda.rcpp_parallel_WMU_markers_sparse(sp.csc_matrix(m), cl),
                 lambda: snn.snn_graph(synth.to_r_matrix(synth.knn_index(3_000, 10, scramble=True))))
        for i, call in enumerate(calls):
            call()
            assert torch.cuda.current_device() == 1, i
    finally:
        torch.cuda.set_device(0)


_WORKER = r"""
import os, sys, numpy as np, torch, torch.distributed as dist
sys.path.insert(0, %(root)r)
import gficf_b200
from gficf_b200 import sharding, synth
from oracle.binding import Oracle
rank = int(os.environ["RANK"]); local = int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
for n, k, dup in ((200_000, 30, False), (10_001, 15, False), (5_000, 100, False), (20_000, 30, True)):
    r = None
    if rank == 0:
        r = synth.to_r_matrix(synth.knn_index(n, k, scramble=True))
        if dup:
            r[n - 1, 0] = r[n - 1, k - 1]
    out = sharding.rcpp_parallel_jaccard_coef_sharded(r, n, k)
    if rank == 0:
        want = Oracle().parallel(r)
        assert np.array_equal(out, want), (n, k)
    else:
        assert out is None
# pipelined gather: uneven split, chunked u8 sends, expand on the host rank
from gficf_b200 import device as D
for n, k, rho in ((300_000, 30, 0.19), (50_001, 15, 0.6), (20_000, 100, 0.0), (7, 3, 0.2)):
    idx0 = synth.knn_index(n, k, scramble=True, device="cuda")
    padded, fl = D.pad_rows(idx0)
    pg = sharding.PipelinedGather(n, k, rho=rho, chunks=4)
    counts = torch.empty(n * k, dtype=torch.uint8, device="cuda")
    out3 = torch.full((3, n * k), -1.0, dtype=torch.float64, device="cuda") if rank == 0 else None
    pg.step(padded, counts, out3)
    pg.step(padded, counts, out3)
    torch.cuda.synchronize()
    if rank == 0:
        ref, _ = D.jaccard_edges(padded, n, k)
        assert torch.equal(out3, ref), (n, k)
        assert int(pg.flags[0]) == 0
    dist.barrier()
    # the gather fused into the count kernel (parity-tagged peer stores over NVLink), streaming expand
    for share, host in ((None, 0), (0.0, 0), (0.37, 0), (0.2, dist.get_world_size() - 1)):
        peer = sharding.PeerGather(n, k, host_share=share, host_rank=host, timeout_ms=5000)
        o3 = torch.full((3, n * k), -1.0, dtype=torch.float64, device="cuda") if rank == host else None
        for it in range(3):  # odd and even epochs on the same buffer
            peer.step(padded, o3)
        assert peer.finish(padded, o3) == 0
        if rank == host:
            ref1, _ = D.jaccard_edges(padded, n, k)
            assert torch.equal(o3, ref1), ("peer", n, k, share, host)
        peer.close()
# the peer-store split: peers store finished doubles of their last rows straight into the host rank's output
for n, k, ds, host in ((300_000, 30, 0.25, 0), (50_001, 15, 0.5, dist.get_world_size() - 1), (40_000, 7, 0.1, 0)):
    idx0 = synth.knn_index(n, k, scramble=True, device="cuda")
    padded, fl = D.pad_rows(idx0)
    peer = sharding.PeerGather(n, k, host_share=0.1, host_rank=host, timeout_ms=5000, direct_share=ds)
    assert (peer.out3 is not None) == (rank == host)
    if rank == host:
        peer.out3.fill_(-1.0)
    torch.cuda.synchronize(); dist.barrier()
    for it in range(3):
        peer.step(padded)
    assert peer.finish(padded) == 0
    if rank == host:
        ref1, _ = D.jaccard_edges(padded, n, k)
        assert torch.equal(peer.out3, ref1), ("peer-store split", n, k, ds, host)
    peer.close()
# streaming peer gather: a repeated id anywhere -> finish() reruns the exact path on the host rank
n, k = 40_000, 30
idx0 = synth.knn_index(n, k, scramble=True, device="cuda")
idx0[n - 3, 0] = idx0[n - 3, k - 1]
padded, fl = D.pad_rows(idx0)
peer = sharding.PeerGather(n, k, timeout_ms=5000)
o3 = torch.full((3, n * k), -1.0, dtype=torch.float64, device="cuda") if rank == 0 else None
peer.step(padded, o3)
assert peer.finish(padded, o3) & (D.FLAG_DUP_ID | D.FLAG_HASH_FAIL)
if rank == 0:
    assert np.array_equal(o3.cpu().numpy().T, Oracle().parallel(synth.to_r_matrix(idx0)))
peer.close()
# configs[4]'s shape (k = 100) at 1M cells over all ranks: whole matrix against the single-GPU fused
# kernel, and the oracle on head / middle / tail rows
n, k = 1_000_000, 100
idx0 = synth.knn_index(n, k, scramble=True, device="cuda")
padded, fl = D.pad_rows(idx0)
peer = sharding.PeerGather(n, k, timeout_ms=5000)
o3 = torch.empty((3, n * k), dtype=torch.float64, device="cuda") if rank == 0 else None
for it in range(2):
    peer.step(padded, o3)
assert peer.finish(padded, o3) == 0
if rank == 0:
    ref1, _ = D.jaccard_edges(padded, n, k)
    assert torch.equal(o3, ref1), "k=100 1M cells"
    del ref1
    r = synth.to_r_matrix(idx0)
    orc = Oracle()
    for lo, hi in ((0, 300), (n // 2, n // 2 + 300), (n - 300, n)):
        assert np.array_equal(o3[:, lo * k:hi * k].cpu().numpy().T, orc.parallel_rows(r, lo, hi)), (lo, hi)
    del r
peer.close()
del o3, padded, idx0
torch.cuda.empty_cache()
# the step after the path, row-sharded: per-rank counts with the mutual bit, all-gather, graph build on the host rank
from gficf_b200 import snn
for n, k, fam in ((120_000, 30, "planted"), (9_000, 6, "uniform")):
    idx0 = synth.knn_index(n, k, family=fam, scramble=True, device="cuda")
    padded, fl = D.pad_rows(idx0)
    res = snn.snn_lower_triangle_sharded(padded, n, k)
    if rank == 0:
        one = snn.snn_lower_triangle(padded, n, k, with_vertex_map=True)
        for a_, b_ in zip(res[:4], one[:4]):
            assert torch.equal(a_, b_), ("snn sharded", n, k)
        assert int(res[4][0]) & ~16 == 0
    else:
        assert res is None
    dist.barrier()
# the library's own one-rank-per-GPU entry on shared page-locked host matrices
from gficf_b200 import multiproc
multiproc.comm_init_from_torch()
for n, k, dup, bad in ((150_000, 30, False, False), (4_001, 100, False, False), (30_000, 30, True, False), (30_000, 15, False, True)):
    tag = "gficf_test_%%d_%%d_%%d" %% (os.getppid(), n, k)
    r_sh = out_sh = None
    if rank == 0:
        r_sh = multiproc.SharedHostMatrix(tag + "_idx", (n, k), create=True)
        out_sh = multiproc.SharedHostMatrix(tag + "_out", (n * k, 3), create=True)
        r_sh.array[...] = synth.to_r_matrix(synth.knn_index(n, k, scramble=True))
        if dup:
            r_sh.array[n - 1, 0] = r_sh.array[n - 1, k - 1]
        if bad:
            r_sh.array[n - 1, 0] = 0
        out_sh.array[...] = -1.0
    dist.barrier()
    if rank != 0:
        r_sh = multiproc.SharedHostMatrix(tag + "_idx", (n, k), create=False)
        out_sh = multiproc.SharedHostMatrix(tag + "_out", (n * k, 3), create=False)
    assert r_sh.pinned and out_sh.pinned
    try:
        multiproc.rcpp_parallel_jaccard_coef_rank(r_sh.array, out_sh.array)
        assert not bad
    except gficf_b200.GficfCudaError as e:
        assert bad and e.code == 2, e      # every rank reports the bad id, whoever owns the row
    dist.barrier()
    if rank == 0 and not bad:
        assert np.array_equal(out_sh.array, Oracle().parallel(np.asfortranarray(r_sh.array))), (n, k)
    dist.barrier()
    r_sh.close(); out_sh.close()
multiproc.comm_destroy()
dist.barrier()
if rank == 0:
    print("SHARDED_OK")
dist.destroy_process_group()
"""


def test_one_process_per_gpu_nccl(cuda, tmp_path):
    nd = _ndev(cuda)
    if nd < 2:
        pytest.skip("needs >= 2 GPUs")
    script = tmp_path / "worker.py"
    script.write_text(_WORKER % {"root": ROOT})
    out = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", str(min(nd, 8)),
                          "--master-addr", "127.0.0.1", "--master-port", "29533", str(script)],
                         capture_output=True, text=True, timeout=1500)
    log = os.path.join(ROOT, "gpurun_out")
    if os.path.isdir(log):
        with open(os.path.join(log, "worker_multi.log"), "w") as f:
            f.write(out.stdout + "\n==== stderr ====\n" + out.stderr)
    err_lines = [ln for ln in out.stderr.splitlines() if "Error" in ln or "assert" in ln.lower()]
    assert out.returncode == 0, "\n".join(err_lines[-30:]) + out.stderr[-1500:]
    assert "SHARDED_OK" in out.stdout
