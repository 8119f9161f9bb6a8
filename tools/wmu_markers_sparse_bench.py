"""Every cluster's Mann-Whitney markers from a sparse matrix: the CSC call (gficf_cuda_wmu_markers_csc) against the
dense call (gficf_cuda_wmu_markers) on the workload of tools/wmu_markers_bench.py (same generator and seed), with a
bitwise comparison of the two; then a scale case the dense call cannot take (its matrix would not fit), with a
64-gene slice checked against the dense call on that slice.  Times are CUDA events inside the library and host
clocks around calls that return with the result on the host; the kernel split comes from torch.profiler in a
pass of its own.
    python tools/wmu_markers_sparse_bench.py [out.json] [scale_genes scale_cells scale_density]
With --devices 1,2,4,8 it runs only the scale case, once per device count (gficf_cuda_wmu_markers_csc_devices;
1 is the single-device call), in rounds that alternate the order of the counts, and checks that every count gives
the bits of the single-device call:
    python tools/wmu_markers_sparse_bench.py --devices 1,2,4,8 [out.json] [scale_genes scale_cells scale_density]
"""
import json, os, resource, subprocess, sys, time
import numpy as np
import scipy.sparse as sp
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gficf_b200

DEVICES = None
if "--devices" in sys.argv:
    i = sys.argv.index("--devices")
    DEVICES = [int(v) for v in sys.argv[i + 1].split(",")]
    del sys.argv[i:i + 2]
out_json = sys.argv[1] if len(sys.argv) > 1 else None
S_GENES = int(sys.argv[2]) if len(sys.argv) > 2 else 20_000
S_CELLS = int(sys.argv[3]) if len(sys.argv) > 3 else 500_000
S_DENS = float(sys.argv[4]) if len(sys.argv) > 4 else 0.05
K = 20


def card():
    return subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                          text=True).stdout.strip().splitlines()


def labels(rng, n):
    """tools/wmu_markers_bench.py: unequal sizes (weights 1 .. 4), interleaved."""
    w = np.linspace(1.0, 4.0, K)
    cl = rng.choice(K, size=n, p=w / w.sum()).astype(np.int32)
    cl[rng.choice(n, size=K, replace=False)] = np.arange(K, dtype=np.int32)
    return cl


def timed(fn, reps=3):
    fn()  # warm-up (module load, workspace allocation)
    runs = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        dt = (time.perf_counter() - t0) * 1e3
        tm = gficf_b200.last_timings()
        runs.append({"call_ms": dt, "wall_ms": tm["wall_ms"], "h2d_ms": tm["h2d_ms"], "kernel_ms": tm["jaccard_ms"]})
    return out, runs, min(runs, key=lambda r: r["call_ms"])


def profile_kernels(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
    ms = {}
    for e in prof.events():
        if e.device_time > 0:
            name = e.name.split("(")[0].replace("void ", "").replace("gficf::", "")
            ms[name] = ms.get(name, 0.0) + e.device_time / 1e3
    return dict(sorted(ms.items(), key=lambda kv: -kv[1]))


def scale_matrix():
    """The scale case, generated column by column in CSC form (geometric gaps between stored rows), never dense.
    Generation peaks at about 30 bytes of host memory per stored value: fewer cells when the host lacks it."""
    global S_CELLS
    avail = int(open("/proc/meminfo").read().split("MemAvailable:")[1].split()[0]) * 1024
    while S_GENES * S_CELLS * S_DENS * 30 > 0.6 * avail:
        S_CELLS //= 2
    rng = np.random.default_rng(2)
    lib = rng.uniform(0.5, 2.0, size=S_CELLS)
    indptr = np.zeros(S_CELLS + 1, dtype=np.int64)
    rows_chunks, x_chunks = [], []
    chunk = 2000
    L = int(S_GENES * S_DENS + 8 * np.sqrt(S_GENES * S_DENS) + 64)
    for j0 in range(0, S_CELLS, chunk):
        j1 = min(S_CELLS, j0 + chunk)
        r = np.cumsum(rng.geometric(S_DENS, size=(j1 - j0, L)), axis=1) - 1
        keep = r < S_GENES
        cnt = keep.sum(axis=1)
        rr = r[keep].astype(np.int32)
        vals = (1 + rng.poisson(0.5, size=rr.size)) * (1e6 / 5000.0) / np.repeat(lib[j0:j1], cnt)
        rows_chunks.append(rr)
        x_chunks.append(vals)
        indptr[j0 + 1:j1 + 1] = cnt
    indptr = np.cumsum(indptr)
    rows = np.concatenate(rows_chunks)
    del rows_chunks
    x = np.concatenate(x_chunks)
    del x_chunks
    return sp.csc_matrix((x, rows, indptr.astype(np.int32)), shape=(S_GENES, S_CELLS)), labels(rng, S_CELLS)


def device_scaling(devices, rounds=3):
    """Every device count on the scale case, warmed up once each (workspaces, NCCL communicators), then `rounds`
    rounds in alternating order.  Phases from gficf_cuda_last_timings (maximum over the devices): upload,
    transpose, exchange, regroup + rank + means; the single-device call reports its transpose inside `kernels`."""
    vis = gficf_b200.lib().gficf_cuda_device_count()
    skipped = [d for d in devices if d > vis]
    devices = [d for d in devices if d <= vis]
    t_gen = time.perf_counter()
    big, cl = scale_matrix()
    t_gen = time.perf_counter() - t_gen
    run = lambda d: gficf_b200.rcpp_parallel_WMU_markers_sparse(big, cl, n_devices=d)  # noqa: E731
    ref = run(1)
    same = {}
    for d in devices:
        same[d] = bool(np.array_equal(run(d).view(np.int64), ref.view(np.int64)))
    calls = {d: [] for d in devices}
    for rep in range(rounds):
        for d in (devices if rep % 2 == 0 else devices[::-1]):
            t0 = time.perf_counter()
            out = run(d)
            dt = (time.perf_counter() - t0) * 1e3
            tm = gficf_b200.last_timings()
            same[d] = same[d] and bool(np.array_equal(out.view(np.int64), ref.view(np.int64)))
            calls[d].append({"call_ms": dt, "wall_ms": tm["wall_ms"], "h2d_ms": tm["h2d_ms"],
                             "transpose_ms": tm["layout_ms"], "exchange_ms": tm["allgather_ms"],
                             "kernels_ms": tm["jaccard_ms"],
                             "device_ms": tm["layout_ms"] + tm["allgather_ms"] + tm["jaccard_ms"]})
    best = {d: min(calls[d], key=lambda r: r["call_ms"]) for d in devices}
    return {"genes": S_GENES, "cells": S_CELLS, "clusters": K, "nnz": int(big.nnz),
            "density": big.nnz / (S_GENES * S_CELLS), "generation_s": t_gen, "visible_devices": vis,
            "skipped_devices": skipped, "calls": calls, "best": best,
            "speedup_call": {d: best[1]["call_ms"] / best[d]["call_ms"] for d in devices} if 1 in devices else None,
            "speedup_device": {d: best[1]["device_ms"] / best[d]["device_ms"] for d in devices} if 1 in devices else None,
            "bitwise_equal_to_one_device": same,
            "timing": "host clock around each call (call_ms); the library's CUDA events, the maximum over the devices "
                      "of each phase (device_ms = transpose + exchange + regroup/rank/means; for one device the "
                      "transpose is inside kernels_ms); best of the rounds by call_ms"}


res = {"card": card()}
if DEVICES:
    res["devices"] = device_scaling(DEVICES)
    print(json.dumps(res), flush=True)
    if out_json:
        os.makedirs(os.path.dirname(os.path.abspath(out_json)), exist_ok=True)
        with open(out_json, "w") as f:
            json.dump(res, f, indent=1)
    sys.exit(0)

# ---- r03 workload: 2000 x 100 000, 20 clusters (tools/wmu_markers_bench.py, seed 1)
genes, N = 2000, 100_000
rng = np.random.default_rng(1)
lib = rng.uniform(0.5, 2.0, size=N)
m = np.asfortranarray((rng.poisson(0.15, size=(genes, N)) * (1e6 / 5000.0) / lib[None, :]).astype(np.float64))
cl = labels(rng, N)
mat = sp.csc_matrix(m)  # built before the timed calls
nnz = int(mat.nnz)
dense_out, dense_runs, dense_best = timed(lambda: gficf_b200.rcpp_parallel_WMU_markers(m, cl))
sparse_out, sparse_runs, sparse_best = timed(lambda: gficf_b200.rcpp_parallel_WMU_markers_sparse(mat, cl))
res["r03"] = {
    "genes": genes, "cells": N, "clusters": K, "nnz": nnz, "density": nnz / (genes * N),
    "h2d_bytes_dense": genes * N * 8 + N * 4 + K * 8,
    "h2d_bytes_sparse": nnz * 12 + (N + 1) * 4 + 3 * N * 4 + K * 16 + 8,
    "dense_runs": dense_runs, "dense_best": dense_best, "sparse_runs": sparse_runs, "sparse_best": sparse_best,
    "speedup_call": dense_best["call_ms"] / sparse_best["call_ms"],
    "bitwise_equal_sparse_vs_dense": bool(np.array_equal(sparse_out.view(np.int64), dense_out.view(np.int64))),
    "profiler_kernel_ms_dense": profile_kernels(lambda: gficf_b200.rcpp_parallel_WMU_markers(m, cl)),
    "profiler_kernel_ms_sparse": profile_kernels(lambda: gficf_b200.rcpp_parallel_WMU_markers_sparse(mat, cl)),
}
del m, mat, dense_out, sparse_out
print(json.dumps(res["r03"]), flush=True)

# ---- scale case
import torch
t_gen = time.perf_counter()
big, cl = scale_matrix()
t_gen = time.perf_counter() - t_gen
assert gficf_b200.lib().gficf_cuda_release() == 0  # empty the workspace so that its growth below is the call's
free0, total = torch.cuda.mem_get_info()
calls = []
for _ in range(2):  # the first call allocates the workspace
    t0 = time.perf_counter()
    out = gficf_b200.rcpp_parallel_WMU_markers_sparse(big, cl)
    dt = (time.perf_counter() - t0) * 1e3
    tm = gficf_b200.last_timings()
    calls.append({"call_ms": dt, "wall_ms": tm["wall_ms"], "h2d_ms": tm["h2d_ms"], "kernel_ms": tm["jaccard_ms"]})
free1, _ = torch.cuda.mem_get_info()
sl = 64
want = gficf_b200.rcpp_parallel_WMU_markers(np.asfortranarray(big[:sl].toarray()), cl)
res["scale"] = {
    "genes": S_GENES, "cells": S_CELLS, "clusters": K, "nnz": int(big.nnz), "density": big.nnz / (S_GENES * S_CELLS),
    "dense_matrix_bytes": S_GENES * S_CELLS * 8, "csc_bytes": int(big.nnz) * 12 + (S_CELLS + 1) * 4,
    "generation_s": t_gen, "calls": calls,
    "device_bytes_held_after_call": free0 - free1,
    "device_total_bytes": total,
    "slice_genes_checked": sl,
    "slice_bitwise_equal_dense": bool(np.array_equal(out[:sl].view(np.int64), want.view(np.int64))),
    "host_max_rss_bytes": resource.getrusage(resource.RUSAGE_SELF).ru_maxrss * 1024,
    "profiler_kernel_ms": profile_kernels(lambda: gficf_b200.rcpp_parallel_WMU_markers_sparse(big, cl)),
}
res["timing"] = ("CUDA events inside the library (h2d_ms, kernel_ms; kernel_ms of the sparse call includes the "
                 "transpose and one synchronisation) and host clocks around calls that return with the result on the "
                 "host (call_ms); per-kernel times from torch.profiler in separate passes; device memory from "
                 "cudaMemGetInfo before the first and after the second scale call (the library's workspace only "
                 "grows, so this is its peak; other processes on the card would show up too)")
print(json.dumps(res["scale"]), flush=True)
if out_json:
    os.makedirs(os.path.dirname(os.path.abspath(out_json)), exist_ok=True)
    with open(out_json, "w") as f:
        json.dump(res, f, indent=1)
