"""Every cluster's one-vs-rest Mann-Whitney test: the batched call (gficf_cuda_wmu_markers) against the loop of
per-cluster rcpp_parallel_WMU_test calls that findClusterMarkers (R/deGenes.R:44-54) makes today, on the same
seeded matrix, with a bitwise comparison of the two and of both against the oracle / the reference's own
sources on a gene subset.  Times are CUDA events inside the library and host clocks around calls that return
with the result on the host.
    python tools/wmu_markers_bench.py [genes] [cells] [clusters] [out.json]
"""
import json, os, subprocess, sys, time
import numpy as np
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gficf_b200
from oracle.binding import WmuOracle, WmuReference

genes = int(sys.argv[1]) if len(sys.argv) > 1 else 2000
N = int(sys.argv[2]) if len(sys.argv) > 2 else 100_000
K = int(sys.argv[3]) if len(sys.argv) > 3 else 20
out_json = sys.argv[4] if len(sys.argv) > 4 else None
rng = np.random.default_rng(1)
# CPM-like as in tools/wmu_bench.py: ~14 % non-zero, library-size scaled, one giant zero tie group per gene
lib = rng.uniform(0.5, 2.0, size=N)
m = np.asfortranarray((rng.poisson(0.15, size=(genes, N)) * (1e6 / 5000.0) / lib[None, :]).astype(np.float64))
# unequal cluster sizes (weights 1 .. 4), labels at random positions so that the clusters interleave
w = np.linspace(1.0, 4.0, K)
cl = rng.choice(K, size=N, p=w / w.sum()).astype(np.int32)
cl[rng.choice(N, size=K, replace=False)] = np.arange(K, dtype=np.int32)
sizes = np.bincount(cl, minlength=K)

card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                      text=True).stdout.strip().splitlines()

reps = 3
gficf_b200.rcpp_parallel_WMU_markers(m, cl)  # warm-up (module load, workspace allocation)
batched = []
for _ in range(reps):
    t0 = time.perf_counter()
    got = gficf_b200.rcpp_parallel_WMU_markers(m, cl)
    dt = (time.perf_counter() - t0) * 1e3
    tm = gficf_b200.last_timings()
    batched.append({"call_ms": dt, "wall_ms": tm["wall_ms"], "h2d_ms": tm["h2d_ms"], "kernel_ms": tm["jaccard_ms"]})

# today's path: one call per cluster on its two submatrices, sliced before the timed call
loop_ms, loop_h2d, loop_kernel = [], [], []
want = np.empty_like(got)
for rep in range(2):
    tot = h2d = ker = 0.0
    for c in range(K):
        x, y = np.asfortranarray(m[:, cl == c]), np.asfortranarray(m[:, cl != c])
        if rep == 0 and c == 0:
            gficf_b200.rcpp_parallel_WMU_test(x, y)  # warm-up
        t0 = time.perf_counter()
        want[:, :, c] = gficf_b200.rcpp_parallel_WMU_test(x, y)
        tot += (time.perf_counter() - t0) * 1e3
        tm = gficf_b200.last_timings()
        h2d += tm["h2d_ms"]
        ker += tm["jaccard_ms"]
        del x, y
    loop_ms.append(tot); loop_h2d.append(h2d); loop_kernel.append(ker)
bitwise = bool(np.array_equal(got.view(np.int64), want.view(np.int64)))

sub = min(genes, 64)
ref = WmuReference() if WmuReference.available() else None
kind = "reference sources" if ref is not None else "oracle port"
ok_sub = True
for c in range(K):
    x, y = np.asfortranarray(m[:sub, cl == c]), np.asfortranarray(m[:sub, cl != c])
    r = ref.wmu(x, y) if ref is not None else WmuOracle().wmu(x, y)
    ok_sub &= bool(np.array_equal(got[:sub, :, c], r, equal_nan=True))

# kernel split of one batched call, in a run of its own (tracing slows the host)
import torch
from torch.profiler import ProfilerActivity, profile
with profile(activities=[ProfilerActivity.CUDA]) as prof:
    gficf_b200.rcpp_parallel_WMU_markers(m, cl)
kernel_ms = {}
for e in prof.events():
    if "wmu" in e.name:
        kernel_ms[e.name] = kernel_ms.get(e.name, 0.0) + e.device_time / 1e3

best = min(batched, key=lambda r: r["call_ms"])
res = {
    "card": card, "genes": genes, "cells": N, "clusters": K, "cluster_sizes": sizes.tolist(),
    "batched": batched, "batched_best": best, "profiler_kernel_ms": kernel_ms,
    "loop_call_ms": loop_ms, "loop_h2d_ms": loop_h2d, "loop_kernel_ms": loop_kernel,
    "speedup_call": min(loop_ms) / best["call_ms"],
    "bitwise_equal_batched_vs_loop": bitwise, "checked_genes": sub, "checked_against": kind, "equal_on_subset": ok_sub,
    "h2d_bytes_batched": genes * N * 8 + N * 4 + K * 8, "h2d_bytes_loop": K * genes * N * 8,
    "means_fp64_adds": genes * N * K + genes * N * -(-K // 8),  # chain adds + the staged v + 1 per cluster block
    "timing": "CUDA events inside the library (h2d_ms, kernel_ms) and host clocks around calls that return with "
              "the result on the host (call_ms); ncu / nsys were not used",
}
print(json.dumps(res))
print("| genes x cells, clusters | batched call ms | H2D ms | kernels ms | loop of %d calls ms | loop H2D ms | loop kernels ms "
      "| speed-up | bitwise equal | == %s (%d genes) |" % (K, kind, sub))
print("|---|---|---|---|---|---|---|---|---|---|")
print("| %d x %d, %d | %.1f | %.1f | %.1f | %.1f | %.1f | %.1f | %.1fx | %s | %s |" % (
    genes, N, K, best["call_ms"], best["h2d_ms"], best["kernel_ms"], min(loop_ms), loop_h2d[int(np.argmin(loop_ms))],
    loop_kernel[int(np.argmin(loop_ms))], res["speedup_call"], bitwise, ok_sub))
if out_json:
    os.makedirs(os.path.dirname(os.path.abspath(out_json)), exist_ok=True)
    with open(out_json, "w") as f:
        json.dump(res, f, indent=1)
