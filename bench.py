#!/usr/bin/env python
"""bench.py -- Jaccard edges/s of the Phenograph graph-weighting path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Workload (BASELINE.json `metric`: "Jaccard edges/s at 4M cells k=30"): a synthetic 4M x 30
planted-cluster kNN index with scrambled cell ids (gficf_b200.synth), E = 1.2e8 edge slots.
A step is one pass of the hot path over the whole matrix.

  value     whole-job edges/s with the padded int32 index resident in HBM on every GPU;
            N=1: one launch of the fused kernel; N>1: rows sharded over the ranks (strong
            scaling: the 4M cells are fixed), ONE count launch per rank whose epilogue stores the
            parity-tagged 1-byte counts into the host rank's HBM over NVLink, ONE streaming expand
            launch on the host rank (gficf_b200.sharding.PeerGather)
  e2e       the same metric through the reference-facing call with HOST buffers (pinned): the f64
            R matrix narrowed to int32 on its way to the device, layout pre-pass, count kernel, and
            the (E x 3) doubles written by host threads from the 1-byte counts and by the copy
            engine at once (include/gficf_cuda.h, gficf_cuda_last_output); bytes as actually moved
  parity    rank 0: value path and e2e result against the reference's own sources (oracle/_ref) on
            head / middle / tail rows; at N>1 the whole matrix against the single-GPU fused kernel
  roofline  the fused/count kernel against MEASURED_PEAKS.json hbm_gbs, algorithmic bytes
            (4k+28) per edge (SURVEY.md 8d); traffic = DRAM bytes of one launch, measured by an ncu
            child process in the same run
  cpu_baseline / cpu_baseline_nt2  the reference's own sources (oracle/_ref, unmodified, R runtime
            stubbed) on a bounded row sample with all host threads / with nt = 2 (clustcells default)

`--impl reference` times only that CPU implementation (rank 0).
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "jaccard_edges_per_s"
UNIT = "edges/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--cells", type=int, default=4_000_000)
    ap.add_argument("--k", type=int, default=30)
    ap.add_argument("--family", default="planted", choices=["planted", "uniform"])
    ap.add_argument("--no-scramble", action="store_true")
    ap.add_argument("--seed", type=int, default=180582)
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = min(steps, 10)")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="CPU baseline sample budget")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--chunks", type=int, default=4, help="N>1, --gather nccl: row chunks of the pipelined gather")
    ap.add_argument("--gather", default="peer", choices=["peer", "nccl"],
                    help="N>1: how the counts reach the host rank (streaming peer stores / NCCL send-recv)")
    ap.add_argument("--config", default="cfg4", choices=["cfg1", "cfg2", "cfg3", "cfg4", "cfg5"],
                    help="BASELINE.json configs[i-1]; cfg4 (4M x 30) is the one the metric is quoted on")
    ap.add_argument("--host-share", type=float, default=-1.0, help="N>1: host rank's row share (default: calibrated)")
    ap.add_argument("--direct-share", type=float, default=-1.0,
                    help="N>1: share of a peer's rows whose finished doubles the peer stores itself into rank 0's "
                         "output (default: GFICF_CUDA_PEER_DIRECT or the built-in choice)")
    ap.add_argument("--no-traffic-probe", action="store_true", help="do not re-run the kernel under ncu for roofline.traffic")
    ap.add_argument("--traffic-probe", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--no-parity", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last step computed as DIR/<name>.npy (see dump_outputs)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl ours)")
    shapes = {"cfg1": (10_000, 15), "cfg2": (100_000, 30), "cfg3": (1_000_000, 30), "cfg4": (4_000_000, 30),
              "cfg5": (10_000_000, 100)}
    if a.config != "cfg4":
        a.cells, a.k = shapes[a.config]
    return a


def workload_name(a):
    return "%dM cells k=%d %s%s kNN index (E=%.3g edge slots)" % (
        a.cells // 1_000_000, a.k, a.family, "" if a.no_scramble else " scrambled-ids", a.cells * a.k) \
        if a.cells % 1_000_000 == 0 else "%d cells k=%d %s%s" % (a.cells, a.k, a.family,
                                                                 "" if a.no_scramble else " scrambled-ids")


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler:
    """SM clock + throttle reasons of one GPU sampled with NVML during the timed region."""

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self.nv = None

    def sample_once(self):
        """One synchronous sample (NVML calls can take tens of ms: the thread alone may see few)."""
        if self.nv is None:
            return
        try:
            self.samples.append(int(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM)))
        except Exception:
            pass

    def _loop(self):
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksThrottleReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksThrottleReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksThrottleReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake_slowdown",
        }
        while not self._stop.is_set():
            try:
                self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
                for bit, nm in names.items():
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.01)

    def start(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()

    def stop(self):
        self.sample_once()  # right behind the last timed kernel
        if self._t is not None:
            self._stop.set()
            self._t.join()
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz,
                "reasons": sorted(self.reasons), "samples": len(s)}


# --------------------------------------------------------------------------- CPU reference
def reference_sampler(r_matrix, k, budget_s, nthreads=0):
    """Times the reference's unmodified JCoefficient worker (oracle/_ref) on rows [0,m) gathering
    from the full matrix; m calibrated so one sample costs about budget_s seconds."""
    from oracle.binding import Oracle, Reference

    if Reference.available():
        ref, kind = Reference(), "reference"
        cores = ref.hw_threads() if nthreads == 0 else nthreads

        def run(lo, hi):
            ref.parallel_rows(r_matrix, lo, hi, nthreads=nthreads)
            return ref.last_seconds
    else:
        orc, kind = Oracle(), "port"
        cores = os.cpu_count() or 1

        def run(lo, hi):
            t0 = time.perf_counter()
            orc.parallel_rows(r_matrix, lo, hi, nthreads=cores)
            return time.perf_counter() - t0

    n = r_matrix.shape[0]
    probe = min(n, 4096 * max(1, cores // 4))
    t = run(0, probe)
    rate = probe / max(t, 1e-6)
    m = int(max(probe, min(n, rate * budget_s)))
    return run, m, kind, cores


def run_reference_arm(a):
    import numpy as np
    import torch

    from gficf_b200 import synth

    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    idx0 = synth.knn_index(a.cells, a.k, family=a.family, seed=a.seed, scramble=not a.no_scramble,
                           device="cuda" if torch.cuda.is_available() else "cpu")
    r = synth.to_r_matrix(idx0)
    del idx0
    per_step = max(0.5, min(10.0, 150.0 / max(1, a.steps + a.warmup)))
    run, m, kind, cores = reference_sampler(r, a.k, per_step)
    for _ in range(a.warmup):
        run(0, m)
    times = [run(0, m) for _ in range(a.steps)]
    tot = float(np.sum(times))
    val = m * a.k * a.steps / tot
    sample = "rows [0,%d) of %d (%.3g edges/step) gathering from the full matrix" % (m, a.cells, m * a.k)
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
        "warmup": a.warmup, "ms_per_step": 1e3 * tot / a.steps, "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(a), "sample": sample},
        "cpu_baseline": {"value": val, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }))


def checker():
    """The CPU checker for parity records: oracle/_ref (the reference's own sources) when it was
    built in the container, else the C restatement."""
    from oracle.binding import Oracle, Reference

    if Reference.available():
        return Reference(), "reference"
    return Oracle(), "port"


def parity_ranges(n, rows=2000):
    """Head, middle and tail row ranges (>= 2000 rows each when the matrix has them)."""
    rows = min(rows, n)
    mid = max(0, min(n - rows, n // 2 - rows // 2))
    out = []
    for lo in (0, mid, n - rows):
        if (lo, lo + rows) not in out:
            out.append((lo, lo + rows))
    return out


def rows_equal(chk, r_matrix, k, ranges, getter):
    """getter(lo, hi) -> ((hi-lo)*k, 3) numpy block of a result; compared with the checker bit for bit."""
    import numpy as np

    ok = True
    for lo, hi in ranges:
        want = chk.parallel_rows(r_matrix, lo, hi)
        ok = ok and bool(np.array_equal(getter(lo, hi), want))
    return ok


def probe_traffic(a):
    """roofline.traffic measured in THIS run: the fused kernel of this workload once more under
    `ncu --metrics dram__bytes_read.sum,dram__bytes_write.sum` in a child process (never the timed
    process).  Returns (bytes per launch, source) or (None, why)."""
    import shutil
    import subprocess

    ncu = shutil.which("ncu") or "/usr/local/cuda/bin/ncu"
    if not os.path.exists(ncu):
        return None, "ncu not found"
    cmd = [ncu, "--metrics", "dram__bytes_read.sum,dram__bytes_write.sum", "--clock-control", "none",
           "--profile-from-start", "off", "-k", "regex:jaccard_(small|wide|large)_k", "-c", "1", "--csv",
           sys.executable, os.path.abspath(__file__), "--traffic-probe", "--cells", str(a.cells), "--k", str(a.k),
           "--family", a.family, "--seed", str(a.seed)] + (["--no-scramble"] if a.no_scramble else [])
    try:
        env = dict(os.environ)
        for v in ("RANK", "LOCAL_RANK", "WORLD_SIZE"):
            env.pop(v, None)
        r = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=env)
        tot = 0.0
        seen = 0
        for ln in r.stdout.splitlines():
            if "dram__bytes_" in ln:
                f = [x.strip('"') for x in ln.split('","')]
                unit, val = f[-2], float(f[-1].replace(",", ""))
                tot += val * {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}.get(unit, 1.0)
                seen += 1
        if seen >= 2:
            return tot, "ncu dram__bytes_read.sum+dram__bytes_write.sum, one launch, captured in this run"
        return None, "ncu gave no counters (rc %d): %s" % (r.returncode, (r.stdout + r.stderr)[-200:].replace("\n", " "))
    except Exception as ex:
        return None, "ncu probe failed: %s" % str(ex)[:120]


def run_traffic_probe(a):
    """Child of probe_traffic(): builds the workload and launches the fused kernel three times."""
    import torch

    from gficf_b200 import device as D
    from gficf_b200 import synth

    dev = torch.device("cuda", 0)
    idx0 = synth.knn_index(a.cells, a.k, family=a.family, seed=a.seed, scramble=not a.no_scramble, device=dev)
    padded, flags = D.pad_rows(idx0)
    del idx0
    out = torch.empty((3, a.cells * a.k), dtype=torch.float64, device=dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    torch.cuda.synchronize()
    torch.cuda.profiler.start()
    for i in range(3):
        flush.fill_(i)
        D.jaccard_edges(padded, a.cells, a.k, out=out, flags=flags)
    torch.cuda.synchronize()
    torch.cuda.profiler.stop()


# --------------------------------------------------------------------------- GPU arm
DUMP_EDGE_COLUMNS = 1_500_000  # 36 MB of edges + 12 MB of their positions: a dump stays under 64 MB


def dump_outputs(path, out, flags):
    """--dump-outputs: what the timed path returned in its last step, as .npy files under `path`, so
    that two builds of the project can be compared output for output on the same seeded input.
      edges.npy         float64 (3, m): the from / to / weight rows of the (3, E) result; all E columns
                        when E <= DUMP_EDGE_COLUMNS, else a sample of DUMP_EDGE_COLUMNS columns drawn
                        with a fixed seed (the same columns in every run with the same E)
      edge_columns.npy  float64 (m,): the column of the result each edges.npy column is
      flags.npy         float64: the flag words the path sets (0 = no repeated or invalid ids)"""
    import numpy as np
    import torch

    os.makedirs(path, exist_ok=True)
    E = out.shape[1]
    if E <= DUMP_EDGE_COLUMNS:
        cols = np.arange(E, dtype=np.int64)
    else:
        cols = np.sort(np.random.default_rng(20261020).choice(E, DUMP_EDGE_COLUMNS, replace=False))
    edges = out[:, torch.from_numpy(cols).to(out.device)].cpu().numpy().astype(np.float64)
    np.save(os.path.join(path, "edges.npy"), edges)
    np.save(os.path.join(path, "edge_columns.npy"), cols.astype(np.float64))
    np.save(os.path.join(path, "flags.npy"), flags.cpu().numpy().astype(np.float64))


def network_record(colptr, srows, sw, n, k, a, dev, flush):
    """The bulk steps of the community detection on the device-resident graph (SURVEY 8f row 3): CSR
    network, quality function, reduced network -- timed once each and, unless --no-parity, checked bit
    for bit against the oracle (oracle/modopt_oracle.c, single-threaded like the reference)."""
    import numpy as np
    import torch

    from gficf_b200 import modularity, synth

    def once(fn):
        flush.fill_(7)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        res_ = fn()
        e1.record()
        torch.cuda.synchronize()
        return res_, e0.elapsed_time(e1)

    modularity.matrix_to_network(colptr, srows, sw)  # warm-up (allocator)
    net, t_net = once(lambda: modularity.matrix_to_network(colptr, srows, sw))
    nv = net.n_nodes
    if nv == n and a.family == "planted":  # the planted communities (what a Louvain run converges towards)
        cl = synth.planted_community(n, k, seed=a.seed, scramble=not a.no_scramble, device=dev).contiguous()
        cl_what = "the planted communities"
    else:
        cl = (torch.arange(nv, device=dev, dtype=torch.int32) // 200).contiguous()
        cl_what = "blocks of 200 vertices"
    nc = int(cl.max()) + 1
    res2 = 0.8 / (2 * net.get_total_edge_weight())  # resolution2 of RModularityOptimizer.cpp:101
    q, t_q = once(lambda: net.calc_quality_function(cl, res2, n_clusters=nc))
    red, t_red = once(lambda: net.create_reduced_network(cl, n_clusters=nc))
    rec = {"network_ms": t_net, "quality_ms": t_q, "reduce_ms": t_red, "vertices": nv,
           "directed_edges": net.n_edges, "clusters": nc, "reduced_edges": red.n_edges, "quality": q,
           "what": "matrixToNetwork / calcQualityFunction / createReducedNetwork "
                   "(src/ModularityOptimizer.cpp:761-806, :462-482, :322-373) on the device-resident graph, "
                   "clustering = " + cl_what + "; the local moving loop itself stays on the host"}
    if not a.no_parity:
        from oracle.binding import NetworkOracle

        orc = NetworkOracle()
        cols = np.repeat(np.arange(nv, dtype=np.int32), np.diff(colptr.cpu().numpy()))
        t0 = time.perf_counter()
        want = orc.network(cols, srows.cpu().numpy(), sw.cpu().numpy())
        t1 = time.perf_counter()
        cl_h = cl.cpu().numpy()
        q_want, _ = orc.quality(want, cl_h, res2)
        t2 = time.perf_counter()
        red_want = orc.reduce(want, cl_h)
        t3 = time.perf_counter()
        rec["cpu_ms"] = {"network": (t1 - t0) * 1e3, "quality": (t2 - t1) * 1e3, "reduce": (t3 - t2) * 1e3,
                         "cores": 1, "kind": "port"}

        def same(x, d):
            return bool(np.array_equal(x.first_neighbor_index.cpu().numpy(), d["first"]) and
                        np.array_equal(x.neighbor.cpu().numpy(), d["neighbor"]) and
                        np.array_equal(x.edge_weight.cpu().numpy(), d["edge_w"]) and
                        np.array_equal(x.node_weight.cpu().numpy(), d["node_w"]))

        rec["parity"] = {"network_arrays_equal": same(net, want),
                         "total_edge_weight_equal": bool(net.get_total_edge_weight() == want["total_w"]),
                         "quality_equal": bool(q == q_want),
                         "reduced_arrays_equal": same(red, red_want),
                         "self_links_equal": bool(red.total_edge_weight_self_links == red_want["self_links"])}
    del net, red
    torch.cuda.empty_cache()
    return rec


def run_ours(a):
    import numpy as np
    import torch
    import torch.distributed as dist

    import gficf_b200
    from gficf_b200 import device as D
    from gficf_b200 import sharding, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        os.environ.setdefault("TORCH_NCCL_HIGH_PRIORITY", "1")
        dist.init_process_group("nccl", device_id=dev)
    gficf_b200.lib()  # fail loudly now if the extension is missing

    n, k = a.cells, a.k
    E = n * k
    bytes_per_edge = 4 * k + 28
    hbm_peak, peak_src = peaks()
    warm = max(3, a.warmup)

    # ---- inputs: every rank generates the same matrix (counter-based generator)
    idx0 = synth.knn_index(n, k, family=a.family, seed=a.seed, scramble=not a.no_scramble, device=dev)
    padded, flags = D.pad_rows(idx0)
    torch.cuda.synchronize()
    assert int(flags[0]) == 0
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def event_ms(fn, reps=5, warmups=2):
        for _ in range(warmups):
            fn()
        ts = []
        for i in range(reps):
            flush.fill_(i)
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        return sum(ts) / len(ts)

    sharding_note = "none"
    pg = None
    if world == 1:
        out = torch.empty((3, E), dtype=torch.float64, device=dev)
        lo, hi = 0, n

        def step():
            D.jaccard_edges(padded, n, k, out=out, flags=flags)
    else:
        out = torch.empty((3, E), dtype=torch.float64, device=dev) if rank == 0 else None
        # calibrate the uneven row split on this GPU: per-row cost of the fused kernel (host rank's own
        # rows), the count kernel (peers' rows) and the expand kernel (host rank, every peer row)
        m = min(n, 1_000_000)
        cal_c = torch.empty(m * k, dtype=torch.uint8, device=dev)
        cal_o = torch.empty((3, m * k), dtype=torch.float64, device=dev)
        t_fused = event_ms(lambda: D.jaccard_edges(padded, n, k, 0, m, out=cal_o, flags=flags))
        t_count = event_ms(lambda: D.jaccard_counts(padded, n, k, 0, m, out=cal_c, flags=flags))
        t_expand = event_ms(lambda: D.expand(padded, k, cal_c, mode=0, row_lo=0, row_hi=m, out=cal_o))
        del cal_c, cal_o
        cal = torch.tensor([t_fused, t_count, t_expand], dtype=torch.float64, device=dev)
        dist.broadcast(cal, src=0)  # every rank must use the same split
        t_fused, t_count, t_expand = (float(x) for x in cal)
        share = a.host_share if a.host_share >= 0 else sharding.balanced_host_share(world, t_fused, t_count, t_expand)
        if a.host_share < 0 and share < 0.08:
            # measured (profiles/r02_scaling.md): a host rank that first spends a few % of the step on
            # own rows starts its streaming expand behind the peers and ends later than one that only expands
            share = 0.0
        if a.gather == "peer" and k <= 127:
            try:
                pg = sharding.PeerGather(n, k, host_share=share,
                                         direct_share=a.direct_share if a.direct_share >= 0 else None)
                if pg.out3 is not None:  # the peer-store split: the output lives in the buffer the gather exports
                    out = pg.out3
            except RuntimeError as ex:  # raised on every rank together
                sys.stderr.write("bench.py: %s; falling back to NCCL send/recv\n" % ex)
                a.gather = "nccl"
        else:
            a.gather = "nccl"
        if a.gather == "peer":
            pg.flags = flags

            def step():
                pg.step(padded, out)
            lo, hi = pg.bounds[rank]
            host_share = pg.rows_of(0) / n
            sharding_note = (
                "rows over %d ranks, host rank takes %.1f%% (calibrated on this GPU: fused %.3f / count %.3f / expand "
                "%.3f ms per 1M rows); resident replicated int32 index; ONE persistent count launch per rank whose "
                "epilogue stores the parity-tagged u8 counts into rank 0's HBM (CUDA IPC mapping over NVLink); rank 0: "
                "fused kernel on its own rows, then ONE streaming expand launch that polls the count bytes (no flags, "
                "no per-chunk launches); peer-store share %.0f%% (finished doubles of a peer's last rows stored by the "
                "peer itself into rank 0's output)" % (world, 100.0 * host_share, t_fused * 1e6 / m, t_count * 1e6 / m,
                                                        t_expand * 1e6 / m, 100.0 * pg.direct_share))
        else:
            counts_all = torch.empty(E, dtype=torch.uint8 if k <= 255 else torch.int16, device=dev)
            pg = sharding.PipelinedGather(n, k, rho=t_expand / t_count, chunks=a.chunks)
            pg.flags = flags

            def step():
                pg.step(padded, counts_all, out)
            lo, hi = pg.bounds[rank]
            host_share = (pg.bounds[0][1] - pg.bounds[0][0]) / n
            sharding_note = ("rows over %d ranks, host rank takes %.1f%%; resident replicated int32 index; %d chunks per "
                             "rank; u8 counts reach rank 0 over NCCL send/recv as counted; expand kernel on rank 0 "
                             "overlapping the next chunk" % (world, 100.0 * host_share, a.chunks))

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    torch.cuda.profiler.start()  # ncu --profile-from-start off: skip the input generator's launches
    for _ in range(warm):
        step()
    barrier()
    launches0 = pg.launches if pg is not None else 0
    if pg is not None and hasattr(pg, "trace") and rank == 0:
        pg.trace = []
    sampler = ClockSampler(local)
    ev0 = [torch.cuda.Event(enable_timing=True) for _ in range(a.steps)]
    ev1 = [torch.cuda.Event(enable_timing=True) for _ in range(a.steps)]
    sampler.start()
    t_wall0 = time.perf_counter()
    for i in range(a.steps):
        flush.fill_(i & 0xFF)  # evict the index and the previous outputs from L2 (not timed)
        if world > 1:
            dist.barrier()
        ev0[i].record()
        step()
        ev1[i].record()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop()
    step_ms = torch.tensor([e0.elapsed_time(e1) for e0, e1 in zip(ev0, ev1)], dtype=torch.float64, device=dev)
    gather_flags = 0
    per_rank = None
    if world > 1:
        mine = torch.tensor([float(step_ms.mean())], dtype=torch.float64, device=dev)
        allm = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allm, mine)
        per_rank = {"step_ms_mean": [round(float(v[0]), 4) for v in allm]}
        if rank == 0 and getattr(pg, "trace", None):
            tr = pg.trace
            per_rank["host_rank_own_rows_ms"] = round(sum(a.elapsed_time(b) for a, b, _ in tr) / len(tr), 4)
            per_rank["host_rank_expand_ms"] = round(sum(b.elapsed_time(c) for _, b, c in tr) / len(tr), 4)
        dist.all_reduce(step_ms, op=dist.ReduceOp.MAX)  # max over ranks, per step
        nl = pg.launches - launches0
        if a.gather == "peer":
            gather_flags = pg.finish(padded, out)  # collective: raises on a peer timeout, exact path on repeated ids
        # the dominant kernel alone (count kernel over this rank's rows; rank 0: its fused kernel), for the roofline
        scratch = torch.empty(max(1, (hi - lo) * k), dtype=torch.uint8 if k <= 255 else torch.int16, device=dev)
        kt = event_ms(lambda: D.jaccard_counts(padded, n, k, lo, hi, out=scratch, flags=flags), reps=5, warmups=3) \
            if hi > lo else 0.0
        del scratch
        kern_t = torch.tensor([kt, float(hi - lo), float(nl)], dtype=torch.float64, device=dev)
        allk = [torch.zeros_like(kern_t) for _ in range(world)]
        dist.all_gather(allk, kern_t)
        slowest = max(allk, key=lambda v: float(v[0]))
        kern_avg_ms = float(slowest[0])
        kern_rows = int(slowest[1])
        total_launches = int(sum(float(v[2]) for v in allk))
    else:
        kern_avg_ms = float(step_ms.mean())
    assert int(flags[0]) == 0 and gather_flags == 0, "fast kernel flagged the synthetic input"
    if rank == 0 and a.dump_outputs:
        dump_outputs(a.dump_outputs, out, flags)
    total_ms = float(step_ms.sum())
    ms_per_step = total_ms / a.steps
    value = E / (ms_per_step * 1e-3)
    edges_per_launch = E if world == 1 else kern_rows * k
    bpe = bytes_per_edge if world == 1 else (4 * k + 4 + 1)  # count kernel writes 1 B/edge
    achieved = edges_per_launch * bpe / (kern_avg_ms * 1e-3) / 1e9

    # ---- parity of the value path (rank 0): the checker on head / middle / tail rows, and at N>1 the
    #      whole matrix against the single-GPU fused kernel
    parity = None
    r_host_matrix = None
    if rank == 0 and not a.no_parity:
        chk, chk_kind = checker()
        r_host_matrix = synth.to_r_matrix(idx0)
        ranges = parity_ranges(n)
        parity = {"checker": chk_kind, "oracle_rows": ranges,
                  "value_path_equals_oracle": rows_equal(
                      chk, r_host_matrix, k, ranges, lambda lo_, hi_: out[:, lo_ * k:hi_ * k].cpu().numpy().T)}
        if world > 1:
            single = torch.empty((3, E), dtype=torch.float64, device=dev)
            fl1 = D.new_flags(dev)
            D.jaccard_edges(padded, n, k, out=single, flags=fl1)
            torch.cuda.synchronize()
            parity["full_matrix_equal"] = bool(torch.equal(single, out)) and int(fl1[0]) == 0
            parity["full_matrix_vs"] = "single-GPU fused kernel on rank 0, torch.equal over all 3 x %d doubles" % E
            del single

    # ---- end to end through the reference-facing call, host buffers
    e2e = None
    if not a.no_e2e:
        e2e_steps = a.e2e_steps or min(a.steps, 10)
        if world == 1:
            if r_host_matrix is None:
                r_host_matrix = synth.to_r_matrix(idx0)

            def timed_call(mat, outbuf, reps, env=None):
                old = {}
                for kk, vv in (env or {}).items():
                    old[kk] = os.environ.get(kk)
                    os.environ[kk] = vv
                try:
                    gficf_b200.rcpp_parallel_jaccard_coef(mat, False, 1, out=outbuf)
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    for _ in range(reps):
                        gficf_b200.rcpp_parallel_jaccard_coef(mat, False, 1, out=outbuf)
                    dt = (time.perf_counter() - t0) / reps
                finally:
                    for kk, vv in old.items():
                        if vv is None:
                            os.environ.pop(kk, None)
                        else:
                            os.environ[kk] = vv
                tm = {kk: round(v, 3) for kk, v in gficf_b200.last_timings().items()}
                return dt, tm, gficf_b200.last_output()

            r_host = gficf_b200.pinned_empty((n, k))
            r_host[...] = r_host_matrix
            out_host = gficf_b200.pinned_empty((E, 3))
            gficf_b200.rcpp_parallel_jaccard_coef(r_host, False, 1, out=out_host)
            dt, tm, om = timed_call(r_host, out_host, e2e_steps)
            e2e = {"value": E / dt, "unit": UNIT, "h2d_bytes_per_step": int(om["h2d_bytes"]),
                   "d2h_bytes_per_step": int(om["d2h_bytes"]),
                   "ms_per_step": dt * 1e3, "call": "gficf_b200.rcpp_parallel_jaccard_coef (f64 R matrix, pinned host buffers)",
                   "output_mode": om, "breakdown_ms": tm}
            if parity is not None:
                oh = np.asarray(out_host)
                parity["e2e_equals_oracle"] = rows_equal(chk, r_host_matrix, k, parity["oracle_rows"],
                                                         lambda lo_, hi_: oh[lo_ * k:hi_ * k])
                dev_res = out.cpu().numpy().T
                parity["e2e_equals_value_path_full_matrix"] = bool(np.array_equal(oh, dev_res))
                del dev_res
            # r01's output path for comparison: the device writes 24 B/edge, the copy engine moves them
            dtd, tmd, omd = timed_call(r_host, out_host, 3, {"GFICF_CUDA_OUT_MODE": "dma", "GFICF_CUDA_H2D_NARROW": "0"})
            e2e["dma_output_mode"] = {"value": E / dtd, "ms_per_step": dtd * 1e3, "h2d_bytes_per_step": int(omd["h2d_bytes"]),
                                      "d2h_bytes_per_step": int(omd["d2h_bytes"]), "breakdown_ms": tmd,
                                      "what": "r01 path: doubles over PCIe both ways (GFICF_CUDA_OUT_MODE=dma, "
                                              "GFICF_CUDA_H2D_NARROW=0)"}
            # the same call on ordinary pageable memory (what R hands over)
            r_page = np.asfortranarray(np.array(r_host))
            out_page = np.zeros((E, 3), dtype=np.float64, order="F")
            dtp, tmp_, omp = timed_call(r_page, out_page, 3)
            e2e["pageable"] = {"value": E / dtp, "ms_per_step": dtp * 1e3, "output_mode": omp,
                               "matches_pinned": bool(np.array_equal(out_page, np.asarray(out_host))),
                               "breakdown_ms": tmp_}
            del r_page, out_page
            # uwot's integer matrix taken as it is (gficf_cuda_jaccard_i32): half the H2D bytes
            r_i32 = gficf_b200.pinned_empty((n, k), dtype=np.int32)
            r_i32[...] = np.asarray(r_host).astype(np.int32)
            dti, tmi, omi = timed_call(r_i32, out_host, 3)
            e2e["int32_input"] = {"value": E / dti, "ms_per_step": dti * 1e3, "h2d_bytes_per_step": int(omi["h2d_bytes"]),
                                  "d2h_bytes_per_step": int(omi["d2h_bytes"]), "output_mode": omi, "breakdown_ms": tmi}
            del r_i32
            # the step after the path through ITS host-buffer entry (gficf_cuda_snn_lower): kNN matrix in,
            # the CSC arrays RunModularityClustering's edge loop produces out -- instead of the edge matrix
            if k <= 127:
                try:
                    from gficf_b200 import snn

                    bufs = {"colptr": gficf_b200.pinned_empty((n + 1,), dtype=np.int64),
                            "row": gficf_b200.pinned_empty((E,), dtype=np.int32),
                            "weight": gficf_b200.pinned_empty((E,), dtype=np.float64),
                            "vertex_cell": gficf_b200.pinned_empty((n,), dtype=np.int32)}
                    snn.snn_graph(r_host, out=bufs)
                    t0 = time.perf_counter()
                    for _ in range(3):
                        g_ = snn.snn_graph(r_host, out=bufs)
                    dts = (time.perf_counter() - t0) / 3
                    tms = gficf_b200.last_timings()
                    e2e["snn_graph"] = {"ms_per_step": dts * 1e3, "nnz": g_["nnz"], "n_vertices": g_["n_vertices"],
                                        "d2h_bytes_per_step": int(tms["d2h_bytes"]),
                                        "breakdown_ms": {kk: round(v, 3) for kk, v in tms.items()},
                                        "call": "gficf_b200.snn.snn_graph (gficf_cuda_snn_lower, pinned host buffers): "
                                                "replaces Jaccard D2H + R filter + igraph + triangle scan"}
                    del bufs, g_
                except Exception as ex:
                    e2e["snn_graph"] = {"error": str(ex)[:200]}
            del r_host, out_host
        else:
            # one process per GPU on SHARED host matrices: every rank moves its own rows over its
            # own PCIe link (gficf_cuda_jaccard_rank); rank 0 owns / fills / checks the matrices
            from gficf_b200 import multiproc

            multiproc.comm_init_from_torch()
            tag = [("gficf_bench_%d_%d" % (os.getpid(), int(time.time()))) if rank == 0 else None]
            dist.broadcast_object_list(tag, src=0)
            numa = multiproc.bind_to_gpu_numa_node(local)
            numa_aware = numa.startswith("node")  # only then is first-touch placement meaningful
            r_sh = out_sh = None
            if rank == 0:
                r_sh = multiproc.SharedHostMatrix(tag[0] + "_idx", (n, k), create=True, pin=not numa_aware)
                out_sh = multiproc.SharedHostMatrix(tag[0] + "_out", (E, 3), create=True, pin=not numa_aware)
                if not numa_aware:
                    r_sh.array[...] = r_host_matrix if r_host_matrix is not None else synth.to_r_matrix(idx0)
            dist.barrier()
            if rank != 0:
                r_sh = multiproc.SharedHostMatrix(tag[0] + "_idx", (n, k), create=False, pin=not numa_aware)
                out_sh = multiproc.SharedHostMatrix(tag[0] + "_out", (E, 3), create=False, pin=not numa_aware)
            if numa_aware:
                s_lo, s_hi = sharding.slab_bounds(n, world, rank)
                r_sh.first_touch_rows(s_lo, s_hi)
                out_sh.first_touch_rows(s_lo * k, s_hi * k)
                dist.barrier()
                if rank == 0:
                    r_sh.array[...] = r_host_matrix if r_host_matrix is not None else synth.to_r_matrix(idx0)
                dist.barrier()
                r_sh.pin()
                out_sh.pin()
            dist.barrier()
            for _ in range(2):
                multiproc.rcpp_parallel_jaccard_coef_rank(r_sh.array, out_sh.array)
            barrier()
            t0 = time.perf_counter()
            for _ in range(e2e_steps):
                multiproc.rcpp_parallel_jaccard_coef_rank(r_sh.array, out_sh.array)
            barrier()
            dt = torch.tensor([(time.perf_counter() - t0) / e2e_steps], dtype=torch.float64, device=dev)
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
            om = gficf_b200.last_output()
            d2h = torch.tensor([om["d2h_bytes"], om["h2d_bytes"]], dtype=torch.float64, device=dev)
            dist.all_reduce(d2h)
            e2e = {"value": E / float(dt[0]), "unit": UNIT, "h2d_bytes_per_step": int(d2h[1]),
                   "d2h_bytes_per_step": int(d2h[0]), "ms_per_step": float(dt[0]) * 1e3,
                   "call": "gficf_b200.multiproc.rcpp_parallel_jaccard_coef_rank (one rank per GPU, shared "
                           "page-locked host matrices; each rank moves its own row slab)",
                   "pinned": bool(r_sh.pinned and out_sh.pinned), "numa_binding_rank0": numa,
                   "output_mode_rank0": om,
                   "breakdown_ms_rank0": {kk: round(v, 3) for kk, v in gficf_b200.last_timings().items()}}
            if rank == 0 and parity is not None:
                parity["e2e_equals_oracle"] = rows_equal(chk, r_host_matrix, k, parity["oracle_rows"],
                                                         lambda lo_, hi_: out_sh.array[lo_ * k:hi_ * k])
                ok = True  # and the whole shared result against the value path, in pieces (host RAM)
                step_e = 8_000_000
                for e0_ in range(0, E, step_e):
                    e1_ = min(E, e0_ + step_e)
                    ok = ok and bool(np.array_equal(out_sh.array[e0_:e1_], out[:, e0_:e1_].cpu().numpy().T))
                parity["e2e_equals_value_path_full_matrix"] = ok
            barrier()
            r_sh.close()
            out_sh.close()
            multiproc.comm_destroy()

    # ---- the step after the path, on the device (SURVEY 8f row 1): counts+mutual -> SNN lower triangle
    snn_rec = None
    if world == 1 and k <= 127:
        try:
            from gficf_b200 import snn

            snn.snn_lower_triangle(padded, n, k)
            torch.cuda.synchronize()
            ts = []
            for i in range(3):
                flush.fill_(i)
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                colptr, srows, sw, sflags = snn.snn_lower_triangle(padded, n, k)
                e1.record()
                torch.cuda.synchronize()
                ts.append(e0.elapsed_time(e1))
            snn_rec = {"ms": sum(ts) / len(ts), "nnz": int(srows.numel()), "flags": int(sflags[0]),
                       "what": "count kernel with mutual bit + CSC of the strictly lower triangle of the summed "
                               "adjacency (replaces the R filter, igraph and the triangle scan), device resident"}
        except Exception as ex:  # an extra record, never a reason to lose the bench line
            snn_rec = {"error": str(ex)[:200]}

    # ---- and the bulk steps of the community detection on that graph (SURVEY 8f row 3)
    net_rec = None
    if snn_rec is not None and "error" not in snn_rec:
        try:
            net_rec = network_record(colptr, srows, sw, n, k, a, dev, flush)
        except Exception as ex:  # an extra record, never a reason to lose the bench line
            net_rec = {"error": str(ex)[:200]}
    colptr = srows = sw = None

    # ---- CPU baseline beside it (rank 0, N=1 only): all host threads, and nt=2 (the clustcells default)
    cpu = cpu_nt2 = None
    if world == 1 and not a.no_cpu_baseline:
        r = r_host_matrix if r_host_matrix is not None else synth.to_r_matrix(idx0)
        run, m, kind, cores = reference_sampler(r, k, a.cpu_seconds)
        t = run(0, m)
        cpu = {"value": m * k / t, "unit": UNIT, "cores": cores, "kind": kind,
               "sample": "rows [0,%d) of %d (%.3g edges) gathering from the full matrix, %.1f s" % (m, n, m * k, t)}
        if parity is not None:
            cpu["gpu_matches_on_sample"] = parity["value_path_equals_oracle"]
        run2, m2, kind2, _ = reference_sampler(r, k, min(6.0, a.cpu_seconds), nthreads=2)
        t2 = run2(0, m2)
        cpu_nt2 = {"value": m2 * k / t2, "unit": UNIT, "cores": 2, "kind": kind2,
                   "what": "RcppParallel::setThreadOptions(numThreads = nt), nt = 2: the clustcells() default "
                           "(R/clustCells.R:46,64)",
                   "sample": "rows [0,%d) of %d (%.3g edges), %.1f s" % (m2, n, m2 * k, t2)}

    traffic, traffic_src = None, None
    if rank == 0 and world == 1:
        if not a.no_traffic_probe:
            del out
            torch.cuda.empty_cache()
            traffic, traffic_src = probe_traffic(a)
        if traffic is None:
            try:  # committed ncu capture of this exact kernel/workload
                tj = json.load(open(os.path.join(ROOT, "profiles", "r02_traffic.json")))
                key = "cells=%d k=%d" % (n, k)
                if key in tj:
                    traffic, traffic_src = tj[key]["traffic_bytes"], "profiles/r02_traffic.json (%s); live probe: %s" % (
                        tj[key].get("from", "ncu --set full"), traffic_src)
            except Exception:
                pass
    if rank == 0:
        g, b, s, v = (C_int32() for _ in range(4))
        gficf_b200.lib().gficf_cuda_last_launch(g, b, s, v)
        if world == 1:
            kname = ("jaccard_small_k_kernel<%d,0>" % D.row_stride(k)) if k <= 32 else \
                ("jaccard_wide_k_kernel<0>" if k <= 128 else "jaccard_large_k_kernel")
        else:
            kname = ("jaccard_small_k_kernel<%d,1>" % D.row_stride(k)) if k <= 32 else \
                ("jaccard_wide_k_kernel<1>" if k <= 128 else "jaccard_large_k_kernel")
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": warm,
            "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "int32 ids / f64 weights", "data": "synthetic",
            "config": {"workload": workload_name(a), "config": a.config, "cells": n, "k": k, "edges": E,
                       "l2": "explicit 256 MiB flush write between timed steps; index %d*n*4 B = %.0f MB vs 126 MB L2"
                             % (D.row_stride(k), n * D.row_stride(k) * 4 / 1e6),
                       "sharding": sharding_note,
                       "launch": {"grid": g.value, "block": b.value, "smem": s.value}},
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": hbm_peak, "unit": "GB/s",
                         "frac": achieved / hbm_peak, "traffic": traffic, "traffic_source": traffic_src,
                         "kernel": kname, "bytes_per_edge": bpe, "edges_per_launch": edges_per_launch,
                         "kernel_ms": kern_avg_ms, "peak_source": peak_src},
            "kernel_only": None if world == 1 else {
                "value": E / (kern_avg_ms * 1e-3), "unit": UNIT, "ms": kern_avg_ms,
                "what": "all ranks counting their rows concurrently, slowest rank's kernel; no gather / expand"},
            "per_rank": per_rank,
            "clocks": clocks,
            "gpu_launches": a.steps if world == 1 else int(total_launches),
            "loop_wall_ms": t_wall * 1e3,
        }
        if parity:
            line["parity"] = parity
        if snn_rec:
            line["snn_next_row"] = snn_rec
        if net_rec:
            line["network_next_row"] = net_rec
        if e2e:
            line["e2e"] = e2e
        if cpu:
            line["cpu_baseline"] = cpu
        if cpu_nt2:
            line["cpu_baseline_nt2"] = cpu_nt2
        print(json.dumps(line))
    if world > 1:
        if a.gather == "peer":
            pg.close()
        dist.destroy_process_group()


def C_int32():
    import ctypes

    return ctypes.c_int32(0)


def main():
    a = parse()
    # exactly ONE JSON line on stdout: libraries (NCCL's version banner ...) write to fd 1 too, so
    # everything else goes to stderr and only the record is written to the real stdout
    real = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    sys.stdout = real
    if a.traffic_probe:
        run_traffic_probe(a)
    elif a.impl == "reference":
        run_reference_arm(a)
    else:
        run_ours(a)
    real.flush()


if __name__ == "__main__":
    main()
