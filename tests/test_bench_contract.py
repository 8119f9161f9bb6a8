"""CPU: bench.py's reference arm prints exactly one JSON line on stdout with the contract's keys
(the GPU arm needs a device; its line is checked on the box by the driver)."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_reference_arm_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--cells", "20000",
                          "--k", "15", "--steps", "2", "--warmup", "1"], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1
    rec = json.loads(lines[0])
    for key in ("impl", "metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "cpu_baseline", "e2e", "gpu_launches"):
        assert key in rec, key
    assert rec["impl"] == "reference" and rec["unit"] == "edges/s" and rec["value"] > 0
    assert rec["cpu_baseline"]["kind"] in ("reference", "port") and rec["cpu_baseline"]["cores"] >= 1
    assert rec["e2e"]["h2d_bytes_per_step"] == 0 and rec["e2e"]["value"] == rec["value"]
    assert "workload" in rec["config"] and "sample" in rec["config"]


def test_non_zero_ranks_of_the_reference_arm_exit_quietly():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                         capture_output=True, text=True, timeout=300, env=env)
    assert out.returncode == 0 and out.stdout.strip() == ""


def test_steps_below_one_are_refused():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"],
                         capture_output=True, text=True, timeout=120)
    assert out.returncode == 2 and "--steps" in out.stderr


def test_dump_outputs_files(tmp_path):
    """bench.dump_outputs on CPU tensors: the whole result when it is small, a fixed sample of
    columns (the same in every run, under 64 MB) when it is large."""
    import numpy as np
    import torch

    import bench

    flags = torch.zeros(2, dtype=torch.int32)
    small = torch.arange(3 * 1000, dtype=torch.float64).reshape(3, 1000)
    bench.dump_outputs(str(tmp_path / "small"), small, flags)
    assert np.array_equal(np.load(tmp_path / "small" / "edges.npy"), small.numpy())
    assert np.array_equal(np.load(tmp_path / "small" / "edge_columns.npy"), np.arange(1000.0))
    assert np.load(tmp_path / "small" / "flags.npy").dtype == np.float64

    E = 3 * bench.DUMP_EDGE_COLUMNS
    big = torch.arange(E, dtype=torch.float64).expand(3, E)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), big, flags)
    total = 0
    for name in ("edges", "edge_columns", "flags"):
        x, y = np.load(tmp_path / "a" / (name + ".npy")), np.load(tmp_path / "b" / (name + ".npy"))
        assert x.dtype == np.float64 and np.array_equal(x, y)
        total += os.path.getsize(tmp_path / "a" / (name + ".npy"))
    assert total < 64e6
    cols = np.load(tmp_path / "a" / "edge_columns.npy")
    edges = np.load(tmp_path / "a" / "edges.npy")
    assert edges.shape == (3, bench.DUMP_EDGE_COLUMNS) and np.unique(cols).size == cols.size
    assert np.array_equal(edges[0], cols)


def test_network_record_of_the_bench_line(monkeypatch, tmp_path):
    """bench.network_record (the `network_next_row` object) driven on CPU tensors through the emulated
    network library: keys, parity record and the planted-community clustering, without a GPU."""
    import argparse
    import contextlib

    import numpy as np
    import torch

    import bench
    from gficf_b200 import _lib, device as D, synth
    from oracle import louvain
    from oracle.binding import Oracle
    from tests.test_network_emu import compile_emu, load_emu

    so = str(tmp_path / "libnetwork_emu.so")
    compile_emu(so)
    emu = load_emu(so)
    for name in ("gficf_cuda_network_scratch_bytes", "gficf_cuda_network_dev", "gficf_cuda_network_quality_dev",
                 "gficf_cuda_network_reduce_dev"):
        res, args = _lib.PROTOTYPES[name]
        getattr(emu, name).restype = res
        getattr(emu, name).argtypes = args

    class FakeEvent:
        def __init__(self, enable_timing=False):
            pass

        def record(self):
            pass

        def elapsed_time(self, other):
            return 1.0

    monkeypatch.setattr(_lib, "lib", lambda: emu)
    monkeypatch.setattr(D, "_require_cuda", lambda t, dtype: None)
    monkeypatch.setattr(D, "_stream_ptr", lambda: 0)
    monkeypatch.setattr(torch.cuda, "device", lambda dev: contextlib.nullcontext())
    monkeypatch.setattr(torch.cuda, "Event", FakeEvent)
    monkeypatch.setattr(torch.cuda, "synchronize", lambda *a, **k: None)
    monkeypatch.setattr(torch.cuda, "empty_cache", lambda: None)

    n, k = 600, 20
    a = argparse.Namespace(family="planted", seed=180582, no_scramble=False, no_parity=False)
    idx0 = synth.knn_index(n, k, family="planted", seed=a.seed, scramble=True)
    names, cols, rows, data = louvain.lower_triangle_edges(Oracle().parallel(synth.to_r_matrix(idx0)))
    assert names.size == n
    colptr = np.zeros(n + 1, np.int64)
    np.add.at(colptr, cols.astype(np.int64) + 1, 1)
    colptr = torch.from_numpy(np.cumsum(colptr))
    rec = bench.network_record(colptr, torch.from_numpy(rows.astype(np.int32)), torch.from_numpy(data), n, k, a,
                               torch.device("cpu"), torch.zeros(16, dtype=torch.uint8))
    assert rec["vertices"] == n and rec["clusters"] == (n - 1) // 256 + 1 and "planted communities" in rec["what"]
    assert set(rec["parity"].values()) == {True}
    assert {"network_ms", "quality_ms", "reduce_ms", "directed_edges", "reduced_edges", "quality", "cpu_ms"} <= set(rec)
