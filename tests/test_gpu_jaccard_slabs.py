"""GPU (-m gpu): the Jaccard kernels on row slabs of one device, at every k; a repeated id that only
the last output chunk of the host ABI sees; and the hash-failure fallback end to end.

* Every k in 1..160 and the large-k edges: the fused kernel and counts + expand write rows
  [row_lo, row_hi) into sentinel-filled buffers with guard zones, and the kernel each k is dispatched
  to (gficf_cuda_last_launch) is the one the CPU emulation reports (tests/cuda_emu/jaccard_emu.cpp,
  emu_jaccard_variant): both run the dispatch of gficf_b200/csrc/jaccard_plan.h.
* The host ABI cuts a device's rows into chunks whose output leaves while the next chunk is counted;
  a repeated id in the last row must still send the whole call down the exact path.
* A build with GFICF_MAX_TRIES=1 makes every row whose ids collide under the first multiplier raise
  the hash-failure flag; run in a child process (two builds of the library never share a process)."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from tests.conftest import random_knn  # noqa: E402

pytestmark = pytest.mark.gpu

K_ALL = list(range(1, 161)) + [255, 256, 257, 511, 512, 1023, 1024]
HASH_FAIL_KS = (16, 30, 33, 100, 128)


def last_variant():
    import gficf_b200

    v = C.c_int32(-1)
    gficf_b200.lib().gficf_cuda_last_launch(None, None, None, C.byref(v))
    return v.value


@pytest.fixture(scope="module")
def emu_variant(tmp_path_factory):
    from tests.test_jaccard_slabs_emu import _build

    return _build(str(tmp_path_factory.mktemp("emu") / "libjaccard_emu.so"), []).emu_jaccard_variant


@pytest.mark.parametrize("k", K_ALL)
def test_every_k_on_device_slabs(cuda, oracle, emu_variant, k):
    import torch

    from gficf_b200 import device as D
    from tests.test_jaccard_slabs_emu import serial_slab, u_of

    rng = np.random.default_rng(k)
    n = 2 * k + 500
    r = random_knn(rng, n, k)
    padded, flags = D.pad_rows(torch.from_numpy(np.ascontiguousarray(r - 1, dtype=np.int32)).cuda())
    kp = padded.shape[1]
    g = n * k + 64  # guards: a store at an absolute instead of a slab-relative edge lands in one
    cb = 1 if k <= 255 else 2
    h = n // 2 + 3
    # above k = 160 the slabs are shorter: the oracle's cost grows with k^2 per row
    slabs = ((7, h), (h, n - 5), (n - 5, n)) if k <= 160 else ((7, 40), (h, h + 33), (n - 5, n))
    for si, (lo, hi) in enumerate(slabs):
        e = (hi - lo) * k
        ref = oracle.parallel_rows(r, lo, hi)
        # fused kernel
        flags.zero_()
        buf = torch.full((3, g + e + g), -7.0, dtype=torch.float64, device="cuda")
        D.jaccard_edges_to(padded, n, k, lo, hi, *(buf[c].data_ptr() + 8 * g for c in range(3)), flags)
        assert last_variant() == emu_variant(k)
        # counts (8- or 16-bit; the 8-bit ones start off any 16-byte boundary) + expand, fixed slots
        off = (lo % 16) if cb == 1 else 0
        cbuf = torch.full(((2 * g + e) * cb + off,), 0xEE, dtype=torch.uint8, device="cuda")
        c0 = g * cb + off
        D.jaccard_counts_to(padded, n, k, lo, hi, cbuf.data_ptr() + c0, flags)
        assert last_variant() == emu_variant(k)
        out = torch.full((3, g + e + g), -7.0, dtype=torch.float64, device="cuda")
        D.expand(padded, k, cbuf[c0:c0 + e * cb], mode=0, row_lo=lo, row_hi=hi, out=out[:, g:g + e])
        torch.cuda.synchronize()
        assert int(flags[0]) == 0
        for b in (buf, out):
            h = b.cpu().numpy()
            assert (h[:, :g] == -7.0).all() and (h[:, g + e:] == -7.0).all(), ("guard", lo, hi)
            assert np.array_equal(h[:, g:g + e].T, ref), (lo, hi)
        hc = cbuf.cpu().numpy()
        assert (hc[:c0] == 0xEE).all() and (hc[c0 + e * cb:] == 0xEE).all(), ("count guard", lo, hi)
        cnt = hc[c0:c0 + e * cb].copy().view(np.uint8 if cb == 1 else np.uint16)
        assert np.array_equal(cnt.reshape(-1, k), u_of(ref, k))
        if si == 0:
            # compaction of the slab's counts, and the layout pre-pass of a slab-shaped source
            # (ld_rows = hi - lo, ld_row0 = lo)
            out1 = torch.full((3, g + e + g), -7.0, dtype=torch.float64, device="cuda")
            _, nw = D.expand(padded, k, cbuf[c0:c0 + e * cb], mode=1, row_lo=lo, row_hi=hi, out=out1[:, g:g + e])
            # the rows list distinct ids, so the serial export's unique-set counts are these multiset ones:
            # its rows are the slab's u > 0 rows in (i, j) order (oracle.serial itself is O(k^2) per edge)
            ser, m = serial_slab(ref, lo, hi, k)
            h = out1.cpu().numpy()
            assert int(nw[0]) == m and np.array_equal(h[:, g:g + e].T, ser)
            assert (h[:, :g] == -7.0).all() and (h[:, g + e:] == -7.0).all()
            src = torch.from_numpy(np.ascontiguousarray(r[lo:hi].T)).cuda()  # (k, rows) C order: column-major
            dst = torch.full((n, kp), 0x7A7A7A7A, dtype=torch.int32, device="cuda")
            flags.zero_()
            cuda.lib().gficf_cuda_layout_dev(src.data_ptr(), hi - lo, lo, n, k, lo, hi, dst.data_ptr(),
                                             flags.data_ptr(), torch.cuda.current_stream().cuda_stream)
            torch.cuda.synchronize()
            assert int(flags[0]) == 0 and torch.equal(dst[lo:hi], padded[lo:hi])
            assert bool((dst[:lo] == 0x7A7A7A7A).all()) and bool((dst[hi:] == 0x7A7A7A7A).all())


@pytest.mark.parametrize("n", [600_000, 200_000])
def test_a_repeat_only_the_last_chunk_sees(cuda, oracle, n, monkeypatch):
    """One repeated id, in the last row.  At 600 000 x 30 the counts-over-PCIe modes count in two
    chunks, at 200 000 x 30 the copy-engine mode runs the fused kernel in two chunks: the first chunk's
    output is already on its way when the flags are read, and the repeat must still send the whole call
    down the exact path."""
    from gficf_b200 import synth

    k = 30
    r = synth.to_r_matrix(synth.knn_index(n, k, scramble=True))
    s = np.sort(r, axis=1)
    assert (np.diff(s, axis=1) > 0).all()  # no other row repeats an id
    r[n - 1, 4] = r[n - 1, 21]
    want, ser = oracle.parallel(r), oracle.serial(r)
    outs = {False: np.empty((n * k, 3), dtype=np.float64, order="F"), True: cuda.pinned_empty((n * k, 3))}
    ins = {}
    for pinned in (False, True):
        for as_int in (False, True):
            src = r.astype(np.int32) if as_int else r
            if pinned:
                buf = cuda.pinned_empty((n, k), dtype=src.dtype)
                buf[...] = src
                src = buf
            ins[pinned, as_int] = np.asfortranarray(src) if not pinned else src
    for mode in ("dma", "host", "hybrid"):
        monkeypatch.setenv("GFICF_CUDA_OUT_MODE", mode)
        for (pinned, as_int), src in ins.items():
            out = outs[pinned]
            out[...] = -7.0
            got = cuda.rcpp_parallel_jaccard_coef(src, False, 1, out=out)
            assert np.array_equal(np.asarray(got), want), (mode, pinned, as_int)
            assert cuda.last_output()["host_share"] == 0.0  # no host thread expanded the discarded counts
            out[...] = -7.0
            got = cuda.jaccard_coeff(src, out=out)
            assert np.array_equal(np.asarray(got), ser), (mode, pinned, as_int)


# ---------------------------------------------------------------- hash failure, end to end
def _hash_fail_child() -> None:
    """Run against a GFICF_MAX_TRIES=1 build (GFICF_CUDA_LIB): one-row slabs raise flag 4 or nothing (both
    occur), whole-matrix device calls raise it, both host exports equal the oracle in every output mode
    without a host thread expanding the discarded fast counts, and the graph build refuses."""
    import torch

    import gficf_b200 as G
    from gficf_b200 import device as D, snn
    from oracle.binding import Oracle

    orc = Oracle()
    for k in HASH_FAIL_KS:
        rng = np.random.default_rng(k)
        n = 20_000  # ids spread over many cells: the first multiplier then collides in some rows, not all
        r = random_knn(rng, n, k)
        padded, flags = D.pad_rows(torch.from_numpy(np.ascontiguousarray(r - 1, dtype=np.int32)).cuda())
        seen = {0: 0, 4: 0}
        for lo in range(0, 400):
            flags.zero_()
            D.jaccard_counts(padded, n, k, lo, lo + 1, flags=flags)
            f = int(flags[0].item())
            assert f in (0, 4), (k, lo, f)
            seen[f] += 1
        assert seen[0] and seen[4], (k, seen)  # the build tries one multiplier; the input discriminates
        for fn in (D.jaccard_counts, D.jaccard_edges):
            flags.zero_()
            fn(padded, n, k, flags=flags)
            torch.cuda.synchronize()
            assert int(flags[0]) == 4, (k, fn.__name__)
        par, ser = orc.parallel(r), orc.serial(r)
        for mode in ("dma", "host", "hybrid"):
            os.environ["GFICF_CUDA_OUT_MODE"] = mode
            for pinned in (False, True):
                for as_int in (False, True):
                    src = r.astype(np.int32) if as_int else r
                    if pinned:
                        buf = G.pinned_empty((n, k), dtype=src.dtype)
                        buf[...] = src
                        src = buf
                    out = G.pinned_empty((n * k, 3)) if pinned else np.empty((n * k, 3), order="F")
                    out[...] = -7.0
                    assert np.array_equal(np.asarray(G.rcpp_parallel_jaccard_coef(src, False, 1, out=out)), par), \
                        (k, mode, pinned, as_int)
                    assert G.last_output()["host_share"] == 0.0, (k, mode, pinned, as_int)  # counts discarded
                    out[...] = -7.0
                    assert np.array_equal(np.asarray(G.jaccard_coeff(src, out=out)), ser), (k, mode, pinned, as_int)
        if k <= 127:
            try:
                snn.snn_graph(r)
            except G.GficfCudaError as e:
                assert e.code == 5, e
            else:
                raise AssertionError("snn_graph returned a graph built from hash-failed counts (k=%d)" % k)
    print("hash-failure child: ok")


@pytest.fixture(scope="module")
def one_try_library(tmp_path_factory):
    d = tmp_path_factory.mktemp("max_tries_1")
    so = str(d / "libgficf_cuda.so")
    out = subprocess.run(["make", "-C", os.path.join(ROOT, "gficf_b200", "csrc"), "OUT=" + so,
                          "EXTRA=-DGFICF_MAX_TRIES=1"], capture_output=True, text=True)
    assert out.returncode == 0, out.stdout[-2000:] + out.stderr[-2000:]
    return so


def test_hash_failure_takes_the_exact_path(cuda, one_try_library):
    env = dict(os.environ, GFICF_CUDA_LIB=one_try_library)
    out = subprocess.run([sys.executable, os.path.abspath(__file__), "--hash-fail-child"], env=env, cwd=ROOT,
                         capture_output=True, text=True, timeout=1800)
    assert out.returncode == 0, out.stdout[-3000:] + out.stderr[-5000:]
    assert "hash-failure child: ok" in out.stdout


if __name__ == "__main__" and sys.argv[1:] == ["--hash-fail-child"]:
    _hash_fail_child()
