"""Child process of tests/test_wmu_markers_sparse_emu.py::test_emulated_sparse_pipeline_under_address_sanitizer:
runs the emulated sparse markers pipeline from a library built with -fsanitize=address (LD_PRELOAD=libasan), on
malformed input (every class of bad row id) and on a small valid matrix.
Usage: asan_markers_sparse_run.py <libwmu_markers_sparse_emu_asan.so>"""
import sys

import numpy as np

from oracle.binding import WmuOracle
from tests.test_wmu_markers_sparse_emu import edge_rows, emu_sparse, load_sparse_emu, malformed_cases, to_csc
from tests.test_wmu_oracle import sc_matrix


def main():
    L = load_sparse_emu(sys.argv[1])
    cl = np.array([0, 1, 0, 1], dtype=np.int32)
    for name, colptr, row in malformed_cases():
        x = np.arange(1.0, row.size + 1.0)
        _, flags = emu_sparse(L, colptr, row, x, 5, cl, 2)
        assert flags == 1, name
    rng = np.random.default_rng(4)
    cells, k = 300, 4
    cl = rng.integers(0, k, cells).astype(np.int32)
    cl[:k] = np.arange(k)
    m = edge_rows(rng, sc_matrix(rng, 14, cells), cl)
    colptr, row, x, m = to_csc(m, rng, 0.1)
    got, flags = emu_sparse(L, colptr, row, x, m.shape[0], cl, k, grid=3, ctas=2)
    assert flags == 0
    for c in range(k):
        want = WmuOracle().wmu(np.asfortranarray(m[:, cl == c]), np.asfortranarray(m[:, cl != c]))
        assert np.array_equal(got[:, :, c], want, equal_nan=True), c
    print("asan run ok")


if __name__ == "__main__":
    main()
