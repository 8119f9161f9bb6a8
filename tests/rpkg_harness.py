"""Builds librpkg_harness.so: the drop-in R-package sources + stand-in R runtime, linked against the
product library (see tests/rpkg_entry.cpp).  The library goes to a temporary directory of the test
process, not into the source tree, which may be read-only."""
import atexit
import ctypes as C
import os
import shutil
import subprocess
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
_OUT = []


def _out():
    """The harness library's path, in a temporary directory made on first use and removed at exit."""
    if not _OUT:
        d = tempfile.mkdtemp(prefix="gficf_rpkg_")
        atexit.register(shutil.rmtree, d, True)
        _OUT.append(os.path.join(d, "librpkg_harness.so"))
    return _OUT[0]


def build():
    import gficf_b200

    src = [os.path.join(ROOT, "gficf_b200", "rpkg", "src", f) for f in
           ("rcpp_parallel_jaccard_coeff.cpp", "jaccard_coeff.cpp", "gficf_cuda_devices.cpp",
            "rcpp_parallel_mann_whitney.cpp")]
    lib = gficf_b200.library_path()
    cmd = ["g++", "-O2", "-std=c++11", "-fPIC", "-shared", "-I" + os.path.join(ROOT, "oracle", "rshim"),
           "-I" + os.path.join(ROOT, "include"), os.path.join(HERE, "rpkg_entry.cpp"), *src, lib,
           "-Wl,-rpath," + os.path.dirname(lib), "-o", _out()]
    r = subprocess.run(cmd, capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError(r.stderr[-3000:])
    return _out()


class RPkg:
    def __init__(self):
        out = _out()
        if not os.path.exists(out) or os.path.getmtime(out) < os.path.getmtime(os.path.join(HERE, "rpkg_entry.cpp")):
            build()
        self.lib = C.CDLL(out)
        self.lib.rpkg_call.argtypes = [C.c_int, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_char_p,
                                       C.c_int, C.c_char_p, C.c_int]
        self.lib.rpkg_call.restype = C.c_int

    def call(self, which, idx, print_output=False):
        a = np.asfortranarray(idx, dtype=np.int32 if which == 2 else np.float64)
        n, k = a.shape
        out = np.empty((n * k, 3), dtype=np.float64, order="F")
        err = C.create_string_buffer(1024)
        printed = C.create_string_buffer(1024)
        rc = self.lib.rpkg_call(which, a.ctypes.data, n, k, out.ctypes.data, int(print_output), err, 1024,
                                printed, 1024)
        if rc != 0:
            raise RuntimeError(err.value.decode())
        return out, printed.value.decode()

    def wmu(self, x, y, print_output=False):
        x = np.asfortranarray(x, dtype=np.float64)
        y = np.asfortranarray(y, dtype=np.float64)
        g = x.shape[0]
        out = np.empty((g, 2), dtype=np.float64, order="F")
        err = C.create_string_buffer(1024)
        printed = C.create_string_buffer(1024)
        fn = self.lib.rpkg_wmu
        fn.argtypes = [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_char_p, C.c_int,
                       C.c_char_p, C.c_int]
        fn.restype = C.c_int
        rc = fn(x.ctypes.data, y.ctypes.data, g, x.shape[1], y.shape[1], out.ctypes.data, int(print_output), err, 1024,
                printed, 1024)
        if rc != 0:
            raise RuntimeError(err.value.decode())
        return out, printed.value.decode()
