"""ctypes binding of libgficf_cuda.so -- exactly the symbols include/gficf_cuda.h declares."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
# GFICF_CUDA_LIB selects another build of the SAME library (A/B tuning variants); never a fallback
_SO = os.environ.get("GFICF_CUDA_LIB") or os.path.join(_HERE, "libgficf_cuda.so")
_lib = None

E_NAMES = {1: "GFICF_E_ARG", 2: "GFICF_E_RANGE", 3: "GFICF_E_CUDA", 4: "GFICF_E_NCCL", 5: "GFICF_E_LIMIT"}

_dp = C.POINTER(C.c_double)
_vp = C.c_void_p

# name -> (restype, argtypes); kept in the order of include/gficf_cuda.h
PROTOTYPES = {
    "gficf_cuda_jaccard": (C.c_int, [_vp, C.c_int64, C.c_int32, _vp, C.c_int32, C.c_int32,
                                     C.POINTER(C.c_int64), C.c_char_p, C.c_size_t]),
    "gficf_cuda_jaccard_i32": (C.c_int, [_vp, C.c_int64, C.c_int32, _vp, C.c_int32, C.c_int32,
                                         C.POINTER(C.c_int64), C.c_char_p, C.c_size_t]),
    "gficf_cuda_set_devices": (C.c_int, [C.c_int32]),
    "gficf_cuda_get_devices": (C.c_int, []),
    "gficf_cuda_device_count": (C.c_int, []),
    "gficf_cuda_host_alloc": (C.c_int, [C.POINTER(_vp), C.c_size_t]),
    "gficf_cuda_host_free": (C.c_int, [_vp]),
    "gficf_cuda_host_register": (C.c_int, [_vp, C.c_size_t]),
    "gficf_cuda_host_unregister": (C.c_int, [_vp]),
    "gficf_cuda_release": (C.c_int, []),
    "gficf_cuda_last_timings": (C.c_int, [_dp]),
    "gficf_cuda_last_output": (C.c_int, [C.POINTER(C.c_int32), _dp, _dp, _dp]),
    "gficf_cuda_expand_host": (C.c_int, [_vp, C.c_int32, C.c_int64, C.c_int32, _vp, C.c_int64, C.c_int64, _vp,
                                         C.c_int32]),
    "gficf_cuda_comm_unique_id": (C.c_int, [_vp]),
    "gficf_cuda_comm_init_rank": (C.c_int, [_vp, C.c_int32, C.c_int32, C.c_int32, C.c_char_p, C.c_size_t]),
    "gficf_cuda_comm_destroy": (C.c_int, []),
    "gficf_cuda_jaccard_rank": (C.c_int, [_vp, C.c_int64, C.c_int32, _vp, C.c_char_p, C.c_size_t]),
    "gficf_cuda_ipc_alloc": (C.c_int, [C.c_size_t, C.POINTER(_vp), _vp]),
    "gficf_cuda_ipc_open": (C.c_int, [_vp, C.POINTER(_vp)]),
    "gficf_cuda_ipc_close": (C.c_int, [_vp]),
    "gficf_cuda_ipc_free": (C.c_int, [_vp]),
    "gficf_cuda_signal_dev": (C.c_int, [_vp, C.c_uint32, _vp]),
    "gficf_cuda_wait_dev": (C.c_int, [_vp, C.c_uint32, _vp, _vp]),
    "gficf_cuda_jaccard_counts_tagged_dev": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int64, C.c_int64, _vp,
                                                       C.c_uint32, _vp, _vp]),
    "gficf_cuda_expand_stream_dev": (C.c_int, [_vp, C.c_int32, C.POINTER(C.c_int64), C.POINTER(C.c_int64),
                                               C.c_int32, _vp, _vp, _vp, _vp, C.c_uint32, C.c_int64, _vp, _vp]),
    "gficf_cuda_row_stride": (C.c_int32, [C.c_int32]),
    "gficf_cuda_layout_dev": (C.c_int, [_vp, C.c_int64, C.c_int64, C.c_int64, C.c_int32, C.c_int64,
                                        C.c_int64, _vp, _vp, _vp]),
    "gficf_cuda_pad_dev": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int64, C.c_int64, _vp, _vp, _vp]),
    "gficf_cuda_jaccard_dev": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int64, C.c_int64, _vp, _vp, _vp,
                                         _vp, _vp]),
    "gficf_cuda_jaccard_counts_dev": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int64, C.c_int64, _vp,
                                                _vp, _vp]),
    "gficf_cuda_jaccard_exact_dev": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int64, C.c_int64,
                                               C.c_int32, _vp, _vp]),
    "gficf_cuda_expand_dev": (C.c_int, [_vp, C.c_int32, C.c_int64, C.c_int64, _vp, C.c_int32, _vp, _vp,
                                        _vp, _vp, _vp, _vp]),
    "gficf_cuda_expand_scratch_bytes": (C.c_size_t, [C.c_int64]),
    "gficf_cuda_jaccard_counts_mutual_dev": (C.c_int, [_vp, C.c_int64, C.c_int32, C.c_int64, C.c_int64, _vp,
                                                       _vp, _vp]),
    "gficf_cuda_snn_scratch_bytes": (C.c_size_t, [C.c_int64, C.c_int64]),
    "gficf_cuda_snn_lower_dev": (C.c_int, [_vp, C.c_int64, C.c_int32, _vp, _vp, _vp, _vp, C.c_int64, _vp, _vp, _vp,
                                           _vp, _vp]),
    "gficf_cuda_snn_lower": (C.c_int, [_vp, C.c_int32, C.c_int64, C.c_int32, _vp, _vp, _vp, C.c_int64, _vp,
                                       C.POINTER(C.c_int64), C.POINTER(C.c_int64), C.c_char_p, C.c_size_t]),
    "gficf_cuda_network_scratch_bytes": (C.c_size_t, [C.c_int64, C.c_int64]),
    "gficf_cuda_network_dev": (C.c_int, [_vp, _vp, _vp, C.c_int64, C.c_int64, _vp, _vp, _vp, _vp, _vp, _vp,
                                         C.c_size_t, _vp, _vp]),
    "gficf_cuda_network_quality_dev": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int64, C.c_int64, _vp, C.c_int32,
                                                 C.c_double, C.c_double, _vp, _vp, _vp, _vp, C.c_size_t, _vp, _vp]),
    "gficf_cuda_network_reduce_dev": (C.c_int, [_vp, _vp, _vp, _vp, C.c_int64, C.c_int64, _vp, C.c_int32,
                                                C.c_double, _vp, _vp, _vp, C.c_int64, _vp, _vp, _vp,
                                                C.POINTER(C.c_int64), _vp, C.c_size_t, _vp, _vp]),
    "gficf_cuda_wmu_test": (C.c_int, [_vp, _vp, C.c_int64, C.c_int64, C.c_int64, _vp, C.c_char_p, C.c_size_t]),
    "gficf_cuda_wmu_markers": (C.c_int, [_vp, C.c_int64, C.c_int64, _vp, C.c_int32, _vp, C.c_char_p, C.c_size_t]),
    "gficf_cuda_wmu_markers_csc": (C.c_int, [_vp, _vp, _vp, C.c_int64, C.c_int64, _vp, C.c_int32, _vp, C.c_char_p,
                                             C.c_size_t]),
    "gficf_cuda_set_launch_ctas_per_sm": (C.c_int, [C.c_int32]),
    "gficf_cuda_last_launch": (C.c_int, [C.POINTER(C.c_int32)] * 4),
    "gficf_cuda_version": (C.c_char_p, []),
}


class GficfCudaError(RuntimeError):
    """A non-zero return of the C ABI (the Rcpp shim turns the same thing into Rcpp::stop)."""

    def __init__(self, code: int, message: str):
        super().__init__("%s: %s" % (E_NAMES.get(code, "error %d" % code), message))
        self.code = code
        self.message = message


def library_path() -> str:
    return _SO


def build(verbose: bool = False) -> str:
    """Compile csrc/ for sm_100a into gficf_b200/libgficf_cuda.so (nvcc; no GPU needed)."""
    out = subprocess.run(["make", "-C", os.path.join(_HERE, "csrc")], capture_output=True, text=True)
    if verbose or out.returncode != 0:
        print(out.stdout[-4000:], out.stderr[-4000:])
    if out.returncode != 0:
        raise RuntimeError("building libgficf_cuda.so failed")
    return _SO


def lib() -> C.CDLL:
    """The loaded library.  Missing library = hard error (there is no fallback path)."""
    global _lib
    if _lib is None:
        if not os.path.exists(_SO):
            raise RuntimeError(
                _SO + " is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "or `make -C gficf_b200/csrc`; this package has no CPU implementation")
        L = C.CDLL(_SO)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(L, name)  # AttributeError if the header and the library drift apart
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def check(code: int, errbuf=None) -> None:
    if code != 0:
        msg = errbuf.value.decode(errors="replace") if errbuf is not None else ""
        raise GficfCudaError(code, msg)
