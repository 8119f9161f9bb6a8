"""gficf_b200 -- B200-native Phenograph Jaccard edge weighting (one hot path of dibbelab/gficf).

The product is the CUDA library ``libgficf_cuda.so`` (sources in ``csrc/``, C ABI in
``include/gficf_cuda.h``).  This package is its host-side mirror of the reference's
operator interface for the path:

* :func:`rcpp_parallel_jaccard_coef`  (reference R/RcppExports.R:16-18 ->
  src/rcpp_parallel_jaccard_coeff.cpp:58-80)
* :func:`jaccard_coeff`               (reference R/RcppExports.R:8-10 ->
  src/jaccard_coeff.cpp:19-45)
* :func:`phenograph_edges`            (the call site, R/clustCells.R:63-66)

plus device-resident entry points (:mod:`gficf_b200.device`), row sharding over
``torch.distributed`` (:mod:`gficf_b200.sharding`) and the steps after the path: the graph the
community detection reads (:mod:`gficf_b200.snn`), its network / quality / reduced-network
steps (:mod:`gficf_b200.modularity`), Mann-Whitney U per gene, for one split or every cluster at
once (:mod:`gficf_b200.wmu`).  There is no CPU implementation here: every call goes to the CUDA
library and fails loudly when it (or a GPU) is missing.
"""
from ._lib import GficfCudaError, build, lib, library_path  # noqa: F401
from .api import (  # noqa: F401
    MODE_PARALLEL,
    MODE_SERIAL,
    jaccard_coeff,
    last_output,
    last_timings,
    phenograph_edges,
    pinned_empty,
    rcpp_parallel_jaccard_coef,
    set_devices,
)

from .wmu import rcpp_parallel_WMU_markers, rcpp_parallel_WMU_test  # noqa: F401,E402

__all__ = [
    "GficfCudaError", "build", "lib", "library_path", "MODE_PARALLEL", "MODE_SERIAL",
    "jaccard_coeff", "rcpp_parallel_jaccard_coef", "phenograph_edges", "pinned_empty",
    "set_devices", "last_timings", "last_output", "rcpp_parallel_WMU_test", "rcpp_parallel_WMU_markers",
]
