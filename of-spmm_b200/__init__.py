"""of-spmm_b200 — B200-native SpMM / A^T·dY / SDDMM operator behind a C ABI (see DESIGN.md).

The directory name carries a hyphen (it mirrors the reference repo's name); import it through
the top-level shim ``import ofspmm_b200`` or ``importlib.import_module("of-spmm_b200")``.

Importing the package does not load the CUDA library; the first op call does, and raises
``OfspmmLibraryError`` if ``lib/libofspmm_b200.so`` is absent (no CPU fallback on this path).
"""
__version__ = "0.1.0"

from . import graphs  # noqa: F401
from ._lib import LIB_PATH, OfspmmError, OfspmmLibraryError, launch_count  # noqa: F401
from .functional import SpmmOpKernelState, sddmm_csr, spmm_csr, spmm_csr_grad_b  # noqa: F401
from .ops import (OpInferError, csr_transpose, merge_path_partition, merge_path_partition_host,  # noqa: F401
                  row_blocks, row_hist, sample_neighbors)
from .sampling import Block, sample_blocks  # noqa: F401
from . import formats  # noqa: E402,F401
