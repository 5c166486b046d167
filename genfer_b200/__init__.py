"""genfer_b200 -- B200 (sm_100a) implementation of genfer's dense truncated Taylor arithmetic.

Layout: ``csrc/`` holds the CUDA kernels and the C ABI (``include/genfer_taylor.h``), ``taylor.py`` is
the host-side mirror of the reference's ``TaylorPoly`` / ``TaylorExpansion`` operator surface, ``build.py``
compiles ``libgenfer_taylor.so`` in-tree.  Importing this package does not need a GPU; creating a
``Context`` does (there is no CPU fallback for the f64 path).
"""
from ._lib import LIB_PATH, MAX_NDIM, SYMBOLS, UNBOUNDED, load  # noqa: F401
from .taylor import (Context, TaylorError, TaylorExpansion, TaylorPanic, TaylorPoly, UniProgram, UniSlot, default_context,  # noqa: F401
                     mul_macs, nccl_unique_id, partition_block, partition_rows, set_default_context, taylor)
from .evaluator import SgclResult, parse_flags, run_sgcl  # noqa: F401,E402
from .interval import IntervalPoly, SgclBounds, run_sgcl_bounds  # noqa: F401,E402
