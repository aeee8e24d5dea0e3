"""ibdgem_b200 — B200-native IBDGem likelihood engine.

The product is the C-ABI shared library `libibdgem_b200.so` (sources under csrc/, header
include/ibdgem_b200.h).  This package is the thin Python host-side mirror of that ABI used
by the tests, the benchmark and the Python entry points; it never computes likelihoods itself
and fails loudly if the CUDA library is missing.
"""
from ._lib import LIB_PATH, load_library, build_library  # noqa: F401
from .engine import Engine, Params, Scores, EngineError, TRACT_DTYPE  # noqa: F401
from .pack import pack_bits  # noqa: F401
from .shard import shard_bounds, shard_targets, gather_window_scores, PeerTable, upload_window_shard_rows  # noqa: F401

__all__ = ["Engine", "Params", "Scores", "EngineError", "TRACT_DTYPE", "pack_bits", "load_library", "build_library", "LIB_PATH"]
