"""Loader for libibdgem_b200.so.  No fallback: a missing library is an error."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(PKG_DIR, "libibdgem_b200.so")
CSRC = os.path.join(PKG_DIR, "csrc")

# every symbol include/ibdgem_b200.h declares
ABI_SYMBOLS = [
    "ibdgem_engine_create", "ibdgem_engine_destroy", "ibdgem_last_error", "ibdgem_abi_version",
    "ibdgem_engine_set_stream", "ibdgem_engine_upload_sites", "ibdgem_engine_upload_panel", "ibdgem_engine_sync_uploads",
    "ibdgem_engine_set_panel_device", "ibdgem_engine_panel_rows_ready",
    "ibdgem_engine_prepare", "ibdgem_engine_invalidate", "ibdgem_engine_get_site_table", "ibdgem_engine_score_nonld",
    "ibdgem_engine_score_ld", "ibdgem_engine_last_ld_path", "ibdgem_engine_force_general_ld",
    "hiddengem_viterbi_batch", "ibdgem_engine_enable_timing", "ibdgem_engine_reset_stats",
    "ibdgem_engine_num_kernels", "ibdgem_engine_kernel_stats", "ibdgem_engine_device_bytes",
    "ibdgem_engine_set_window_shard", "ibdgem_engine_window_shard", "ibdgem_peer_alloc", "ibdgem_peer_open",
    "ibdgem_peer_close", "hiddengem_viterbi_batch_device", "hiddengem_last_flagged", "ibdgem_engine_clone_panel", "ibdgem_engine_set_shard_compact_output",
    "hiddengem_posterior_batch", "hiddengem_posterior_batch_device",
    "hiddengem_posterior_moments_batch", "hiddengem_posterior_moments_device",
    "hiddengem_tract_counts_batch", "hiddengem_tract_counts_device",
    "hiddengem_tract_lengths_batch", "hiddengem_tract_lengths_device",
    "hiddengem_tracts_batch", "hiddengem_tracts_device", "hiddengem_last_tracts",
]


def build_library(verbose: bool = False) -> str:
    """Compile csrc/*.cu for sm_100a into the in-tree shared library (nvcc cross-compiles
    without a GPU)."""
    r = subprocess.run(["make", "-C", CSRC], capture_output=True, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout[-4000:])
        print(r.stderr[-4000:])
    if r.returncode != 0:
        raise RuntimeError("building libibdgem_b200.so failed")
    return LIB_PATH


_lib = None


def load_library():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            f"{LIB_PATH} is missing — the CUDA engine is not built (run `python -c 'import __graft_entry__ as g; "
            "g.build()'` or `make -C ibdgem_b200/csrc`).  There is no CPU fallback.")
    lib = C.CDLL(LIB_PATH)
    lib.ibdgem_last_error.restype = C.c_char_p
    lib.ibdgem_engine_device_bytes.restype = C.c_int64
    lib.hiddengem_last_flagged.restype = C.c_int64
    for name in ABI_SYMBOLS:
        getattr(lib, name)  # raises AttributeError if the ABI is incomplete
    _lib = lib
    return lib
