"""ctypes binding of libicr_b200.so (the C ABI of include/icr_b200.h).

The library is built in-tree by ``build.py`` (nvcc, sm_100a). There is no CPU or
PyTorch-eager fallback: if the shared object is missing, or the device is not a B200,
every compute entry point raises.
"""

from __future__ import annotations

import ctypes
from ctypes import c_char_p, c_float, c_int, c_int64, c_size_t, c_uint32, c_void_p
from pathlib import Path

import os

# ICR_B200_LIB: a development build of the same sources (e.g. lib/libicr_b200_trace.so, built with -DICR_TRACE by
# `python -m ...build --trace`); the default is the library build() produces
LIB_PATH = Path(os.environ.get("ICR_B200_LIB") or Path(__file__).resolve().parent / "lib" / "libicr_b200.so")

ICR_F32, ICR_BF16, ICR_F16, ICR_I8 = 0, 1, 2, 3  # ICR_I8: top-k catalogs only (codes + factors of icr_quantize_rows)
PATH_AUTO, PATH_GEMV, PATH_GEMM = 0, 1, 2
PATH_WS_RESIDENT = 0x100  # OR-ed into a path: resident workspace, see include/icr_b200.h
MAX_K = 256
ABI_VERSION = 3  # include/icr_b200.h ICR_ABI_VERSION

_STATUS = {
    -1: ("ICR_ERR_ARG", ValueError),
    -2: ("ICR_ERR_DTYPE", TypeError),
    -3: ("ICR_ERR_ALIGN", ValueError),
    -4: ("ICR_ERR_K", ValueError),
    -5: ("ICR_ERR_WORKSPACE", RuntimeError),
    -6: ("ICR_ERR_CUDA", RuntimeError),
    -7: ("ICR_ERR_DEVICE", RuntimeError),
}

# name -> (restype, argtypes); mirrors include/icr_b200.h one to one
SIGNATURES = {
    "icr_abi_version": (c_int, []),
    "icr_last_error_string": (c_char_p, []),
    "icr_device_supported": (c_int, []),
    "icr_last_launch_count": (c_int, []),
    "icr_profile_enable": (c_int, [c_int]),
    "icr_profile_collect": (c_int, [c_void_p, c_void_p, c_void_p, c_void_p]),
    "icr_row_inv_norms": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_int, c_void_p, c_void_p]),
    "icr_split_f16_planes": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p]),
    "icr_planes_row_elems": (c_int64, [c_int64]),
    "icr_screen_plane": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_void_p, c_void_p]),
    "icr_screen_plane_row_elems": (c_int64, [c_int64]),
    "icr_convert_rows": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64, c_int, c_int, c_void_p]),
    "icr_quantize_rows": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64, c_void_p, c_void_p]),
    "icr_update_rows": (
        c_int,
        [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int64, c_int, c_void_p, c_int64, c_void_p, c_void_p, c_int, c_void_p],
    ),
    "icr_cos_topk_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int, c_int, c_int, c_int]),
    "icr_cos_topk": (
        c_int,
        [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int64,
         c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p],
    ),
    "icr_query_exclusion_bits": (c_int, [c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "icr_cos_topk_excl": (
        c_int,
        [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int,
         c_int64, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p],
    ),
    "icr_cos_topk_subset_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int, c_int]),
    "icr_cos_topk_subset": (
        c_int,
        [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_int64, c_int,
         c_int64, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p],
    ),
    "icr_cos_sim_dense_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int]),
    "icr_cos_sim_dense": (
        c_int,
        [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, c_int64, c_int, c_void_p, c_int64, c_void_p, c_size_t, c_void_p],
    ),
    "icr_topk_merge_workspace_bytes": (c_size_t, [c_int64, c_int, c_int, c_int]),
    "icr_topk_merge": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p]),
    "icr_peer_buffer_bytes": (c_size_t, [c_int64, c_int]),
    "icr_peer_exchange": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_void_p, c_uint32, c_int64, c_void_p, c_void_p, c_void_p]),
    "icr_peer_exchange_merge": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_int, c_int, c_void_p, c_uint32, c_int64, c_void_p, c_void_p, c_void_p]),
    "icr_cos_topk_sharded_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64, c_int, c_int, c_int, c_int]),
    "icr_cos_topk_sharded": (
        c_int,
        [c_void_p, c_int64, c_int64, c_void_p, c_int64, c_int64, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_int, c_int64,
         c_int, c_int, c_int, c_void_p, c_uint32, c_int64, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p],
    ),
    "icr_mnrl_workspace_bytes": (c_size_t, [c_int64, c_int64]),
    "icr_mnrl_fwd": (
        c_int,
        [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p,
         c_void_p, c_size_t, c_void_p],
    ),
    "icr_mnrl_fwd_bwd": (
        c_int,
        [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p,
         c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_size_t, c_void_p],
    ),
    "icr_mnrl_scale_grads": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p, c_void_p]),
    "icr_mnrl_rect_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int64]),
    "icr_mnrl_fwd_rect": (
        c_int,
        [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int64, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p,
         c_void_p, c_size_t, c_void_p],
    ),
    "icr_mnrl_bwd_rect": (
        c_int,
        [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_int64, c_int64, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p,
         c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_size_t, c_void_p],
    ),
    "icr_ir_metrics": (
        c_int,
        [c_void_p, c_int64, c_int, c_int64, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_int, c_void_p, c_void_p, c_void_p],
    ),
    "icr_mnrl_bwd": (
        c_int,
        [c_void_p, c_int64, c_void_p, c_int64, c_int64, c_int64, c_int, c_float, c_void_p, c_void_p, c_void_p, c_void_p,
         c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_size_t, c_void_p],
    ),
}

_lib = None


class NativeLibraryMissing(RuntimeError):
    pass


def load() -> ctypes.CDLL:
    """Load the shared object once; raise loudly if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        raise NativeLibraryMissing(
            f"{LIB_PATH} not found: build it with `python -m instacart_next_order_recommendation_b200.build` "
            "(or __graft_entry__.build()). This package has no CPU / PyTorch fallback path."
        )
    lib = ctypes.CDLL(str(LIB_PATH))
    for name, (res, args) in SIGNATURES.items():
        fn = getattr(lib, name)  # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    if lib.icr_abi_version() != ABI_VERSION:
        raise RuntimeError(f"libicr_b200.so ABI version {lib.icr_abi_version()} != {ABI_VERSION}: rebuild it (python -m ...build --force)")
    _lib = lib
    return lib


def check(rc: int) -> None:
    if rc == 0:
        return
    name, exc = _STATUS.get(rc, (f"status {rc}", RuntimeError))
    msg = load().icr_last_error_string().decode(errors="replace")
    raise exc(f"libicr_b200: {name}: {msg}")
