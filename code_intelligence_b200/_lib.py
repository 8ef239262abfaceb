"""ctypes binding of libissue_emb_b200.so (C ABI: include/issue_emb_b200.h).

There is deliberately NO fallback: if the CUDA library is missing or cannot be loaded this module raises, and
every entry point fails when no sm_100 device is present.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
from pathlib import Path

_PKG = Path(__file__).resolve().parent
LIB_PATH = _PKG / "libissue_emb_b200.so"

IE_OK, IE_ERR_INVALID, IE_ERR_CUDA, IE_ERR_OOM, IE_ERR_STATE, IE_ERR_TOKEN = 0, -1, -2, -3, -4, -5
IE_FLAG_DEVICE_PTRS = 1
IE_MAX_BATCH = 3072          # upper bound; a handle's own limit is ie_encoder_max_batch() (1280 by default)
IE_CFG_ACCURATE_GATES, IE_CFG_FP32, IE_CFG_F32_GX = 1, 2, 4


class ie_config(C.Structure):
    _fields_ = [("n_layers", C.c_int32), ("emb_sz", C.c_int32), ("n_hid", C.c_int32), ("vocab_sz", C.c_int32),
                ("pad_idx", C.c_int32), ("device", C.c_int32), ("flags", C.c_int32)]


# name -> (restype, argtypes); must list every symbol declared in include/issue_emb_b200.h
PROTOTYPES = {
    "ie_version": (C.c_int, []),
    "ie_last_error": (C.c_char_p, []),
    "ie_encoder_create": (C.c_int, [C.POINTER(ie_config), C.POINTER(C.c_void_p)]),
    "ie_encoder_destroy": (None, [C.c_void_p]),
    "ie_encoder_load_embedding": (C.c_int, [C.c_void_p, C.c_void_p]),
    "ie_encoder_load_layer": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "ie_encoder_encode": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                    C.c_void_p]),
    "ie_encoder_raw_features": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_int32,
                                          C.c_void_p]),
    "ie_encoder_launch_count": (C.c_int64, [C.c_void_p]),
    "ie_encoder_max_batch": (C.c_int32, [C.c_void_p]),
    "ie_encoder_check_errors": (C.c_int, [C.c_void_p]),
    "ie_encoder_last_phase_ms": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32]),
    "ie_encoder_last_phase_mhz": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32]),
    "ie_debug_seq_trace": (C.c_int64, [C.c_void_p, C.c_int32, C.c_void_p, C.c_int64]),
    "ie_mlp_create": (C.c_int, [C.c_int32, C.POINTER(C.c_int32), C.c_int32, C.POINTER(C.c_void_p)]),
    "ie_mlp_load_layer": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "ie_mlp_predict_proba": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p]),
    "ie_mlp_destroy": (None, [C.c_void_p]),
    "ie_pr_thresholds": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_double, C.c_double, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "ie_knn_create": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                C.POINTER(C.c_void_p)]),
    "ie_knn_search": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                C.c_int32, C.c_void_p]),
    "ie_knn_destroy": (None, [C.c_void_p]),
    "ie_debug_gemm": (C.c_int,[C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_int32,
                                C.c_void_p, C.c_int32]),
}

_lib = None


def build(verbose: bool = False) -> Path:
    """Compile the CUDA sources for sm_100a (nvcc cross-compiles without a GPU)."""
    r = subprocess.run(["make", "-C", str(_PKG / "csrc"), "-j8"], capture_output=True, text=True)
    if verbose or r.returncode != 0:
        print(r.stdout[-4000:])
        print(r.stderr[-4000:])
    if r.returncode != 0:
        raise RuntimeError("building libissue_emb_b200.so failed")
    return LIB_PATH


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    if not LIB_PATH.exists():
        if os.environ.get("IE_B200_NO_AUTOBUILD"):
            raise ImportError(f"{LIB_PATH} is missing (run `python -c 'import __graft_entry__ as g; g.build()'`)")
        build()
    lib = C.CDLL(str(LIB_PATH))
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


def check(rc: int) -> None:
    """Map C error codes to the exceptions the reference's callers expect (SURVEY.md section 8b):
    RuntimeError for CUDA failures / OOM (so the batch-halving loop of
    py/code_intelligence/inference.py:214-223 still works), ValueError for bad shapes / token ids."""
    if rc == IE_OK:
        return
    msg = (load().ie_last_error() or b"").decode("utf-8", "replace")
    if rc in (IE_ERR_INVALID, IE_ERR_TOKEN):
        raise ValueError(msg)
    if rc == IE_ERR_OOM:
        raise RuntimeError("CUDA out of memory. " + msg)
    raise RuntimeError(msg)
