"""ctypes binding of ``libnsc_b200.so`` (C ABI declared in ``include/nsc_b200.h``).

The library is built in-tree by ``csrc/Makefile`` (``build()`` here runs it). There is no
fallback: if the shared object is missing or a symbol cannot be resolved, importing the
encoder raises.
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess
import threading

_HERE = os.path.dirname(os.path.abspath(__file__))
# NSC_LIB selects a tuning build (csrc/Makefile VARIANT=...); the default is the product library.
LIB_PATH = os.environ.get("NSC_LIB") or os.path.join(_HERE, "libnsc_b200.so")
CSRC = os.path.join(_HERE, "csrc")

NSC_ABI_VERSION = 2
N_AZIMUTH = 360
N_FREQS = 181
MAX_ELEVATION = 128
MAX_ELEVATION_SHORT = 64    # without FLAG_TALL_IMAGES
FLAG_TALL_IMAGES = 1
MAX_DESCRIPTOR = 4096
MAX_PEERS = 8
STAGE_PROJECTED = 0
STAGE_INTERPOLATED = 1
QUANT_EPSILON = 1e-8     # the reference HistogramQuantizer's default epsilon (the uint16 encode paths)


class NscParams(C.Structure):
    """``nsc_params`` of include/nsc_b200.h."""
    _fields_ = [
        ("struct_size", C.c_int32),
        ("n_elevation", C.c_int32),
        ("n_azimuth", C.c_int32),
        ("n_bins", C.c_int32),
        ("target_rows", C.c_int32),
        ("interpolate_empty", C.c_int32),
        ("min_range", C.c_float),
        ("max_range", C.c_float),
        ("el_min_rad", C.c_double),
        ("el_max_rad", C.c_double),
        ("epsilon", C.c_float),
        ("flags", C.c_int32),
    ]


class NscError(RuntimeError):
    def __init__(self, status: int, where: str):
        lib = load()
        msg = lib.nsc_strerror(status).decode()
        if status == -9:
            msg += " -- " + lib.nsc_last_cuda_error().decode()
        super().__init__(f"{where}: {msg} (nsc_status {status})")
        self.status = status


# name -> (restype, argtypes): every symbol include/nsc_b200.h declares.
_VP, _I, _I64, _SZ = C.c_void_p, C.c_int, C.c_int64, C.c_size_t
_PP = C.POINTER(NscParams)
SYMBOLS = {
    "nsc_abi_version": (_I, []),
    "nsc_strerror": (C.c_char_p, [_I]),
    "nsc_last_cuda_error": (C.c_char_p, []),
    "nsc_default_params": (None, [_PP]),
    "nsc_freq_to_bin": (_I, [C.c_float, _PP, _VP]),
    "nsc_workspace_bytes": (_SZ, [_I, _PP]),
    "nsc_encode_batch": (_I, [_VP, _I, _VP, _I64, _I, _PP, _VP, _VP, _VP, _SZ, _VP]),
    "nsc_encode_batch_u16": (_I, [_VP, _I, _VP, _I64, _I, _PP, _VP, C.c_float, _VP, _VP, _SZ, _VP]),
    "nsc_encode_batch_peers": (_I, [_VP, _I, _VP, _I64, _I, _PP, _VP, _VP, _I, _I64, _VP, _SZ, _VP]),
    "nsc_peer_signal_wait": (_I, [_VP, _I, _I, C.c_uint32, C.c_uint32, _VP]),
    "nsc_project_batch": (_I, [_VP, _I, _VP, _I64, _I, _PP, _I, _VP, _VP, _SZ, _VP]),
    "nsc_project_intensity_batch": (_I, [_VP, _VP, _I64, _I, _PP, _VP, _VP, _VP]),
    "nsc_encode_range_images": (_I, [_VP, _I, _I, _PP, _VP, _VP, _VP]),
    "nsc_interpolate_range_images": (_I, [_VP, _I, _I, _I, _VP, _VP]),
    "nsc_anywidth_workspace_bytes": (_SZ, [_I, _I, _PP]),
    "nsc_anywidth_points": (_I, [_VP, _I, _VP, _I64, _I, _PP, _VP, _VP, _VP, _I, _VP, _SZ, _VP]),
    "nsc_anywidth_points_u16": (_I, [_VP, _I, _VP, _I64, _I, _PP, _VP, C.c_float, _VP, _VP, _SZ, _VP]),
    "nsc_anywidth_images": (_I, [_VP, _I, _I, _PP, _VP, _I, _VP, _VP, _VP, _SZ, _VP]),
    "nsc_pipeline_create": (_I, [_I64, _I, _I, C.POINTER(_VP)]),
    "nsc_pipeline_destroy": (None, [_VP]),
    "nsc_pipeline_encode": (_I, [_VP, _VP, _I, _I64, _VP, _I, _PP, _VP, _VP]),
    "nsc_pipeline_encode_u16": (_I, [_VP, _VP, _I, _I64, _VP, _I, _PP, _VP, C.c_float, _VP]),
    "nsc_pipeline_encode_scan": (_I, [_VP, _VP, _I, _I64, _PP, _VP, _VP, _VP]),
    "nsc_pipeline_encode_scans": (_I, [_VP, _VP, _VP, _I, _I, _PP, _VP, _VP]),
    "nsc_pipeline_encode_scans_u16": (_I, [_VP, _VP, _VP, _I, _I, _PP, _VP, C.c_float, _VP]),
    "nsc_voxel_overlap_workspace_bytes": (_SZ, [_I64, _I64, _I]),
    "nsc_voxel_overlap_batch": (_I, [_VP, _I, _I, _VP, _I64, _I64, _VP, _I, C.c_double, _VP, _VP, _VP, _SZ, _VP]),
    "nsc_wasserstein_cdf": (_I, [_VP, _I64, _I, C.c_float, _VP, _VP]),
    "nsc_wasserstein_workspace_bytes": (_SZ, [_I]),
    "nsc_wasserstein_query": (_I, [_VP, _I, _VP, _I64, _I, C.c_float, _VP, _VP, C.c_double, _VP, _I,
                                   _VP, _VP, _VP, _VP, _SZ, _VP]),
    "nsc_wasserstein_cdf_u16": (_I, [_VP, _I64, _I, _VP, _VP]),
    "nsc_wasserstein_query_u16": (_I, [_VP, _I, _VP, _I64, _I, C.c_float, _VP, _VP, C.c_double, _VP, _I,
                                       _VP, _VP, _VP, _VP, _SZ, _VP]),
    "nsc_wasserstein_rank_workspace_bytes": (_SZ, [_I, _I64]),
    "nsc_wasserstein_rank": (_I, [_VP, _I, _VP, _I64, _I, C.c_float, _VP, _VP, C.c_double, _VP, _I64,
                                  _VP, _VP, _VP, _VP, _SZ, _VP]),
    "nsc_wasserstein_rank_u16": (_I, [_VP, _I, _VP, _I64, _I, C.c_float, _VP, _VP, C.c_double, _VP, _I64,
                                      _VP, _VP, _VP, _VP, _SZ, _VP]),
    "nsc_quantize_histograms": (_I, [_VP, _I64, _I, C.c_float, _VP, _VP]),
    "nsc_dequantize_histograms": (_I, [_VP, _I64, _I, C.c_float, _VP, _VP]),
    "nsc_test_pairwise_sum_plan": (_I, [_I, _VP, _VP, _VP, _VP, _VP, _VP, _VP]),
    "nsc_test_host_classify": (_I, [_VP, _I, _I64, _PP, _VP, _VP, _VP]),
    "nsc_test_row_mode": (_I, [_PP]),
    "nsc_test_anywidth_path": (_I, [_PP, _I, _I]),
    "nsc_test_anywidth_fft": (_I, [_I, _VP, _VP]),
}

_lib = None
_lock = threading.Lock()


TUNE_LIB_PATH = os.path.join(_HERE, "libnsc_b200_tune.so")


def build(verbose: bool = False, tuning: bool = True) -> str:
    """Compile the CUDA sources for sm_100a into ``libnsc_b200.so`` (in-tree), and -- for the
    A/B tools and the bit-identity tests -- the tuning build ``libnsc_b200_tune.so``
    (``-DNSC_TUNING``: the only build that reads NSC_SPLIT / NSC_WS / NSC_TAILSPLIT from the
    environment; ``-DNSC_SEL_CAP=128``: a small candidate list, so that tests reach the overflow
    path of the retrieval selection; selected with ``NSC_LIB=<path>``)."""
    cmds = [["make", "-C", CSRC, "-j4"]]
    if tuning:
        cmds.append(["make", "-C", CSRC, "-j4", "VARIANT=tune", "DEFS=-DNSC_TUNING -DNSC_SEL_CAP=128"])
    for cmd in cmds:
        r = subprocess.run(cmd, capture_output=True, text=True)
        if verbose or r.returncode != 0:
            print(r.stdout)
            print(r.stderr)
        if r.returncode != 0:
            raise RuntimeError("building libnsc_b200.so failed:\n" + r.stderr[-4000:])
    return LIB_PATH


def load() -> C.CDLL:
    global _lib
    if _lib is not None:
        return _lib
    with _lock:
        if _lib is not None:
            return _lib
        if not os.path.exists(LIB_PATH):
            raise ImportError(
                f"{LIB_PATH} is missing: run `make -C {CSRC}` (or __graft_entry__.build()). "
                "There is no CPU or PyTorch fallback for the encoder.")
        lib = C.CDLL(LIB_PATH)
        for name, (res, args) in SYMBOLS.items():
            fn = getattr(lib, name)   # AttributeError if the symbol is not exported
            fn.restype = res
            fn.argtypes = args
        if lib.nsc_abi_version() != NSC_ABI_VERSION:
            raise ImportError("libnsc_b200.so ABI version mismatch")
        _lib = lib
    return _lib


def check(status: int, where: str) -> None:
    if status != 0:
        raise NscError(status, where)
