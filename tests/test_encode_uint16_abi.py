"""Device-free checks of the uint16 encode entry points (nsc_encode_batch_u16,
nsc_pipeline_encode_u16, nsc_pipeline_encode_scans_u16): argument validation happens before any
CUDA call, in the order and with the status codes of the float32 entry points."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from neural_spectral_codec_b200 import _lib
from oracle import nsc_oracle as orc


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.load()


def default_params(lib, **kw):
    p = _lib.NscParams()
    lib.nsc_default_params(C.byref(p))
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def test_encode_batch_u16_validates_like_the_float_entry(lib):
    p = default_params(lib)
    lut = orc.freq_to_bin(orc.OracleConfig()).numpy().astype(np.int32)

    def call(pts=16, stride=4, offs=16, n=1, pp=p, l=lut, out=16, ws=16, wsz=256):
        return lib.nsc_encode_batch_u16(C.c_void_p(pts) if pts else None, stride, C.c_void_p(offs) if offs else None,
                                        0, n, C.byref(pp), l.ctypes.data, 1e-8, C.c_void_p(out) if out else None,
                                        C.c_void_p(ws) if ws else None, wsz, None)

    assert call(pp=default_params(lib, n_azimuth=359)) == -4
    assert call(pp=default_params(lib, n_elevation=65)) == -4
    assert call(pp=default_params(lib, target_rows=64, n_bins=181)) == -4
    assert call(pp=default_params(lib, struct_size=12)) == -10
    bl = lut.copy()
    bl[100] = 0
    assert call(l=bl) == -5
    assert call(stride=2) == -2
    assert call(pts=20) == -7
    assert call(offs=0) == -1
    assert call(out=0) == -1
    assert call(n=-1) == -3
    assert call(ws=0) == -6 and call(wsz=4) == -6
    assert call(n=0, out=0, ws=0, wsz=0) == 0             # empty batch is a no-op
    # the float entry gives the same codes for the same arguments
    assert lib.nsc_encode_batch(C.c_void_p(20), 4, C.c_void_p(16), 0, 1, C.byref(p), lut.ctypes.data,
                                C.c_void_p(16), C.c_void_p(16), 256, None) == call(pts=20)


def test_pipeline_u16_entries_refuse_a_null_pipeline(lib):
    p = default_params(lib)
    lut = orc.freq_to_bin(orc.OracleConfig()).numpy().astype(np.int32)
    pts = np.zeros((16, 4), np.float32)
    offs = np.array([0, 16], np.int64)
    out = np.zeros((1, 800), np.uint16)
    assert lib.nsc_pipeline_encode_u16(None, pts.ctypes.data, 4, 16, offs.ctypes.data, 1, C.byref(p),
                                       lut.ctypes.data, 1e-8, out.ctypes.data) == -1
    ptrs = (C.c_void_p * 1)(pts.ctypes.data)
    counts = np.array([16], np.int64)
    assert lib.nsc_pipeline_encode_scans_u16(None, ptrs, counts.ctypes.data, 4, 1, C.byref(p), lut.ctypes.data,
                                             1e-8, out.ctypes.data) == -1


def test_python_methods_check_dtype_and_out_without_a_device(lib):
    from neural_spectral_codec_b200 import SpectralEncoder
    enc = SpectralEncoder(n_elevation=16)
    with pytest.raises(RuntimeError, match="no CPU implementation"):
        enc.encode_points_batch(torch.zeros(4, 4), torch.tensor([0, 4]), dtype=torch.uint16)
    with pytest.raises(ValueError, match="dtype"):
        enc.encode_points_batch(torch.zeros(4, 4), torch.tensor([0, 4]), dtype=torch.float16)
    with pytest.raises(ValueError, match="dtype"):
        enc.encode_scans([np.zeros((4, 4), np.float32)], dtype=np.int16)
