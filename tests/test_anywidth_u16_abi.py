"""CPU-only checks of the uint16 entry point for image widths other than 360
(nsc_anywidth_points_u16) and of the host-buffer pipeline's parameter checks at those widths. Every
call here returns before any CUDA call: the checks run in a fixed order, and those made before the
device is touched are the ones tested."""
import ctypes as C
import os

import numpy as np
import pytest

from neural_spectral_codec_b200 import _lib

OK, NULL, BAD_STRIDE, BAD_COUNT, BAD_PARAMS, BAD_LUT, BAD_STRUCT = 0, -1, -2, -3, -4, -5, -10


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.load()


def params(lib, **kw):
    p = _lib.NscParams()
    lib.nsc_default_params(C.byref(p))
    p.flags = _lib.FLAG_TALL_IMAGES
    p.n_azimuth, p.n_elevation, p.target_rows, p.n_bins = 1024, 16, 16, 50
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def lut_for(p, bad=False):
    lut = np.minimum(np.arange(p.n_azimuth // 2 + 1) * p.n_bins // (p.n_azimuth // 2 + 1), p.n_bins - 1)
    lut = np.ascontiguousarray(lut, np.int32)
    if bad:
        lut[-1] = p.n_bins           # out of range
    return lut


def bad_param_blocks(lib):
    """(label, params or None) in the order the checks meet them."""
    short = params(lib)
    short.struct_size = 4
    return [("null", None), ("struct", short), ("width 1", params(lib, n_azimuth=1)),
            ("width 4097", params(lib, n_azimuth=4097)), ("rows 129", params(lib, n_elevation=129)),
            ("rows 65 without the flag", params(lib, n_elevation=65, flags=0)),
            ("target rows 0", params(lib, target_rows=0)), ("bins above W/2+1", params(lib, n_bins=514)),
            ("descriptor above 4096", params(lib, target_rows=64, n_bins=65)),
            ("max_range < min_range", params(lib, min_range=5.0, max_range=1.0)),
            ("fov", params(lib, el_min_rad=0.1, el_max_rad=0.1)), ("epsilon", params(lib, epsilon=-1.0))]


def anywidth(lib, p, n=2, stride=4, offsets=True, out=True, lut=None):
    """nsc_anywidth_points (float32) and nsc_anywidth_points_u16 on the same arguments."""
    fake = C.c_void_p(16)              # never dereferenced: every case returns before the device is used
    pp = C.byref(p) if p is not None else None
    lut_p = lut.ctypes.data if lut is not None else None
    f32 = lib.nsc_anywidth_points(fake, stride, fake if offsets else None, 0, n, pp, lut_p, fake if out else None,
                                  None, _lib.STAGE_INTERPOLATED, None, 0, None)
    u16 = lib.nsc_anywidth_points_u16(fake, stride, fake if offsets else None, 0, n, pp, lut_p, 1e-8,
                                      fake if out else None, None, 0, None)
    return f32, u16


def test_u16_entry_returns_the_float_entrys_codes_in_its_order(lib):
    for label, p in bad_param_blocks(lib):
        f32, u16 = anywidth(lib, p, n=-1, stride=5)        # a parameter error comes first
        assert f32 == u16 != OK, (label, f32, u16)
    p = params(lib)
    assert anywidth(lib, p, n=-1, stride=5) == (BAD_COUNT, BAD_COUNT)
    assert anywidth(lib, p, n=1, stride=5) == (BAD_STRIDE, BAD_STRIDE)
    assert anywidth(lib, p, n=0, offsets=False, out=False) == (OK, OK)
    assert anywidth(lib, p, n=1, offsets=False) == (NULL, NULL)
    assert anywidth(lib, p, n=1, out=False) == (NULL, NULL)
    assert anywidth(lib, None)[1] == NULL
    assert anywidth(lib, params(lib, n_azimuth=4097))[1] == BAD_PARAMS


class Pipeline:
    """The five pipeline entries with a handle that is never dereferenced: a null handle, or a
    dummy one for calls that a parameter check stops first."""

    def __init__(self, lib):
        self.lib = lib
        self.dummy = C.create_string_buffer(4096)
        self.pts = np.zeros((8, 4), np.float32)
        self.offs = np.array([0, 8], np.int64)
        self.counts = np.array([8], np.int64)
        self.ptrs = (C.c_void_p * 1)(self.pts.ctypes.data)
        self.out = np.zeros(4096, np.float32)

    def calls(self, p, lut, null_handle=False, n=1, stride=4):
        pl = None if null_handle else C.cast(self.dummy, C.c_void_p)
        pp, lp, out = C.byref(p), (lut.ctypes.data if lut is not None else None), self.out.ctypes.data
        L = self.lib
        return {
            "encode": L.nsc_pipeline_encode(pl, self.pts.ctypes.data, stride, 8, self.offs.ctypes.data, n, pp, lp, out),
            "encode_u16": L.nsc_pipeline_encode_u16(pl, self.pts.ctypes.data, stride, 8, self.offs.ctypes.data, n, pp,
                                                    lp, 1e-8, out),
            "encode_scans": L.nsc_pipeline_encode_scans(pl, self.ptrs, self.counts.ctypes.data, stride, n, pp, lp, out),
            "encode_scans_u16": L.nsc_pipeline_encode_scans_u16(pl, self.ptrs, self.counts.ctypes.data, stride, n,
                                                                pp, lp, 1e-8, out),
            # the per-scan entry has no count: its first check after the parameters is the stride
            "encode_scan": L.nsc_pipeline_encode_scan(pl, self.pts.ctypes.data, 5 if n < 0 else stride, 8, pp, lp,
                                                      out, None),
        }


@pytest.mark.parametrize("W,rows", [(2, 1), (77, 16), (180, 128), (512, 64), (1009, 16), (1024, 16), (4096, 64)])
def test_pipeline_accepts_every_width_in_the_envelope(lib, W, rows):
    """An in-envelope width passes parameter validation: a null pipeline gives the null-pointer
    code, a bad table BAD_LUT, a missing table the null-pointer code, and a good one reaches the
    count / stride checks that follow the parameters."""
    pl = Pipeline(lib)
    p = params(lib, n_azimuth=W, n_elevation=rows, n_bins=min(50, W // 2 + 1), target_rows=min(16, rows))
    assert set(pl.calls(p, lut_for(p), null_handle=True).values()) == {NULL}
    assert set(pl.calls(p, lut_for(p, bad=True)).values()) == {BAD_LUT}
    assert set(pl.calls(p, None).values()) == {NULL}
    got = pl.calls(p, lut_for(p), n=-1)
    assert got.pop("encode_scan") == BAD_STRIDE
    assert set(got.values()) == {BAD_COUNT}


def test_pipeline_keeps_refusing_widths_outside_the_envelope(lib):
    pl = Pipeline(lib)
    for W in (1, 4097):
        p = params(lib, n_azimuth=W)
        lut = np.zeros(2049, np.int32)
        assert set(pl.calls(p, lut).values()) == {BAD_PARAMS}, W
    for label, p in bad_param_blocks(lib):
        if p is None:
            continue
        expected = BAD_STRUCT if label == "struct" else BAD_PARAMS
        assert set(pl.calls(p, np.zeros(2049, np.int32)).values()) == {expected}, label


def test_pipeline_keeps_the_360_column_checks(lib):
    """Width 360 still takes nsc_encode_batch's checks: 181 table entries, n_bins <= 181."""
    pl = Pipeline(lib)
    p = params(lib, n_azimuth=360)
    assert set(pl.calls(p, lut_for(p, bad=True)).values()) == {BAD_LUT}
    got = pl.calls(p, lut_for(p), n=-1)
    assert got.pop("encode_scan") == BAD_STRIDE
    assert set(got.values()) == {BAD_COUNT}
