"""CPU-only checks of range images of 65..128 rows (one row per beam of a 128-beam sensor): the
per-point function of the tall kernels against the oracle, both row rules at 128 rows, and the
envelope: 128 rows for a parameter block with NSC_FLAG_TALL_IMAGES, 64 without it, as before
(no GPU compute calls)."""
import ctypes as C
import os

import numpy as np
import pytest

from neural_spectral_codec_b200 import _lib, synth
from oracle import nsc_oracle as orc

FOVS = [(-24.8, 2.0), (-60.0, 60.0)]


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.load()


def default_params(lib, **kw):
    """nsc_default_params with NSC_FLAG_TALL_IMAGES set, then the given fields."""
    p = _lib.NscParams()
    lib.nsc_default_params(C.byref(p))
    p.flags = _lib.FLAG_TALL_IMAGES
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def fov_params(lib, rows, fov, **kw):
    return default_params(lib, n_elevation=rows, el_min_rad=float(np.deg2rad(fov[0])),
                          el_max_rad=float(np.deg2rad(fov[1])), **kw)


@pytest.mark.parametrize("fov", FOVS)
@pytest.mark.parametrize("shape", [synth.HDL64, synth.BEAM128], ids=lambda s: s.name)
@pytest.mark.parametrize("rows", [65, 96, 128])
def test_host_classify_matches_oracle_pixels_at_tall_rows(lib, rows, shape, fov):
    """The row and column of every kept point equal the oracle's, except within 1e-5 rad of an
    edge; the same points are kept."""
    pts = np.concatenate([synth.make_scan(shape, i).numpy() for i in range(2)])
    p = fov_params(lib, rows, fov)
    n = len(pts)
    row, col, keep = np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.uint8)
    assert lib.nsc_test_host_classify(pts.ctypes.data, 4, n, C.byref(p), row.ctypes.data, col.ctypes.data,
                                      keep.ctypes.data) == 0
    keep = keep.astype(bool)
    cfg = orc.OracleConfig(n_elevation=rows, elevation_range=fov)
    s = orc.spherical(pts, cfg)
    okeep = np.zeros(n, bool)
    okeep[s["kept"]] = True
    np.testing.assert_array_equal(keep, okeep)
    orow, ocol = np.full(n, -1), np.full(n, -1)
    orow[s["kept"]], ocol[s["kept"]] = s["row"], s["col"]
    d_az, d_el = orc.edge_distance(pts, cfg)
    clear = keep & (d_az > 1e-5) & (d_el > 1e-5)
    assert clear.sum() > 0.9 * keep.sum()
    np.testing.assert_array_equal(row[clear], orow[clear])
    np.testing.assert_array_equal(col[clear], ocol[clear])
    assert row[keep].max() <= rows - 1
    if rows == 128 and fov == (-60.0, 60.0):
        assert row[keep].max() >= 64           # the search reaches the upper half of the rows


def test_both_row_rules_at_128_rows(lib):
    """The polynomial row rule holds at 128 rows for a narrow field of view, and the binary
    search takes the wide one."""
    assert lib.nsc_test_row_mode(C.byref(fov_params(lib, 128, (-24.8, 2.0)))) == 0
    assert lib.nsc_test_row_mode(C.byref(fov_params(lib, 128, (-25.0, 15.0)))) == 0
    assert lib.nsc_test_row_mode(C.byref(fov_params(lib, 128, (-60.0, 60.0)))) == 1


def test_128_rows_are_accepted_and_129_refused(lib):
    for rows in (65, 128):
        assert lib.nsc_workspace_bytes(10, C.byref(default_params(lib, n_elevation=rows))) > 0
        assert lib.nsc_anywidth_workspace_bytes(10, rows, C.byref(default_params(lib, n_azimuth=500))) > 0
        assert lib.nsc_test_row_mode(C.byref(default_params(lib, n_elevation=rows))) in (0, 1)
    bad = default_params(lib, n_elevation=129)
    assert lib.nsc_workspace_bytes(10, C.byref(bad)) == 0
    assert lib.nsc_anywidth_workspace_bytes(10, 129, C.byref(default_params(lib, n_azimuth=500))) == 0
    assert lib.nsc_anywidth_workspace_bytes(10, 16, C.byref(default_params(lib, n_azimuth=500, n_elevation=129))) == 0
    assert lib.nsc_test_row_mode(C.byref(bad)) == -4


def test_129_rows_refused_by_every_entry_point(lib):
    """Bad parameters are reported before any pointer is touched, so dummy pointers are safe."""
    bad = default_params(lib, n_elevation=129)
    good = default_params(lib)
    lut = orc.freq_to_bin(orc.OracleConfig()).numpy().astype(np.int32)
    P = C.c_void_p(16)
    assert lib.nsc_encode_batch(P, 4, P, 0, 1, C.byref(bad), lut.ctypes.data, P, P, 256, None) == -4
    assert lib.nsc_encode_batch_u16(P, 4, P, 0, 1, C.byref(bad), lut.ctypes.data, 1e-8, P, P, 256, None) == -4
    peers = (C.c_void_p * 1)(16)
    assert lib.nsc_encode_batch_peers(P, 4, P, 0, 1, C.byref(bad), lut.ctypes.data, peers, 1, 0, P, 256,
                                      None) == -4
    assert lib.nsc_project_batch(P, 4, P, 0, 1, C.byref(bad), 0, P, P, 256, None) == -4
    assert lib.nsc_project_intensity_batch(P, P, 0, 1, C.byref(bad), P, P, None) == -4
    assert lib.nsc_encode_range_images(P, 1, 129, C.byref(good), lut.ctypes.data, P, None) == -4
    assert lib.nsc_interpolate_range_images(P, 1, 129, 0, P, None) == -4
    wide = default_params(lib, n_azimuth=500, n_elevation=129)
    assert lib.nsc_anywidth_points(P, 4, P, 0, 1, C.byref(wide), None, None, P, 0, P, 1 << 20, None) == -4
    assert lib.nsc_anywidth_images(P, 1, 129, C.byref(default_params(lib, n_azimuth=500)), None, -1, None, P, P,
                                   1 << 20, None) == -4


def test_without_the_flag_the_envelope_stays_64_rows(lib):
    """A parameter block without NSC_FLAG_TALL_IMAGES (nsc_default_params leaves it clear) keeps the
    64-row envelope of earlier libraries at every entry point; with the flag, 64 rows are unchanged."""
    assert default_params(lib, flags=0).flags == 0
    plain = _lib.NscParams()
    lib.nsc_default_params(C.byref(plain))
    assert plain.flags == 0
    lut = orc.freq_to_bin(orc.OracleConfig()).numpy().astype(np.int32)
    P = C.c_void_p(16)
    for rows, want in ((64, True), (65, False), (128, False)):
        p = default_params(lib, n_elevation=rows, flags=0)
        assert (lib.nsc_workspace_bytes(10, C.byref(p)) > 0) == want
        assert (lib.nsc_test_row_mode(C.byref(p)) >= 0) == want
        assert (lib.nsc_anywidth_workspace_bytes(10, rows, C.byref(default_params(lib, n_azimuth=500, flags=0))) > 0) == want
        if not want:
            assert lib.nsc_encode_batch(P, 4, P, 0, 1, C.byref(p), lut.ctypes.data, P, P, 256, None) == -4
            assert lib.nsc_encode_batch_u16(P, 4, P, 0, 1, C.byref(p), lut.ctypes.data, 1e-8, P, P, 256, None) == -4
            assert lib.nsc_project_batch(P, 4, P, 0, 1, C.byref(p), 0, P, P, 256, None) == -4
            assert lib.nsc_project_intensity_batch(P, P, 0, 1, C.byref(p), P, P, None) == -4
            assert lib.nsc_encode_range_images(P, 1, rows, C.byref(default_params(lib, flags=0)), lut.ctypes.data, P,
                                               None) == -4
    for rows in (65, 128):
        p = default_params(lib, n_elevation=rows)
        assert lib.nsc_workspace_bytes(10, C.byref(p)) == 256       # tall images split no scan
