"""CPU-only checks of the C-ABI library and the host logic (no GPU compute calls)."""
import ctypes as C
import glob
import os
import re

import numpy as np
import pytest
import torch

from conftest import GOLDEN_DIR, POINT_CASES, ROOT
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


def test_every_declared_symbol_is_exported(lib):
    header = open(os.path.join(ROOT, "include", "nsc_b200.h")).read()
    declared = set(re.findall(r"\b(nsc_[a-z0-9_]+)\s*\(", header))
    declared -= {"nsc_status", "nsc_params", "nsc_pipeline"}
    assert declared, "no declarations parsed"
    assert declared == set(_lib.SYMBOLS), declared ^ set(_lib.SYMBOLS)
    for name in declared:
        assert hasattr(lib, name)
    assert lib.nsc_abi_version() == _lib.NSC_ABI_VERSION == 2
    assert C.sizeof(_lib.NscParams) == default_params(lib).struct_size == 56


def test_default_params_are_the_reference_defaults(lib):
    p = default_params(lib)
    cfg = orc.OracleConfig()
    assert (p.n_elevation, p.n_azimuth, p.n_bins, p.target_rows, p.interpolate_empty) == (16, 360, 50, 16, 1)
    assert p.min_range == 1.0 and p.max_range == 80.0 and p.epsilon == np.float32(1e-8)
    assert p.el_min_rad == float(cfg.el_min) and p.el_max_rad == float(cfg.el_max)


@pytest.mark.parametrize("alpha,n_bins", [(2.0, 50), (1.0, 50), (3.5, 50), (2.0, 32), (0.5, 100), (2.0, 181)])
def test_c_freq_to_bin_equals_torch_table(lib, alpha, n_bins):
    """nsc_freq_to_bin (for non-Python callers) against the reference's torch formula."""
    p = default_params(lib, n_bins=n_bins, target_rows=16)
    lut = np.zeros(181, np.int32)
    assert lib.nsc_freq_to_bin(alpha, C.byref(p), lut.ctypes.data) == 0
    cfg = orc.OracleConfig(alpha=alpha, n_bins=n_bins)
    np.testing.assert_array_equal(lut, orc.freq_to_bin(cfg).numpy())


def test_python_mirror_table_and_attributes(lib):
    from neural_spectral_codec_b200 import SpectralEncoder
    enc = SpectralEncoder(n_elevation=16, n_azimuth=360, n_bins=50, alpha=2.0, learnable_alpha=True,
                          target_elevation_bins=16)
    g = np.load(os.path.join(GOLDEN_DIR, "hdl64_full.npz"))
    np.testing.assert_array_equal(enc.freq_to_bin(), g["freq_to_bin"])
    np.testing.assert_array_equal(enc._compute_bin_edges(enc.alpha).numpy(), g["bin_edges"])
    assert enc.output_dim == 800 and enc.n_freqs == 181
    assert isinstance(enc.alpha, torch.nn.Parameter) and enc.alpha.device.type == "cpu"
    assert enc.projector.n_elevation == 16 and enc.projector.max_range == 80.0
    assert enc.projector.elevation_min == np.deg2rad(-24.8)
    with torch.no_grad():
        enc.alpha.fill_(1.0)     # in-place update bumps the version counter -> table recomputed
    np.testing.assert_array_equal(enc.freq_to_bin(), orc.freq_to_bin(orc.OracleConfig(alpha=1.0)).numpy())
    buf = SpectralEncoder(learnable_alpha=False)
    assert not isinstance(buf.alpha, torch.nn.Parameter) and "alpha" in dict(buf.named_buffers())


def test_no_cpu_fallback(lib):
    from neural_spectral_codec_b200 import SpectralEncoder
    enc = SpectralEncoder(n_elevation=16)
    with pytest.raises(RuntimeError, match="no CPU implementation"):
        enc.encode_points(np.zeros((4, 4), np.float32))
    with pytest.raises(RuntimeError, match="no CPU implementation"):
        enc(torch.zeros(1, 16, 360))
    with pytest.raises(RuntimeError, match="no CPU implementation"):
        enc.encode_points_batch(torch.zeros(4, 4), torch.tensor([0, 4]))
    with pytest.raises(RuntimeError, match="no CPU implementation"):
        enc.projector.project(np.zeros((4, 4), np.float32), keep_intensity=False)


def test_product_package_never_imports_the_oracle():
    """oracle/ is test infrastructure: nothing under the product package may import it."""
    pat = re.compile(r"^\s*(from|import)\s+[\w.]*oracle", re.M)
    for path in glob.glob(os.path.join(ROOT, "neural_spectral_codec_b200", "**", "*.py"), recursive=True):
        assert not pat.search(open(path).read()), path


def test_argument_validation_without_a_device(lib):
    p = default_params(lib)
    lut = orc.freq_to_bin(orc.OracleConfig()).numpy().astype(np.int32)
    args = lambda pp=p, l=lut: (C.c_void_p(16), 4, C.c_void_p(16), 0, 1, C.byref(pp), l.ctypes.data,
                                C.c_void_p(16), C.c_void_p(16), 256, None)
    bad = default_params(lib, n_azimuth=359)
    assert lib.nsc_encode_batch(*args(pp=bad)) == -4
    bad = default_params(lib, n_elevation=65)
    assert lib.nsc_encode_batch(*args(pp=bad)) == -4
    bad = default_params(lib, target_rows=64, n_bins=181)
    assert lib.nsc_encode_batch(*args(pp=bad)) == -4
    bad = default_params(lib, struct_size=12)
    assert lib.nsc_encode_batch(*args(pp=bad)) == -10
    bl = lut.copy()
    bl[100] = 0
    assert lib.nsc_encode_batch(*args(l=bl)) == -5
    assert lib.nsc_encode_batch(C.c_void_p(16), 2, C.c_void_p(16), 0, 1, C.byref(p), lut.ctypes.data,
                                C.c_void_p(16), C.c_void_p(16), 256, None) == -2
    assert lib.nsc_encode_batch(C.c_void_p(20), 4, C.c_void_p(16), 0, 1, C.byref(p), lut.ctypes.data,
                                C.c_void_p(16), C.c_void_p(16), 256, None) == -7
    assert lib.nsc_encode_batch(C.c_void_p(16), 4, None, 0, 1, C.byref(p), lut.ctypes.data,
                                C.c_void_p(16), C.c_void_p(16), 256, None) == -1
    assert lib.nsc_encode_batch(C.c_void_p(16), 4, C.c_void_p(16), 0, 0, C.byref(p), lut.ctypes.data,
                                None, None, 0, None) == 0          # empty batch is a no-op
    assert lib.nsc_workspace_bytes(10, C.byref(p)) >= 8
    assert lib.nsc_strerror(-4).decode().startswith("nsc_params")
    assert lib.nsc_strerror(0).decode() == "ok"


def host_classify(lib, pts, **kw):
    p = default_params(lib, **kw)
    pts = np.ascontiguousarray(pts, np.float32)
    n = len(pts)
    row, col, keep = np.zeros(n, np.int32), np.zeros(n, np.int32), np.zeros(n, np.uint8)
    st = lib.nsc_test_host_classify(pts.ctypes.data, pts.shape[1], n, C.byref(p), row.ctypes.data,
                                    col.ctypes.data, keep.ctypes.data)
    assert st == 0
    return row, col, keep.astype(bool)


@pytest.mark.parametrize("name", POINT_CASES)
def test_point_function_matches_oracle_pixels(lib, name):
    """The kernel's per-point function (evaluated on the host through the test hook) keeps and
    drops exactly the oracle's points and assigns the same pixel, except for points within
    1e-5 rad of a row / column edge (BASELINE.json north_star)."""
    pts = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))["points"]
    E = 64 if name.startswith("elev64") else 16
    cfg = orc.OracleConfig(n_elevation=E)
    row, col, keep = host_classify(lib, pts, n_elevation=E)
    s = orc.spherical(pts, cfg)
    okeep = np.zeros(len(pts), bool)
    okeep[s["kept"]] = True
    np.testing.assert_array_equal(keep, okeep)
    if len(pts) == 0:
        return
    orow, ocol = np.full(len(pts), -1), np.full(len(pts), -1)
    orow[s["kept"]], ocol[s["kept"]] = s["row"], s["col"]
    d_az, d_el = orc.edge_distance(pts, cfg)
    clear = keep & (d_az > 1e-5) & (d_el > 1e-5)
    np.testing.assert_array_equal(row[clear], orow[clear])
    np.testing.assert_array_equal(col[clear], ocol[clear])
    assert ((row != orow) | (col != ocol)).sum() <= (~clear & keep).sum()


@pytest.mark.parametrize("er,rows,mode", [((-24.8, 2.0), 16, 0), ((-15.0, 15.0), 16, 0), ((-30.67, 10.67), 32, 0),
                                          ((-60.0, 60.0), 32, 1), ((-89.0, 89.0), 64, 1), ((-25.0, 15.0), 64, 0)])
def test_row_rules_on_other_fields_of_view(lib, er, rows, mode):
    p = default_params(lib, n_elevation=rows, el_min_rad=float(np.deg2rad(er[0])),
                       el_max_rad=float(np.deg2rad(er[1])))
    assert lib.nsc_test_row_mode(C.byref(p)) == mode
    rng = np.random.default_rng(rows)
    n = 200000
    az, el, r = rng.uniform(-np.pi, np.pi, n), rng.uniform(-1.5, 1.5, n), rng.uniform(0.5, 90, n)
    pts = np.stack([r * np.cos(el) * np.cos(az), r * np.cos(el) * np.sin(az), r * np.sin(el)], 1).astype(np.float32)
    cfg = orc.OracleConfig(n_elevation=rows, elevation_range=er)
    row, col, keep = host_classify(lib, pts, n_elevation=rows, el_min_rad=float(cfg.el_min), el_max_rad=float(cfg.el_max))
    s = orc.spherical(pts, cfg)
    okeep = np.zeros(n, bool)
    okeep[s["kept"]] = True
    np.testing.assert_array_equal(keep, okeep)
    orow, ocol = np.full(n, -1), np.full(n, -1)
    orow[s["kept"]], ocol[s["kept"]] = s["row"], s["col"]
    d_az, d_el = orc.edge_distance(pts, cfg)
    clear = keep & (d_az > 1e-5) & (d_el > 1e-5)
    np.testing.assert_array_equal(row[clear], orow[clear])
    np.testing.assert_array_equal(col[clear], ocol[clear])


def host_classify_cfg(lib, pts, cfg):
    return host_classify(lib, pts, n_elevation=cfg.n_elevation, el_min_rad=float(cfg.el_min),
                         el_max_rad=float(cfg.el_max), min_range=cfg.min_range, max_range=cfg.max_range)


# (elevation range, rows, min_range, max_range, row rule): both row rules, E = 1 and E = 2
HOST_CONFIGS = [((-24.8, 2.0), 16, 1.0, 80.0, 0), ((-15.0, 15.0), 16, 1.0, 80.0, 0), ((-60.0, 60.0), 32, 1.0, 80.0, 1),
                ((-89.0, 89.0), 64, 0.5, 120.0, 1), ((-30.0, 30.0), 1, 2.0, 50.0, 0), ((-30.0, 30.0), 2, 1.0, 80.0, 0)]


def host_config(lib, er, rows, lo, hi, mode):
    cfg = orc.OracleConfig(n_elevation=rows, elevation_range=er, min_range=lo, max_range=hi)
    p = default_params(lib, n_elevation=rows, el_min_rad=float(cfg.el_min), el_max_rad=float(cfg.el_max))
    assert lib.nsc_test_row_mode(C.byref(p)) == mode
    return cfg


@pytest.mark.parametrize("er,rows,lo,hi,mode", HOST_CONFIGS)
def test_near_axis_points_get_the_oracle_pixel(lib, er, rows, lo, hi, mode):
    """|x|, |y| in [1e-45, 1e-20] with z inside the range limits: points on the vertical axis's
    doorstep, kept, with the row clamped and the column of atan2(y, x). The octant reduction
    min(|x|,|y|) / max(|x|,|y|) must not depend on the scale of x and y (a floor of 1e-30 on the
    denominator once sent these points to arbitrary columns). No row edge is near; points within
    1e-5 rad of a column edge may take the column across it, every other one the oracle's."""
    from point_sets import across_edges, near_axis, oracle_pixels
    cfg = host_config(lib, er, rows, lo, hi, mode)
    pts = near_axis(np.random.default_rng(rows), 40000, cfg)
    row, col, keep = host_classify_cfg(lib, pts, cfg)
    okeep, orow, ocol, _, d_az, d_el = oracle_pixels(pts, cfg)
    assert okeep.all() and keep.all()
    assert (d_el > 1e-5).all()
    np.testing.assert_array_equal(row, orow)
    clear = d_az > 1e-5
    assert clear.sum() > 0.5 * len(pts)
    np.testing.assert_array_equal(col[clear], ocol[clear])
    _, col_x = across_edges(pts, cfg, orow, ocol)
    assert ((col == ocol) | (col == col_x))[~clear].all()


@pytest.mark.parametrize("er,rows,lo,hi,mode", HOST_CONFIGS)
def test_axes_and_signed_zeros_match_the_oracle_exactly(lib, er, rows, lo, hi, mode):
    """Points on the x, y and z axes with +0 and -0 in every coordinate, and the azimuth wrap
    (x < 0, y = +-0: atan2 = +-pi, the reference's column 0). They sit exactly on column edges,
    yet the pixel must be the oracle's with no excuse."""
    from point_sets import oracle_pixels, signed_zeros
    cfg = host_config(lib, er, rows, lo, hi, mode)
    pts = signed_zeros(cfg)
    row, col, keep = host_classify_cfg(lib, pts, cfg)
    okeep, orow, ocol, _, _, _ = oracle_pixels(pts, cfg)
    np.testing.assert_array_equal(keep, okeep)
    assert okeep.sum() >= len(pts) // 2
    np.testing.assert_array_equal(row[keep], orow[keep])
    np.testing.assert_array_equal(col[keep], ocol[keep])


@pytest.mark.parametrize("er,rows,lo,hi,mode", HOST_CONFIGS)
def test_adversarial_coordinates_keep_like_the_oracle_and_stay_in_the_image(lib, er, rows, lo, hi, mode):
    """NaN, +-Inf, subnormals, +-1e38 and coordinates whose squares overflow, alone in one
    coordinate of in-range points and in every triple: the keep/drop decision is the oracle's and
    every kept point gets 0 <= row < E, 0 <= column < 360."""
    from point_sets import adversarial, oracle_pixels
    cfg = host_config(lib, er, rows, lo, hi, mode)
    pts = adversarial(np.random.default_rng(7), 200, cfg)
    row, col, keep = host_classify_cfg(lib, pts, cfg)
    okeep = oracle_pixels(pts, cfg)[0]
    np.testing.assert_array_equal(keep, okeep)
    assert 0 < keep.sum() < len(pts)
    assert ((row[keep] >= 0) & (row[keep] < rows)).all()
    assert ((col[keep] >= 0) & (col[keep] < 360)).all()


@pytest.mark.parametrize("lo,hi", [(0.5, 120.0), (2.0, 50.0), (0.0, 30.0), (1.0, 80.0)])
def test_keep_drop_is_exact_for_other_range_limits(lib, lo, hi):
    """The float32 thresholds on s are derived per (min_range, max_range); the keep/drop decision
    must equal the oracle's test on sqrt(s) for ranges packed around both limits."""
    rng = np.random.default_rng(int(hi))
    n = 60000
    r = np.concatenate([lo + rng.normal(0, 2e-6, n // 3) * max(lo, 1.0), hi + rng.normal(0, 2e-6, n // 3) * hi,
                        rng.uniform(0.01, hi * 1.5, n - 2 * (n // 3))])
    az, el = rng.uniform(-np.pi, np.pi, n), rng.uniform(-0.4, 0.02, n)
    pts = np.stack([r * np.cos(el) * np.cos(az), r * np.cos(el) * np.sin(az), r * np.sin(el)], 1).astype(np.float32)
    cfg = orc.OracleConfig(min_range=lo, max_range=hi)
    _, _, keep = host_classify(lib, pts, min_range=lo, max_range=hi)
    okeep = np.zeros(n, bool)
    okeep[orc.spherical(pts, cfg)["kept"]] = True
    np.testing.assert_array_equal(keep, okeep)
    assert 0.1 * n < keep.sum() < 0.95 * n


def test_range_thresholds_are_exact_preimages(lib):
    """SURVEY.md 8(c) P2: the filter on s = x^2+y^2+z^2 must keep exactly the points whose
    float32 sqrt lies in [min_range, max_range], including the last ulps around 1 and 80."""
    f = np.float32
    vals = []
    for centre in (f(1.0), f(6400.0)):
        v = centre
        for _ in range(6):
            v = np.nextafter(v, f(0))
        for _ in range(13):
            vals.append(v)
            v = np.nextafter(v, f(1e9))
    s = np.array(vals, f)
    pts = np.stack([np.sqrt(s.astype(np.float64)), np.zeros_like(s, np.float64), np.zeros_like(s, np.float64)], 1)
    # build points whose float32 x*x reproduces s exactly where possible; otherwise skip
    x = pts[:, 0].astype(f)
    ok = (x * x) == s
    pts = np.stack([x, np.zeros_like(x), np.zeros_like(x)], 1)[ok]
    assert ok.sum() >= 8
    _, _, keep = host_classify(lib, pts)
    rng = np.sqrt(pts[:, 0] * pts[:, 0])
    np.testing.assert_array_equal(keep, (rng >= f(1.0)) & (rng <= f(80.0)))


def test_header_is_plain_c_and_the_c_demo_links(lib, tmp_path):
    """include/nsc_b200.h must be usable from C (the boundary is a C ABI, not C++): compile the
    example caller with gcc -std=c99 and link it against the shared library."""
    import subprocess
    exe = tmp_path / "c_abi_demo"
    cmd = ["gcc", "-std=c99", "-Wall", "-Werror", "-I" + os.path.join(ROOT, "include"),
           os.path.join(ROOT, "examples", "c_abi_demo.c"), "-L" + os.path.dirname(_lib.LIB_PATH), "-lnsc_b200",
           "-lm", "-Wl,-rpath," + os.path.dirname(_lib.LIB_PATH), "-o", str(exe)]
    r = subprocess.run(cmd, capture_output=True, text=True)
    assert r.returncode == 0, r.stderr
    # without a GPU the demo must fail with the library's CUDA status, not crash
    r = subprocess.run([str(exe)], capture_output=True, text=True)
    if not torch.cuda.is_available():
        assert r.returncode == 1 and "CUDA runtime error" in r.stderr
