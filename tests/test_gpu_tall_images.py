"""Range images of 65..128 rows on the GPU (one row per beam of a 128-beam sensor): the tall
encode kernels, their pooling before the spectrum, and every other entry point that takes rows,
against the oracle (which takes any n_elevation and pools with adaptive_avg_pool2d).

Tolerances as in test_gpu_parity.py: range images bit-exact once points within 1e-5 rad of an
edge are removed, and at most one differing pixel per such point otherwise; descriptors
allclose(rtol=1e-4, atol=1e-7) with relative L2 <= 1e-5."""
import ctypes as C

import numpy as np
import pytest
import torch

from neural_spectral_codec_b200 import SpectralEncoder, RangeImageProjector, interpolate_range_image, synth
from neural_spectral_codec_b200 import _lib
from oracle import nsc_oracle as orc

pytestmark = pytest.mark.gpu

RTOL, ATOL, L2REL = 1e-4, 1e-7, 1e-5
WIDE = (-60.0, 60.0)                  # a field of view that takes the binary row search
BEAM_S = synth.SensorShape("beam128_s", 128, -25.0, 15.0, 700)
HDL_S = synth.SensorShape("hdl64_s", 64, -24.8, 2.0, 900)


def assert_descriptor(got, ref):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    np.testing.assert_allclose(got, ref, rtol=RTOL, atol=ATOL)
    assert np.linalg.norm(got - ref) <= L2REL * np.linalg.norm(ref)


def encoder(rows, T=16, fov=(-24.8, 2.0), **kw):
    return SpectralEncoder(n_elevation=rows, n_azimuth=kw.pop("n_azimuth", 360), n_bins=kw.pop("n_bins", 50),
                           target_elevation_bins=T, elevation_range=fov, **kw).to("cuda")


def config(rows, T=16, fov=(-24.8, 2.0), **kw):
    return orc.OracleConfig(n_elevation=rows, target_elevation_bins=T, elevation_range=fov, **kw)


def batch(scans):
    offs = np.cumsum([0] + [len(s) for s in scans])
    return torch.from_numpy(np.concatenate(scans)).cuda(), torch.from_numpy(offs).cuda()


def scans(shape, first, n, cfg=None):
    out = [synth.make_scan(shape, first + i).numpy() for i in range(n)]
    return [orc.strip_ambiguous(s, cfg) for s in out] if cfg is not None else out


@pytest.mark.parametrize("shape", [BEAM_S, HDL_S], ids=lambda s: s.name)
@pytest.mark.parametrize("rows", [65, 96, 128])
def test_range_images_at_tall_rows(rows, shape):
    cfg = config(rows)
    proj = RangeImageProjector(n_elevation=rows, elevation_range=cfg.elevation_range)
    clean = scans(shape, 10, 3, cfg)
    pts, offs = batch(clean)
    got = proj.project_batch(pts, offs).cpu().numpy()
    filled = proj.project_batch(pts, offs, interpolate=True).cpu().numpy()
    for i, s in enumerate(clean):
        np.testing.assert_array_equal(got[i], orc.project(s, cfg))
        np.testing.assert_array_equal(filled[i], orc.interpolate_range_image(got[i]))
    raw = scans(shape, 20, 3)
    pts, offs = batch(raw)
    got = proj.project_batch(pts, offs).cpu().numpy()
    for i, s in enumerate(raw):
        d_az, d_el = orc.edge_distance(s, cfg)
        n_amb = int(((d_az <= 1e-5) | (d_el <= 1e-5)).sum())
        assert int((got[i] != orc.project(s, cfg)).sum()) <= n_amb


@pytest.mark.parametrize("interp", [True, False])
@pytest.mark.parametrize("fov", [(-25.0, 15.0), WIDE], ids=["poly", "search"])
@pytest.mark.parametrize("rows,T", [(128, 16), (128, 64), (100, 16), (96, 32), (65, 5)])
def test_descriptors_at_tall_rows(rows, T, fov, interp):
    cfg = config(rows, T, fov, interpolate_empty=interp)
    enc = encoder(rows, T, fov, interpolate_empty=interp)
    assert _lib.load().nsc_test_row_mode(C.byref(enc._params())) == (0 if fov != WIDE else 1)
    clean = scans(BEAM_S, 100 + rows, 3, cfg)
    got = enc.encode_points_batch(*batch(clean)).cpu().numpy()
    for i, s in enumerate(clean):
        assert_descriptor(got[i], orc.encode_points(s, cfg).numpy())


def test_largest_descriptor_at_128_rows():
    """T = 64, 64 bins (D = 4096): the largest histogram next to a 128-row image."""
    cfg = config(128, 64, n_bins=64)
    enc = encoder(128, 64, n_bins=64)
    clean = scans(BEAM_S, 300, 2, cfg)
    got = enc.encode_points_batch(*batch(clean)).cpu().numpy()
    for i, s in enumerate(clean):
        assert_descriptor(got[i], orc.encode_points(s, cfg).numpy())


def test_paths_agree_bit_for_bit_at_128_rows():
    """One scan, a small batch (cluster kernel), a batch larger than 2 x SMs (persistent kernel),
    the host pipeline and the uint16 epilogue all give the same rows."""
    from neural_spectral_codec_b200.quantization import HistogramQuantizer
    enc = encoder(128, 16, (-25.0, 15.0))
    shape = synth.SensorShape("beam128_xs", 128, -25.0, 15.0, 200)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = 2 * sms + 7
    host = scans(shape, 500, n)
    pts, offs = batch(host)
    big = enc.encode_points_batch(pts, offs)
    big_h = big.cpu().numpy()
    one = enc.encode_points(host[0]).cpu().numpy()
    np.testing.assert_array_equal(one, big_h[0])
    three = enc.encode_points_batch(*batch(host[1:4])).cpu().numpy()
    np.testing.assert_array_equal(three, big_h[1:4])
    np.testing.assert_array_equal(enc.encode_scans(host), big_h)
    q = enc.encode_points_batch(pts, offs, dtype=torch.uint16)
    np.testing.assert_array_equal(q.cpu().numpy(), HistogramQuantizer(big.shape[1]).quantize(big).cpu().numpy())
    q3 = enc.encode_points_batch(*batch(host[1:4]), dtype=torch.uint16)
    np.testing.assert_array_equal(q3.cpu().numpy(), q.cpu().numpy()[1:4])
    cfg = config(128, 16, (-25.0, 15.0))
    for i in (0, n - 1):
        ref = orc.encode_points(host[i], cfg).numpy()
        assert np.abs(big_h[i] - ref).max() < 1e-4


@pytest.mark.parametrize("T", [16, 64])
def test_forward_on_128_row_images(T):
    cfg = config(128, T)
    enc = encoder(128, T)
    g = torch.Generator().manual_seed(T)
    x = torch.rand(5, 128, 360, generator=g) * 40
    x[x < 4] = 0
    x[1, 50:90] = 0
    got = enc(x.cuda()).detach().cpu().numpy()
    ref = orc.encode_batch(x, cfg).numpy()
    for i in range(x.shape[0]):
        assert_descriptor(got[i], ref[i])


@pytest.mark.parametrize("method", ["linear", "nearest"])
def test_interpolate_128_row_images(method):
    rng = np.random.default_rng(7)
    imgs = rng.uniform(1, 50, (3, 128, 360)).astype(np.float32)
    imgs[rng.random(imgs.shape) < 0.3] = 0
    imgs[0, 10:20] = 0
    imgs[1, :5] = 0
    imgs[2, 120:] = 0
    got = interpolate_range_image(imgs, method=method)
    for i in range(3):
        np.testing.assert_array_equal(got[i], orc.interpolate_range_image(imgs[i], method))


def test_intensity_image_at_128_rows():
    cfg = config(128, fov=(-25.0, 15.0))
    proj = RangeImageProjector(n_elevation=128, elevation_range=cfg.elevation_range, device="cuda")
    s = scans(BEAM_S, 40, 1, cfg)[0]
    rng, inten = proj.project(s, keep_intensity=True)
    orng, ointen = orc.project_with_intensity(s, cfg)
    np.testing.assert_array_equal(rng, orng)
    np.testing.assert_array_equal(inten, ointen)


def test_general_kernel_at_128_rows():
    cfg = config(128, n_azimuth=500)
    enc = encoder(128, n_azimuth=500)
    clean = scans(synth.SensorShape("beam128_w", 128, -24.0, 1.5, 400), 60, 2, cfg)
    got = enc.encode_points_batch(*batch(clean)).cpu().numpy()
    for i, s in enumerate(clean):
        assert_descriptor(got[i], orc.encode_points(s, cfg).numpy())


def test_129_rows_fail_in_python():
    s = synth.make_scan(BEAM_S, 1).numpy()
    with pytest.raises(_lib.NscError):
        encoder(129).encode_points(s)
    with pytest.raises(ValueError):
        encoder(129, n_azimuth=500).encode_points(s)
