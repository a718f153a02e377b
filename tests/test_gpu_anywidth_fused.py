"""The fused kernel for image widths other than 360 (csrc/nsc_anywidth.cu) against the general
kernel on the same inputs. The product library runs the fused kernel; the tuning build, with
NSC_ANYWIDTH=0 in the environment at its first call, runs the general kernel for every call.

Bars: range images (projected and interpolated) bit-identical; descriptors allclose(rtol=1e-4,
atol=1e-7) with relative L2 <= 1e-5; calls outside the fused kernel's envelope bit-identical."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from neural_spectral_codec_b200 import SpectralEncoder, _lib, synth
from oracle import nsc_oracle as orc

pytestmark = pytest.mark.gpu

RTOL, ATOL, L2REL = 1e-4, 1e-7, 1e-5
WIDTHS = [77, 90, 180, 500, 512, 720, 1024, 2048]
ROWS = [(8, 8), (16, 16), (32, 16), (64, 16), (128, 16)]
SHAPES = [synth.HDL64, synth.HDL32, synth.BEAM128]
SMALL = synth.SensorShape("hdl64_small", 64, -24.8, 2.0, 300)
FOV = {"hdl64": (-24.8, 2.0), "hdl64_small": (-24.8, 2.0), "hdl32": (-30.67, 10.67), "beam128": (-25.0, 15.0)}

_GENERAL = []


def general_lib():
    """The tuning build with the fused kernel switched off (NSC_ANYWIDTH is read once, at the
    first call; the variable is restored so that no other test sees it)."""
    if not _GENERAL:
        old = os.environ.get("NSC_ANYWIDTH")
        os.environ["NSC_ANYWIDTH"] = "0"
        try:
            lib = C.CDLL(_lib.TUNE_LIB_PATH)
            for name, (res, args) in _lib.SYMBOLS.items():
                fn = getattr(lib, name)
                fn.restype, fn.argtypes = res, args
            p = encoder(16, 512)._params()
            assert lib.nsc_test_anywidth_path(C.byref(p), 16, 1) == 0
        finally:
            if old is None:
                del os.environ["NSC_ANYWIDTH"]
            else:
                os.environ["NSC_ANYWIDTH"] = old
        _GENERAL.append(lib)
    return _GENERAL[0]


def assert_descriptor(got, ref):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    np.testing.assert_allclose(got, ref, rtol=RTOL, atol=ATOL)
    assert np.linalg.norm(got - ref) <= L2REL * np.linalg.norm(ref)


def encoder(rows, W, T=16, fov=(-24.8, 2.0), **kw):
    return SpectralEncoder(n_elevation=rows, n_azimuth=W, n_bins=min(50, W // 2 + 1), target_elevation_bins=T,
                           elevation_range=fov, **kw).to("cuda")


def fused_applies(enc, rows=None):
    p = enc._params()
    return _lib.load().nsc_test_anywidth_path(C.byref(p), rows or p.n_elevation, 1) == 1


def batch(scans, stride=4):
    offs = np.cumsum([0] + [len(s) for s in scans])
    pts = np.concatenate(scans)[:, :stride] if scans else np.zeros((0, stride), np.float32)
    return torch.from_numpy(np.ascontiguousarray(pts)).cuda(), torch.from_numpy(offs).cuda()


def workspace(lib, n, rows, p, fill=0):
    nbytes = int(lib.nsc_anywidth_workspace_bytes(n, rows, C.byref(p)))
    return torch.full(((nbytes + 3) // 4,), fill, dtype=torch.int32, device="cuda"), nbytes


def run_points(lib, enc, pts, offs, stage, fill=0, stream=None):
    """nsc_anywidth_points with descriptors and the image at `stage`."""
    p, lut = enc._params(), enc.freq_to_bin()
    n, E, W = offs.numel() - 1, p.n_elevation, p.n_azimuth
    out = torch.full((n, enc.output_dim), -1.0, device="cuda")
    img = torch.full((n, E, W), -1.0, device="cuda")
    ws, nbytes = workspace(lib, n, E, p, fill)
    s = stream or torch.cuda.current_stream()
    torch.cuda.synchronize()
    st = lib.nsc_anywidth_points(pts.data_ptr(), pts.shape[1], offs.data_ptr(), 0, n, C.byref(p), lut.ctypes.data,
                                 out.data_ptr(), img.data_ptr(), stage, ws.data_ptr(), nbytes, s.cuda_stream)
    assert st == 0, st
    torch.cuda.synchronize()
    return out.cpu().numpy(), img.cpu().numpy()


def run_images(lib, enc, x, method=-1, fill=0):
    p, lut = enc._params(), enc.freq_to_bin()
    out = torch.full((x.shape[0], enc.output_dim), -1.0, device="cuda")
    ws, nbytes = workspace(lib, x.shape[0], x.shape[1], p, fill)
    st = lib.nsc_anywidth_images(x.data_ptr(), x.shape[0], x.shape[1], C.byref(p), lut.ctypes.data, method,
                                 out.data_ptr(), None, ws.data_ptr(), nbytes, torch.cuda.current_stream().cuda_stream)
    assert st == 0, st
    torch.cuda.synchronize()
    return out.cpu().numpy()


def compare_points(enc, scans, stride, interpolate):
    pts, offs = batch(scans, stride)
    stage = _lib.STAGE_INTERPOLATED if interpolate else _lib.STAGE_PROJECTED
    d_f, img_f = run_points(_lib.load(), enc, pts, offs, stage)
    d_g, img_g = run_points(general_lib(), enc, pts, offs, stage)
    np.testing.assert_array_equal(img_f, img_g)
    for i in range(len(scans)):
        assert_descriptor(d_f[i], d_g[i])
    return d_f, d_g


@pytest.mark.parametrize("rows,T", ROWS, ids=lambda v: str(v))
@pytest.mark.parametrize("W", WIDTHS)
def test_fused_equals_general_on_scans(W, rows, T):
    """Whole synthetic scans (edge points included): identical images at both stages, descriptors
    to the suite's bars; strides 3 and 4, interpolation on and off, three sensors."""
    k = WIDTHS.index(W) + rows
    shape = SHAPES[k % 3]
    for interpolate in (True, False):
        enc = encoder(rows, W, T, FOV[shape.name], interpolate_empty=interpolate)
        if not fused_applies(enc):
            pytest.skip(f"{rows} x {W} does not fit the fused kernel's shared memory")
        scans = [synth.make_scan(shape, 40 + i).numpy() for i in range(3)]
        compare_points(enc, scans, 3 + (k + interpolate) % 2, interpolate)


@pytest.mark.parametrize("n", [1, 3, 148, 600])
def test_batches_with_empty_and_filtered_scans(n):
    """Batch sizes around the grid (one CTA per SM); empty scans and scans whose points are all
    out of range give the uniform row, in both kernels."""
    enc = encoder(16, 512, fov=FOV["hdl64_small"])
    assert fused_applies(enc)
    scans = [synth.make_scan(SMALL, 100 + i).numpy() for i in range(n)]
    special = {}
    if n >= 3:
        special = {1: np.zeros((0, 4), np.float32), n - 1: scans[n - 1] * np.float32(1e3)}
        for i, s in special.items():
            scans[i] = s
    d_f, _ = compare_points(enc, scans, 4, True)
    uniform = np.float32(1.0) / np.float32(enc.output_dim)
    for i in special:
        assert (d_f[i] == uniform).all(), i


def test_workspace_prefilled_and_non_default_stream():
    """The fused kernel needs no zeroed workspace and follows the caller's stream."""
    enc = encoder(32, 1024, 16, FOV["hdl32"])
    assert fused_applies(enc)
    pts, offs = batch([synth.make_scan(synth.HDL32, 7 + i).numpy() for i in range(5)])
    lib = _lib.load()
    ref = run_points(lib, enc, pts, offs, _lib.STAGE_INTERPOLATED)
    s = torch.cuda.Stream()
    got = run_points(lib, enc, pts, offs, _lib.STAGE_INTERPOLATED, fill=-1, stream=s)
    np.testing.assert_array_equal(got[0], ref[0])
    np.testing.assert_array_equal(got[1], ref[1])


def random_images(n, rows, W, seed):
    rng = np.random.default_rng(seed)
    x = rng.uniform(1, 60, (n, rows, W)) * (rng.uniform(0, 1, (n, rows, W)) > 0.4)
    x[0, 2:5] = 0                              # empty rows
    x[min(1, n - 1)] = 0                       # an empty image
    return torch.from_numpy(x.astype(np.float32)).cuda()


@pytest.mark.parametrize("W", WIDTHS)
def test_forward_and_interpolated_images(W):
    """forward() (no interpolation, as the reference's), and the C entry with linear and nearest
    interpolation before the descriptor."""
    enc = encoder(32, W, 16)
    if not fused_applies(enc):
        pytest.skip("does not fit")
    x = random_images(6, 32, W, W)
    fwd = enc(x).cpu().numpy()
    for method in (-1, 0, 1):
        got = run_images(_lib.load(), enc, x, method)
        ref = run_images(general_lib(), enc, x, method)
        for i in range(len(x)):
            assert_descriptor(got[i], ref[i])
        if method == -1:
            np.testing.assert_array_equal(fwd, got)


@pytest.mark.parametrize("W", [180, 1024])
def test_encode_scans_matches_general(W):
    enc = encoder(16, W, 16, FOV["hdl64"])
    scans = [synth.make_scan(synth.HDL64, 60 + i).numpy() for i in range(4)]
    got = enc.encode_scans(scans)
    pts, offs = batch(scans)
    ref, _ = run_points(general_lib(), enc, pts, offs, _lib.STAGE_INTERPOLATED)
    for i in range(len(scans)):
        assert_descriptor(got[i], ref[i])


@pytest.mark.parametrize("W,rows", [(1009, 16), (4096, 64), (512, 128)])
def test_outside_the_envelope_is_the_general_kernel(W, rows):
    """A prime width above 13 and images too large for shared memory keep the general kernel:
    the product library's output equals the general kernel's bit for bit."""
    enc = encoder(rows, W, 16, FOV["beam128"])
    assert not fused_applies(enc)
    pts, offs = batch([synth.make_scan(SMALL, 5 + i).numpy() for i in range(2)])
    got = run_points(_lib.load(), enc, pts, offs, _lib.STAGE_INTERPOLATED)
    ref = run_points(general_lib(), enc, pts, offs, _lib.STAGE_INTERPOLATED)
    np.testing.assert_array_equal(got[0], ref[0])
    np.testing.assert_array_equal(got[1], ref[1])


@pytest.mark.parametrize("W", [90, 500, 2048])
def test_rolling_columns_keeps_the_descriptor(W):
    """|FFT| is invariant under a circular shift of the columns."""
    enc = encoder(16, W, 16)
    x = random_images(3, 16, W, 7)
    base = enc(x).cpu().numpy()
    for shift in (1, W // 3, W - 1):
        np.testing.assert_allclose(enc(torch.roll(x, shift, dims=2)).cpu().numpy(), base, rtol=0, atol=1e-6)


@pytest.mark.parametrize("W", [180, 512, 1024, 2048])
def test_error_against_float64_is_no_worse_than_the_reference(W):
    """As test_gpu_parity's bar at 360 columns: the fused kernel is no further from a float64
    evaluation than the reference's own float32 path."""
    kw = dict(n_elevation=16, n_azimuth=W, n_bins=50, target_elevation_bins=16)
    cfg = orc.OracleConfig(**kw)
    pts = orc.strip_ambiguous(synth.make_scan(synth.HDL64, 3).numpy(), cfg)
    truth = orc.descriptor_f64(pts, cfg)
    ref = orc.encode_points(pts, cfg).numpy().astype(np.float64)
    enc = SpectralEncoder(**kw).to("cuda")
    assert fused_applies(enc)
    got = enc.encode_points(pts).cpu().numpy().astype(np.float64)
    err_ref, err_gpu = np.abs(ref - truth).max(), np.abs(got - truth).max()
    assert err_gpu <= 2.0 * err_ref + 1e-9, (err_gpu, err_ref)
    assert np.linalg.norm(got - truth) <= 2.0 * np.linalg.norm(ref - truth) + 1e-9
