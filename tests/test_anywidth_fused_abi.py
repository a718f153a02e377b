"""CPU-only checks of the fused kernel for image widths other than 360 (csrc/nsc_anywidth.cu):
which calls it takes (nsc_test_anywidth_path, a host function of the arguments), and its
mixed-radix FFT run on the host (nsc_test_anywidth_fft) against numpy.fft.fft in float64
(no GPU compute calls)."""
import ctypes as C
import os

import numpy as np
import pytest

from neural_spectral_codec_b200 import _lib

SMEM_OPT_IN = 227 * 1024
FUSED_THREADS = 512
ENVELOPE_WIDTHS = [77, 90, 180, 500, 512, 720, 1024, 1800, 2048]


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.load()


def params(lib, **kw):
    p = _lib.NscParams()
    lib.nsc_default_params(C.byref(p))
    p.flags = _lib.FLAG_TALL_IMAGES
    for k, v in kw.items():
        setattr(p, k, v)
    return p


def max_prime(n):
    f, big = 2, 1
    while f * f <= n:
        while n % f == 0:
            big, n = f, n // f
        f += 1
    return max(big, n) if n > 1 else big


def layout_bytes(rows, W, T, n_bins, n_sig):
    def up(b):
        return (b + 15) & ~15
    return (up(FUSED_THREADS // 32 * 8) + up(rows * W * 4) + up(rows * ((W + 31) // 32) * 4) + up(W * 8)
            + 2 * up(n_sig * W * 8) + up(T * n_bins * 4) + up((n_bins + 1) * 4) + 2 * up(rows * 4))


def expected_path(rows, W, T, n_bins, want):
    return int(bool(want) and max_prime(W) <= 13 and layout_bytes(rows, W, T, n_bins, 1) <= SMEM_OPT_IN)


@pytest.mark.parametrize("W", ENVELOPE_WIDTHS + [1009, 2 * 17, 3 * 19, 4096, 4095, 2 * 2 * 2 * 23])
def test_selection_follows_factors_rows_and_shared_memory(lib, W):
    """The fused kernel for every call with a descriptor whose width factors into primes <= 13
    and whose image fits, across rows 1..128 with and without pooling; never without a
    descriptor (image-only and interpolation-only calls)."""
    for rows in (1, 2, 7, 8, 16, 31, 32, 33, 64, 65, 100, 128):
        for T in sorted({min(rows, 64), 16, 1}):
            n_bins = min(50, W // 2 + 1)
            p = params(lib, n_azimuth=W, n_elevation=rows, target_rows=T, n_bins=n_bins)
            for want in (0, 1):
                got = lib.nsc_test_anywidth_path(C.byref(p), rows, want)
                assert got == expected_path(rows, W, T, n_bins, want), (W, rows, T, want, got)


def test_selection_examples(lib):
    def path(W, rows, T=16, want=1, n_bins=None):
        p = params(lib, n_azimuth=W, n_elevation=rows, target_rows=T, n_bins=n_bins or min(50, W // 2 + 1))
        return lib.nsc_test_anywidth_path(C.byref(p), rows, want)
    for W in ENVELOPE_WIDTHS:
        assert path(W, 16) == 1, W
        assert path(W, 16, want=0) == 0, W
    assert path(1009, 16) == 0                     # a prime above 13
    assert path(4096, 64) == 0                     # a 1 MB image
    assert path(512, 128) == 0                     # 256 KB
    assert path(180, 128) == 1 and path(77, 128, T=8, n_bins=10) == 1
    assert path(512, 64) == 1 and path(1024, 32) == 1 and path(2048, 16) == 1


def test_selection_at_the_shared_memory_boundary(lib):
    """For each width, the largest row count whose one-pair layout fits takes the fused kernel,
    one row more takes the general kernel."""
    for W in (180, 500, 512, 720, 1024, 1800, 2048, 4096):
        n_bins = 50
        fits = [r for r in range(1, 129) if layout_bytes(r, W, 16 if r >= 16 else r, n_bins, 1) <= SMEM_OPT_IN]
        if not fits or fits[-1] == 128:
            continue
        last = fits[-1]
        for rows, want in ((last, 1), (last + 1, 0)):
            T = 16 if rows >= 16 else rows
            p = params(lib, n_azimuth=W, n_elevation=rows, target_rows=T, n_bins=n_bins)
            assert lib.nsc_test_anywidth_path(C.byref(p), rows, 1) == want, (W, rows)


def test_selection_reports_the_entry_points_status(lib):
    p = params(lib, n_azimuth=512)
    assert lib.nsc_test_anywidth_path(None, 16, 1) == -1
    bad = params(lib, n_azimuth=512)
    bad.struct_size = 4
    assert lib.nsc_test_anywidth_path(C.byref(bad), 16, 1) == -10
    assert lib.nsc_test_anywidth_path(C.byref(params(lib, n_azimuth=4097)), 16, 1) == -4
    assert lib.nsc_test_anywidth_path(C.byref(p), 0, 1) == -4
    assert lib.nsc_test_anywidth_path(C.byref(p), 129, 1) == -4
    assert lib.nsc_test_anywidth_path(C.byref(params(lib, n_azimuth=512, flags=0)), 65, 1) == -4


def fft_widths():
    return [w for w in range(2, 65) if max_prime(w) <= 13] + ENVELOPE_WIDTHS


def run_fft(lib, x):
    W = len(x)
    buf = np.empty(2 * W, np.float32)
    buf[0::2], buf[1::2] = x.real, x.imag
    out = np.empty(2 * W, np.float32)
    assert lib.nsc_test_anywidth_fft(W, buf.ctypes.data, out.ctypes.data) == 0
    return out[0::2].astype(np.float64) + 1j * out[1::2]


@pytest.mark.parametrize("W", fft_widths())
def test_fft_matches_numpy_in_float64(lib, W):
    rng = np.random.default_rng(W)
    x = (rng.standard_normal(W) + 1j * rng.standard_normal(W)).astype(np.complex64)
    ref = np.fft.fft(x.astype(np.complex128))
    got = run_fft(lib, x)
    assert np.abs(got - ref).max() <= 2e-6 * np.sqrt(W) * np.abs(x).max() * max(1.0, np.log2(W))
    assert np.linalg.norm(got - ref) <= 1e-6 * np.linalg.norm(ref)
    for k in (0, 1, W // 2, W - 1):                 # impulses: a pure exponential
        e = np.zeros(W, np.complex64)
        e[k] = 1.0 - 0.5j
        ref = np.fft.fft(e.astype(np.complex128))
        np.testing.assert_allclose(run_fft(lib, e), ref, rtol=0, atol=2e-6)


def test_fft_refuses_widths_outside_the_plan(lib):
    buf = np.zeros(2 * 4097, np.float32)
    for W in (0, 1, 17, 1009, 4097):
        assert lib.nsc_test_anywidth_fft(W, buf.ctypes.data, buf.ctypes.data) == -4, W
    assert lib.nsc_test_anywidth_fft(64, None, buf.ctypes.data) == -1
