"""Image widths other than 360 from host memory to the wire format: the uint16 epilogue of both
kernels of csrc/nsc_anywidth.cu (nsc_anywidth_points_u16) and the host-buffer pipeline at those
widths. Every comparison is bit for bit: uint16 rows against nsc_quantize_histograms /
HistogramQuantizer of nsc_anywidth_points' float32 rows for the same call, pipeline rows against
the device entry points on the same scans."""
import ctypes as C

import numpy as np
import pytest
import torch

from neural_spectral_codec_b200 import SpectralEncoder, _lib, synth
from neural_spectral_codec_b200.quantization import HistogramQuantizer

pytestmark = pytest.mark.gpu

SMALL = synth.SensorShape("hdl64_small", 64, -24.8, 2.0, 300)
FUSED = [(16, 180), (16, 500), (16, 512), (16, 1024), (16, 2048), (16, 77), (64, 512), (128, 180)]
GENERAL = [(16, 1009), (64, 1024), (128, 2048)]


def encoder(rows, W, T=16, interpolate=True):
    return SpectralEncoder(n_elevation=rows, n_azimuth=W, n_bins=min(50, W // 2 + 1), target_elevation_bins=min(T, rows),
                           elevation_range=(-24.8, 2.0), interpolate_empty=interpolate).to("cuda")


def fused(enc):
    return _lib.load().nsc_test_anywidth_path(C.byref(enc._params()), enc.n_elevation, 1)


def scans_for(n, seed, special=True, shape=SMALL):
    scans = [synth.make_scan(shape, seed + i).numpy() for i in range(n)]
    if special and n >= 3:
        scans[1] = np.zeros((0, 4), np.float32)              # empty: the uniform row
        scans[n - 1] = scans[n - 1] * np.float32(1e3)        # every point out of range
    return scans


def device_batch(scans, stride=4):
    offs = np.cumsum([0] + [len(s) for s in scans])
    pts = np.concatenate(scans)[:, :stride] if scans else np.zeros((0, stride), np.float32)
    return torch.from_numpy(np.ascontiguousarray(pts)).cuda(), torch.from_numpy(offs).cuda()


def workspace(lib, n, p, fill=0):
    nbytes = int(lib.nsc_anywidth_workspace_bytes(n, p.n_elevation, C.byref(p)))
    return torch.full(((nbytes + 3) // 4,), fill, dtype=torch.int32, device="cuda"), nbytes


def run_f32(enc, pts, offs):
    lib, p, lut = _lib.load(), enc._params(), enc.freq_to_bin()
    n = offs.numel() - 1
    out = torch.full((n, enc.output_dim), -1.0, device="cuda")
    ws, nbytes = workspace(lib, n, p)
    st = lib.nsc_anywidth_points(pts.data_ptr(), pts.shape[1], offs.data_ptr(), 0, n, C.byref(p), lut.ctypes.data,
                                 out.data_ptr(), None, _lib.STAGE_INTERPOLATED, ws.data_ptr(), nbytes,
                                 torch.cuda.current_stream().cuda_stream)
    assert st == 0, st
    return out


def run_u16(enc, pts, offs, q_eps=1e-8, fill=0, stream=None, misalign=False):
    """nsc_anywidth_points_u16 into a buffer pre-filled with 0xAAAA; misalign: rows start 2 bytes
    past a 16-byte boundary."""
    lib, p, lut = _lib.load(), enc._params(), enc.freq_to_bin()
    n, D = offs.numel() - 1, enc.output_dim
    off = 1 if misalign else 0
    buf = torch.full((n * D + 8,), -0x5556, dtype=torch.int16, device="cuda")      # 0xAAAA
    ws, nbytes = workspace(lib, n, p, fill)
    s = stream or torch.cuda.current_stream()
    torch.cuda.synchronize()
    st = lib.nsc_anywidth_points_u16(pts.data_ptr(), pts.shape[1], offs.data_ptr(), 0, n, C.byref(p),
                                     lut.ctypes.data, q_eps, buf.data_ptr() + 2 * off, ws.data_ptr(), nbytes,
                                     s.cuda_stream)
    assert st == 0, st
    torch.cuda.synchronize()
    host = buf.cpu().numpy().view(np.uint16)
    assert (host[:off] == 0xAAAA).all() and (host[off + n * D:] == 0xAAAA).all()   # nothing written outside
    return host[off:off + n * D].reshape(n, D)


def quantise(rows, q_eps=1e-8):
    lib = _lib.load()
    q = torch.empty(rows.shape, dtype=torch.uint16, device="cuda")
    st = lib.nsc_quantize_histograms(rows.data_ptr(), rows.shape[0], rows.shape[1], q_eps, q.data_ptr(),
                                     torch.cuda.current_stream().cuda_stream)
    assert st == 0, st
    return q


def check_u16(enc, scans, stride=4, q_eps=1e-8, **kw):
    pts, offs = device_batch(scans, stride)
    ref_f = run_f32(enc, pts, offs)
    ref = quantise(ref_f, q_eps).cpu().numpy()
    got = run_u16(enc, pts, offs, q_eps, **kw)
    np.testing.assert_array_equal(got, ref)
    if q_eps == 1e-8 and len(scans):
        np.testing.assert_array_equal(got, HistogramQuantizer(enc.output_dim).quantize(ref_f.cpu().numpy()))
    sums = got.astype(np.int64).sum(axis=1)
    assert ((sums == 65535) | (sums == 0)).all()
    return got


@pytest.mark.parametrize("rows,W", FUSED + GENERAL, ids=lambda v: str(v))
def test_u16_rows_equal_the_quantised_float_rows(rows, W):
    """Both strides, interpolation on and off, q_epsilon 1e-8 and 0, empty and filtered scans."""
    for k, interpolate in enumerate((True, False)):
        enc = encoder(rows, W, interpolate=interpolate)
        assert fused(enc) == int((rows, W) in FUSED)
        scans = scans_for(4, 10 * W + rows + k)
        for stride in (3, 4):
            for q_eps in (1e-8, 0.0):
                got = check_u16(enc, scans, stride, q_eps)
                if interpolate and q_eps:
                    assert (got[1] == got[3]).all()      # the empty and the filtered scan: the uniform row


@pytest.mark.parametrize("n", [1, 2, 148, 297, 600])
def test_u16_batch_sizes_workspace_stream_and_alignment(n):
    enc = encoder(16, 1024)
    scans = scans_for(n, 500)
    check_u16(enc, scans)
    check_u16(enc, scans, fill=-1, stream=torch.cuda.Stream(), misalign=True)


def test_u16_general_kernel_workspace_stream_and_alignment():
    enc = encoder(16, 1009)
    check_u16(enc, scans_for(5, 900), fill=-1, stream=torch.cuda.Stream(), misalign=True)


def test_u16_takes_the_float_calls_kernel_at_the_shared_memory_boundary():
    """The configs of test_anywidth_fused_abi's boundary test, on both sides: the uint16 rows are
    those of the float call's kernel (a different kernel would quantise different floats)."""
    def up(b):
        return (b + 15) & ~15

    def layout_bytes(rows, W, T, n_bins, n_sig):          # test_anywidth_fused_abi's model of the layout
        return (up(512 // 32 * 8) + up(rows * W * 4) + up(rows * ((W + 31) // 32) * 4) + up(W * 8)
                + 2 * up(n_sig * W * 8) + up(T * n_bins * 4) + up((n_bins + 1) * 4) + 2 * up(rows * 4))
    SMEM_OPT_IN = 227 * 1024
    lib = _lib.load()
    for W in (180, 500, 512, 720, 1024, 1800, 2048, 4096):
        fits = [r for r in range(1, 129) if layout_bytes(r, W, 16 if r >= 16 else r, 50, 1) <= SMEM_OPT_IN]
        if not fits or fits[-1] == 128:
            continue
        for rows, want in ((fits[-1], 1), (fits[-1] + 1, 0)):
            enc = SpectralEncoder(n_elevation=rows, n_azimuth=W, n_bins=50, target_elevation_bins=min(16, rows),
                                  elevation_range=(-24.8, 2.0)).to("cuda")
            assert lib.nsc_test_anywidth_path(C.byref(enc._params()), rows, 1) == want
            check_u16(enc, scans_for(2, W + rows, special=False))


# ---- the host-buffer pipeline ------------------------------------------------------------------

def create(chunk, n_buffers):
    h = C.c_void_p()
    assert _lib.load().nsc_pipeline_create(chunk, n_buffers, torch.cuda.current_device(), C.byref(h)) == 0
    return h


def pipeline_rows(pl, enc, scans, u16, as_list, stride=4):
    lib, p, lut = _lib.load(), enc._params(), enc.freq_to_bin()
    n = len(scans)
    out = np.full((n, enc.output_dim), 0xAAAA if u16 else -1, np.uint16 if u16 else np.float32)
    arrs = [np.ascontiguousarray(s[:, :stride]) for s in scans]
    if as_list:
        ptrs = (C.c_void_p * n)(*[a.ctypes.data for a in arrs])
        counts = np.array([len(a) for a in arrs], np.int64)
        args = (pl, ptrs, counts.ctypes.data, stride, n, C.byref(p), lut.ctypes.data)
        name = "nsc_pipeline_encode_scans"
    else:
        pts = np.concatenate(arrs) if arrs else np.zeros((0, stride), np.float32)
        offs = np.cumsum([0] + [len(a) for a in arrs]).astype(np.int64)
        args = (pl, pts.ctypes.data, stride, pts.shape[0], offs.ctypes.data, n, C.byref(p), lut.ctypes.data)
        name = "nsc_pipeline_encode"
    if u16:
        name, args = name + "_u16", args + (1e-8,)
    st = getattr(lib, name)(*args, out.ctypes.data)
    return st, out


def device_rows(enc, scans, u16, stride=4):
    pts, offs = device_batch(scans, stride)
    f = run_f32(enc, pts, offs)
    return run_u16(enc, pts, offs) if u16 else f.cpu().numpy()


@pytest.mark.parametrize("n_buffers", [1, 2, 3, 4])
@pytest.mark.parametrize("rows,W", [(16, 1024), (64, 1024), (16, 77)], ids=lambda v: str(v))
def test_pipeline_rows_equal_the_device_entry(rows, W, n_buffers):
    """Concatenated buffer and list of arrays, float32 and uint16, small chunks that force many
    of them (the rows do not depend on how the scans are chunked)."""
    enc = encoder(rows, W)
    scans = scans_for(40, 70 + n_buffers)
    pl = create(40000, n_buffers)                             # two or three scans per chunk
    try:
        for u16 in (False, True):
            ref = device_rows(enc, scans, u16, stride=3 + n_buffers % 2)
            for as_list in (False, True):
                st, got = pipeline_rows(pl, enc, scans, u16, as_list, stride=3 + n_buffers % 2)
                assert st == 0, st
                np.testing.assert_array_equal(got, ref)
    finally:
        _lib.load().nsc_pipeline_destroy(pl)


def test_pipeline_crosses_the_1024_scan_chunk_bound():
    enc = encoder(16, 512)
    rng = np.random.default_rng(3)
    base = synth.make_scan(SMALL, 1).numpy()
    scans = [base[rng.integers(0, len(base), int(rng.integers(0, 60)))] for _ in range(2500)]
    pl = create(1 << 20, 2)
    try:
        for u16 in (False, True):
            ref = device_rows(enc, scans, u16)
            for as_list in (False, True):
                st, got = pipeline_rows(pl, enc, scans, u16, as_list)
                assert st == 0
                np.testing.assert_array_equal(got, ref)
    finally:
        _lib.load().nsc_pipeline_destroy(pl)


def test_pipeline_refuses_an_oversized_scan_before_copying():
    enc = encoder(16, 1024)
    scans = scans_for(3, 5, special=False)
    pl = create(len(scans[0]) - 1, 2)
    try:
        for u16 in (False, True):
            for as_list in (False, True):
                st, out = pipeline_rows(pl, enc, scans, u16, as_list)
                assert st == -6
                assert (out == (0xAAAA if u16 else -1)).all()
    finally:
        _lib.load().nsc_pipeline_destroy(pl)


def test_one_pipeline_across_widths_and_workspace_growth():
    """360 -> 1024 -> 64 x 1024 (the general kernel's larger scratch) -> 360 on one pipeline."""
    pl = create(1 << 20, 2)
    try:
        for rows, W in ((16, 360), (16, 1024), (64, 1024), (16, 360)):
            enc = encoder(rows, W)
            scans = scans_for(300, W + rows)
            for u16 in (False, True):
                st, got = pipeline_rows(pl, enc, scans, u16, as_list=True)
                assert st == 0
                if W == 360:
                    pts, offs = device_batch(scans)
                    ref = enc.encode_points_batch(pts, offs, dtype=torch.uint16 if u16 else torch.float32)
                    np.testing.assert_array_equal(got, ref.cpu().numpy())
                else:
                    np.testing.assert_array_equal(got, device_rows(enc, scans, u16))
    finally:
        _lib.load().nsc_pipeline_destroy(pl)


def test_encode_scan_on_a_side_stream_mixed_with_batches():
    lib = _lib.load()
    enc = encoder(64, 1024)
    p, lut = enc._params(), enc.freq_to_bin()
    scans = scans_for(12, 40)
    ref = device_rows(enc, scans, False)
    pl = create(1 << 18, 3)
    side = torch.cuda.Stream()
    try:
        outs = []
        for i, s in enumerate(scans):
            d = torch.full((enc.output_dim,), -1.0, device="cuda")
            a = np.ascontiguousarray(s)
            with torch.cuda.stream(side):
                assert lib.nsc_pipeline_encode_scan(pl, a.ctypes.data, 4, len(a), C.byref(p), lut.ctypes.data,
                                                    d.data_ptr(), side.cuda_stream) == 0
            outs.append(d)
            if i % 4 == 3:
                st, got = pipeline_rows(pl, enc, scans, False, as_list=i % 8 == 3)
                assert st == 0
                np.testing.assert_array_equal(got, ref)
        side.synchronize()
        np.testing.assert_array_equal(torch.stack(outs).cpu().numpy(), ref)
    finally:
        lib.nsc_pipeline_destroy(pl)


@pytest.mark.parametrize("rows,W", [(16, 1024), (16, 1009), (128, 180)], ids=lambda v: str(v))
def test_python_host_calls_equal_the_device_batch(rows, W):
    enc = encoder(rows, W)
    scans = scans_for(7, 3 * W)
    pts, offs = device_batch(scans)
    for dtype, tdtype in ((np.float32, torch.float32), (np.uint16, torch.uint16)):
        ref = enc.encode_points_batch(pts, offs, dtype=tdtype).cpu().numpy()
        np.testing.assert_array_equal(enc.encode_scans(scans, dtype=dtype), ref)
        cat = np.concatenate(scans)
        np.testing.assert_array_equal(enc.encode_scans((cat, offs.cpu().numpy()), dtype=dtype), ref)
        np.testing.assert_array_equal(enc.encode_scans(scans, dtype=dtype, max_chunk_points=len(scans[0])), ref)
    ref = enc.encode_points_batch(pts, offs).cpu().numpy()
    for i, s in enumerate(scans):
        np.testing.assert_array_equal(enc.encode_points(s).cpu().numpy(), ref[i])
