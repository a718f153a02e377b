"""uint16 wire format straight out of the encode kernels (nsc_encode_batch_u16 and the *_u16
pipeline entry points): for every kernel, geometry and store path, the integers equal
HistogramQuantizer.quantize applied to the float32 descriptors of the same call, and a sample of
rows equals the NumPy oracle of the reference quantiser. Run on the B200 box (148 SMs): batch
sizes are picked so that each encode kernel runs."""
import ctypes as C
import os

import numpy as np
import pytest
import torch

from conftest import GOLDEN_DIR, POINT_CASES
from oracle import quantization_oracle as qo

pytestmark = pytest.mark.gpu

CTOR = {"elev64_pooled": dict(n_elevation=64), "elev64_sparse": dict(n_elevation=64),
        "no_interp": dict(interpolate_empty=False)}
SMALL = ("s", 64, -24.8, 2.0, 700)    # 64 rings x 700 azimuth steps: small scans, quick batches


def make_encoder(**kw):
    from neural_spectral_codec_b200 import SpectralEncoder
    args = dict(n_elevation=16, n_azimuth=360, n_bins=50, alpha=2.0, learnable_alpha=True,
                target_elevation_bins=16)
    args.update(kw)
    return SpectralEncoder(**args).to("cuda")


def small_batch(first, n, device="cuda"):
    from neural_spectral_codec_b200 import synth
    return synth.make_batch(synth.SensorShape(*SMALL), first, n, device=device)


def quantize(rows, epsilon=1e-8):
    from neural_spectral_codec_b200.quantization import HistogramQuantizer
    return HistogramQuantizer(rows.shape[1], epsilon=epsilon).quantize(rows)


def same(a, b):
    """torch.equal for uint16 CUDA tensors (compared as their int16 bits)."""
    return a.dtype == b.dtype == torch.uint16 and torch.equal(a.view(torch.int16), b.view(torch.int16))


def assert_wire_rows(enc, pts, offs, sample=(0, -1)):
    """uint16 encode == quantize(float32 encode) for every row, and == the oracle on a sample."""
    q = enc.encode_points_batch(pts, offs, dtype=torch.uint16)
    f = enc.encode_points_batch(pts, offs)
    assert q.dtype == torch.uint16 and q.shape == f.shape and q.is_cuda
    assert same(q, quantize(f))
    qh, fh = q.cpu().numpy(), f.cpu().numpy()
    for i in sample:
        np.testing.assert_array_equal(qh[i], qo.quantize(fh[i]))
    sums = qh.astype(np.int64).sum(1)
    assert ((sums == 65535) | (sums == 0)).all()
    return qh, fh


@pytest.mark.parametrize("name", POINT_CASES)
def test_golden_cases(name):
    """One scan per call (cluster kernel), 3-float points for xyz_only, 64 -> 16 pooled rows, the
    uniform rows of empty and fully filtered scans."""
    g = np.load(os.path.join(GOLDEN_DIR, name + ".npz"))
    enc = make_encoder(**CTOR.get(name, {}))
    pts = torch.from_numpy(np.ascontiguousarray(g["points"], np.float32)).cuda()
    if pts.shape[1] > 4:
        pts = pts[:, :3].contiguous()
    offs = torch.tensor([0, pts.shape[0]])
    qh, fh = assert_wire_rows(enc, pts, offs)
    if name in ("empty", "all_out_of_range"):
        assert (fh == np.float32(1.0 / 800)).all()
    # the same scan inside a batch of 170 (warp-specialised kernel, tail-split last wave)
    bp, bo = small_batch(40, 169)
    allp = torch.cat([bp[:, :pts.shape[1]], pts]).contiguous()
    allo = torch.cat([bo.cpu(), torch.tensor([bo[-1].item() + pts.shape[0]])])
    qb, _ = assert_wire_rows(enc, allp, allo, sample=(0, 168, 169))
    np.testing.assert_array_equal(qb[-1], qh[0])


@pytest.mark.parametrize("n", [1, 2, 18, 170, 296])
def test_batch_sizes_reach_every_kernel(n):
    """1, 2, 18: clusters of 8 (cluster kernel); 170: warp-specialised with the last 22 scans split
    over the grid; 296: warp-specialised, two full waves. Empty scans inside the batch."""
    pts, offs = small_batch(7, n)
    offs = offs.cpu()
    if n >= 18:                       # scans 3 and n - 1 empty: their rows are the uniform descriptor
        cnt = torch.diff(offs)
        keep = torch.ones(pts.shape[0], dtype=torch.bool)
        for i in (3, n - 1):
            keep[offs[i]:offs[i + 1]] = False
            cnt[i] = 0
        pts = pts[keep.cuda()].contiguous()
        offs = torch.cat([torch.zeros(1, dtype=torch.int64), torch.cumsum(cnt, 0)])
    enc = make_encoder()
    qh, fh = assert_wire_rows(enc, pts, offs, sample=(0, n // 2, n - 1))
    if n >= 18:
        assert (fh[3] == np.float32(1.0 / 800)).all()
        np.testing.assert_array_equal(qh[3], qo.quantize(fh[3]))


def test_generic_kernel_with_three_float_points():
    """3-float points never take the warp-specialised kernel: 300 scans run the generic one."""
    pts, offs = small_batch(300, 300)
    assert_wire_rows(make_encoder(), pts[:, :3].contiguous(), offs, sample=(0, 150, 299))


def test_plain_store_paths():
    """2 D % 16 != 0 (n_bins 45, 3 rows: D = 135) and a destination one element off 16 bytes take
    plain stores instead of the bulk copy; a pooled geometry with D % 8 == 0 the bulk one."""
    pts, offs = small_batch(11, 170)
    for kw in (dict(n_bins=45, target_elevation_bins=3), dict(n_elevation=40, target_elevation_bins=16, n_bins=30)):
        enc = make_encoder(**kw)
        assert_wire_rows(enc, pts, offs)
        assert_wire_rows(enc, pts[:offs[2]], offs[:3])
    enc = make_encoder()
    want = quantize(enc.encode_points_batch(pts, offs))
    for n in (170, 2):
        buf = torch.zeros(n * 800 + 1, dtype=torch.uint16, device="cuda")
        view = buf[1:].view(n, 800)
        assert view.data_ptr() % 16 != 0
        got = enc.encode_points_batch(pts[:offs[n]], offs[:n + 1], out=view, dtype=torch.uint16)
        assert got.data_ptr() == view.data_ptr()
        assert same(view, want[:n]) and buf[:1].view(torch.int16).item() == 0
    with pytest.raises(ValueError):
        enc.encode_points_batch(pts, offs, out=torch.empty(170, 800, device="cuda"), dtype=torch.uint16)


@pytest.mark.parametrize("eps", [1e-8, 0.0])
def test_quantiser_epsilon_through_the_c_abi(eps):
    from neural_spectral_codec_b200 import _lib
    lib = _lib.load()
    enc = make_encoder()
    p, lut = enc._params(), enc.freq_to_bin()
    for n in (2, 170):
        pts, offs = small_batch(21, n)
        ws = torch.zeros(1 << 20, dtype=torch.int32, device="cuda")
        out = torch.empty((n, 800), dtype=torch.uint16, device="cuda")
        st = lib.nsc_encode_batch_u16(pts.data_ptr(), 4, offs.data_ptr(), 0, n, C.byref(p), lut.ctypes.data, eps,
                                      out.data_ptr(), ws.data_ptr(), ws.numel() * 4,
                                      torch.cuda.current_stream().cuda_stream)
        assert st == 0
        f = enc.encode_points_batch(pts, offs)
        assert same(out, quantize(f, epsilon=eps))
        np.testing.assert_array_equal(out[0].cpu().numpy(), qo.quantize(f[0].cpu().numpy(), epsilon=eps))


def test_pipeline_status_codes():
    """Codes that need a created pipeline: bad host offsets, counts, stride, null buffers."""
    from neural_spectral_codec_b200 import _lib
    lib = _lib.load()
    enc = make_encoder()
    p, lut = enc._params(), enc.freq_to_bin()
    h = C.c_void_p()
    assert lib.nsc_pipeline_create(1 << 16, 2, 0, C.byref(h)) == 0
    try:
        hp = np.ones((16, 4), np.float32)
        ho = np.zeros((1, 800), np.uint16)
        def call(offs, n_points=16, stride=4, out=ho.ctypes.data):
            o = np.asarray(offs, np.int64)            # kept alive across the call
            return lib.nsc_pipeline_encode_u16(h, hp.ctypes.data, stride, n_points, o.ctypes.data, 1, C.byref(p),
                                               lut.ctypes.data, 1e-8, out)
        assert call([0, 16]) == 0
        np.testing.assert_array_equal(ho[0], quantize(enc.encode_points_batch(
            torch.from_numpy(hp).cuda(), torch.tensor([0, 16])))[0].cpu().numpy())
        assert call([0, 17]) == -8 and call([-1, 16]) == -8 and call([9, 3]) == -8
        assert call([0, 16], n_points=-1) == -3
        assert call([0, 16], stride=5) == -2
        assert call([0, 16], out=None) == -1
        ptrs = (C.c_void_p * 1)(hp.ctypes.data)

        def scall(counts, stride=4):
            c = np.asarray(counts, np.int64)
            return lib.nsc_pipeline_encode_scans_u16(h, ptrs, c.ctypes.data, stride, 1, C.byref(p), lut.ctypes.data,
                                                     1e-8, ho.ctypes.data)
        assert scall([16]) == 0
        assert scall([-1]) == -8 and scall([1 << 17]) == -6 and scall([16], stride=2) == -2
    finally:
        lib.nsc_pipeline_destroy(h)


def test_encode_scans_both_input_forms():
    enc = make_encoder()
    pts, offs = small_batch(50, 23, device="cpu")
    host = pts.numpy()
    offs_np = offs.numpy()
    scans = [host[offs_np[i]:offs_np[i + 1]] for i in range(23)]
    scans[4] = host[:0]                                            # an empty scan
    f_list = enc.encode_scans(scans)
    q_list = enc.encode_scans(scans, dtype=np.uint16)
    assert q_list.dtype == np.uint16
    np.testing.assert_array_equal(q_list, quantize(torch.from_numpy(f_list).cuda()).cpu().numpy())
    f_tup = enc.encode_scans((host, offs_np))
    q_tup = enc.encode_scans((host, offs_np), dtype=np.uint16, max_chunk_points=40_000)   # several chunks
    np.testing.assert_array_equal(q_tup, quantize(torch.from_numpy(f_tup).cuda()).cpu().numpy())
    np.testing.assert_array_equal(q_tup, enc.encode_points_batch(pts.cuda(), offs, dtype=torch.uint16).cpu().numpy())
    out = np.zeros((23, 800), np.uint16)
    assert enc.encode_scans(scans, out=out, dtype=np.uint16) is out
    np.testing.assert_array_equal(out, q_list)
    np.testing.assert_array_equal(q_list[7], qo.quantize(f_list[7]))
    with pytest.raises(ValueError):
        enc.encode_scans(scans, out=np.zeros((23, 800), np.float32), dtype=np.uint16)


def test_other_image_width_takes_two_launches():
    """No fused kernel for 512 columns: general kernel to float32, then the quantiser."""
    enc = make_encoder(n_azimuth=512)
    pts, offs = small_batch(60, 5)
    assert_wire_rows(enc, pts, offs, sample=(0, 4))
    scans = [pts[offs[i]:offs[i + 1]].cpu().numpy() for i in range(5)]
    np.testing.assert_array_equal(enc.encode_scans(scans, dtype=np.uint16),
                                  quantize(torch.from_numpy(enc.encode_scans(scans)).cuda()).cpu().numpy())


def test_tuning_builds_give_the_same_integers(tmp_path):
    """The tuning build with the generic kernel instead of the warp-specialised one (NSC_WS=0), no
    clusters (NSC_SPLIT=0), no split last wave (NSC_TAILSPLIT=0): same integers as the product build."""
    import subprocess
    import sys
    from conftest import ROOT
    from neural_spectral_codec_b200 import _lib
    enc = make_encoder()
    for n in (2, 170):
        pts, offs = small_batch(5, n)
        np.save(tmp_path / f"want{n}.npy", enc.encode_points_batch(pts, offs, dtype=torch.uint16).cpu().numpy())
    code = f"""
import sys, numpy as np, torch
sys.path.insert(0, {ROOT!r})
sys.path.insert(0, {os.path.join(ROOT, "tests")!r})
from test_gpu_encode_uint16 import make_encoder, small_batch
enc = make_encoder()
for n in (2, 170):
    pts, offs = small_batch(5, n)
    got = enc.encode_points_batch(pts, offs, dtype=torch.uint16).cpu().numpy()
    assert np.array_equal(got, np.load(r"{tmp_path}/want%d.npy" % n)), n
print("same")
"""
    for env in ({"NSC_WS": "0"}, {"NSC_SPLIT": "0"}, {"NSC_TAILSPLIT": "0"}):
        r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True,
                           env=dict(os.environ, NSC_LIB=_lib.TUNE_LIB_PATH, **env), timeout=600)
        assert r.returncode == 0 and "same" in r.stdout, (env, r.stderr[-2000:])
