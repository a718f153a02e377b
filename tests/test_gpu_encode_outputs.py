"""The encode outputs that no other single-GPU test pins, through every point kernel: descriptor
rows stored into peer databases (nsc_encode_batch_peers, here with two local buffers) and range
images at both stages (nsc_project_batch). Four batch shapes reach the four kernel paths: a
2-scan batch (cluster kernel), 2 x SMs stride-4 scans (warp-specialised kernel), 2 x SMs + 5
scans (warp-specialised, the last wave's scans split over the grid) and 2 x SMs + 5 stride-3
scans (generic kernel). The two scans under test are the last two of each batch, so in the split
shape they are among the split ones."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu

SMALL = ("s", 64, -24.8, 2.0, 700)    # 64 rings x 700 azimuth steps: small scans, quick batches
SHAPES = ["cluster", "ws", "ws_split", "stride3"]
SENTINEL = -7.25


def make_encoder():
    from neural_spectral_codec_b200 import SpectralEncoder
    return SpectralEncoder(n_elevation=16, n_azimuth=360, n_bins=50, alpha=2.0, learnable_alpha=True,
                           target_elevation_bins=16).to("cuda")


def batch(shape):
    """Concatenated device points and host offsets of `shape`; its last two scans are seeds 7, 8."""
    from neural_spectral_codec_b200 import synth
    sensor = synth.SensorShape(*SMALL)
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    n = {"cluster": 2, "ws": 2 * sms, "ws_split": 2 * sms + 5, "stride3": 2 * sms + 5}[shape]
    head_p, head_o = synth.make_batch(sensor, 100, n - 2, device="cuda")
    tail_p, tail_o = synth.make_batch(sensor, 7, 2, device="cuda")
    pts = torch.cat([head_p, tail_p])
    offs = torch.cat([head_o.cpu(), tail_o.cpu()[1:] + head_o[-1].item()])
    if shape == "stride3":
        pts = pts[:, :3]
    return pts.contiguous(), offs


def stream_and_workspace(p, n):
    from neural_spectral_codec_b200.encoder import _workspace
    stream = torch.cuda.current_stream().cuda_stream
    return stream, _workspace(torch.device("cuda", torch.cuda.current_device()), stream, p, n)


@pytest.mark.parametrize("shape", SHAPES)
def test_peer_rows_equal_the_batch_rows(shape):
    """Two peer databases on this GPU, first row 7: rows [7, 7 + n) of both are the rows of
    nsc_encode_batch bit for bit, every other row keeps the sentinel."""
    from neural_spectral_codec_b200 import _lib
    enc = make_encoder()
    pts, offs = batch(shape)
    n = offs.numel() - 1
    rows = enc.encode_points_batch(pts, offs.cuda())
    dbs = [torch.full((n + 10, enc.output_dim), SENTINEL, device="cuda") for _ in range(2)]
    h_db = (C.c_void_p * 2)(*[d.data_ptr() for d in dbs])
    p = enc._params()
    stream, ws = stream_and_workspace(p, n)
    d_offs = offs.cuda()
    st = _lib.load().nsc_encode_batch_peers(pts.data_ptr(), pts.shape[1], d_offs.data_ptr(), 0, n, C.byref(p),
                                            enc.freq_to_bin().ctypes.data, h_db, 2, 7, ws.data_ptr(),
                                            ws.numel() * 4, stream)
    _lib.check(st, "nsc_encode_batch_peers")
    torch.cuda.synchronize()
    for d in dbs:
        assert torch.equal(d[7:7 + n].view(torch.int32), rows.view(torch.int32))
        assert (d[:7] == SENTINEL).all() and (d[7 + n:] == SENTINEL).all()


@pytest.mark.parametrize("interpolate", [False, True], ids=["projected", "interpolated"])
@pytest.mark.parametrize("shape", SHAPES[1:])
def test_images_are_the_same_through_every_kernel(shape, interpolate):
    """The images of the last two scans of each batch equal those of the 2-scan batch (cluster
    kernel) bit for bit, at both stages."""
    from neural_spectral_codec_b200.encoder import RangeImageProjector
    proj = RangeImageProjector(n_elevation=16, device="cuda")
    ref_p, ref_o = batch("cluster")
    ref = proj.project_batch(ref_p, ref_o.cuda(), interpolate=interpolate)
    pts, offs = batch(shape)
    got = proj.project_batch(pts, offs.cuda(), interpolate=interpolate)[-2:]
    assert (ref > 0).any()
    assert torch.equal(got.view(torch.int32), ref.view(torch.int32))
