"""The host-buffer pipeline (nsc_pipeline_*, csrc/nsc_pipeline.cu) through ctypes: every row it
returns equals encode_points_batch on the device bit for bit, for the same seeded scans. Covered:
its encode entry points mixed on one pipeline (single scans left running on another stream while
batch calls reuse the slots), every slot count with both host input forms and both row formats,
chunks cut at 1024 scans, and an oversized scan refused before anything is copied."""
import ctypes as C

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

TINY = ("tiny", 16, -24.8, 2.0, 200)     # ~2.9 k points a scan
SPECK = ("speck", 4, -24.8, 2.0, 11)     # ~40 points a scan
CHUNK = 6000                              # two TINY scans a chunk
SENTINEL = -7.25


@pytest.fixture(scope="module")
def lib():
    from neural_spectral_codec_b200 import _lib
    return _lib.load()


@pytest.fixture(scope="module")
def enc():
    from neural_spectral_codec_b200 import SpectralEncoder
    return SpectralEncoder(n_elevation=16, n_azimuth=360, n_bins=50, alpha=2.0, learnable_alpha=True,
                           target_elevation_bins=16).to("cuda")


def make_scans(shape, first, n):
    """n seeded host scans, float32 (N, 4) numpy arrays."""
    from neural_spectral_codec_b200 import synth
    pts, offs = synth.make_batch(synth.SensorShape(*shape), first, n)
    p, o = pts.numpy(), offs.numpy()
    return [p[o[i]:o[i + 1]] for i in range(n)]


def concat(scans):
    offs = np.zeros(len(scans) + 1, np.int64)
    np.cumsum([len(s) for s in scans], out=offs[1:])
    return np.ascontiguousarray(np.concatenate(scans)), offs


def reference(enc, scans, dtype):
    """encode_points_batch of the scans on the device, as host rows."""
    pts, offs = concat(scans)
    tdtype = torch.uint16 if dtype == np.uint16 else torch.float32
    return enc.encode_points_batch(torch.from_numpy(pts).cuda(), torch.from_numpy(offs).cuda(),
                                   dtype=tdtype).cpu().numpy()


def same_bits(a, b):
    return a.dtype == b.dtype and a.shape == b.shape and np.array_equal(a.view(np.uint16), b.view(np.uint16))


class Pipeline:
    def __init__(self, lib, enc, max_chunk_points, n_buffers):
        self.lib, self.enc = lib, enc
        self.p, self.lut = enc._params(), enc.freq_to_bin()
        self.h = C.c_void_p()
        assert lib.nsc_pipeline_create(max_chunk_points, n_buffers, torch.cuda.current_device(), C.byref(self.h)) == 0

    def close(self):
        self.lib.nsc_pipeline_destroy(self.h)

    def batch(self, scans, form, dtype=np.float32):
        """One nsc_pipeline_encode[_scans][_u16] call -> (status, host rows). "buffer" passes the
        scans concatenated with offsets, "list" one pointer per scan (null for an empty one)."""
        from neural_spectral_codec_b200 import _lib
        out = np.full((len(scans), self.enc.output_dim), SENTINEL if dtype == np.float32 else 0xbeef, dtype)
        if form == "buffer":
            pts, offs = concat(scans)
            name = "nsc_pipeline_encode"
            args = (self.h, pts.ctypes.data, 4, pts.shape[0], offs.ctypes.data, len(scans), C.byref(self.p),
                    self.lut.ctypes.data)
        else:
            ptrs = (C.c_void_p * len(scans))(*[s.ctypes.data if len(s) else None for s in scans])
            counts = np.array([len(s) for s in scans], np.int64)
            name = "nsc_pipeline_encode_scans"
            args = (self.h, ptrs, counts.ctypes.data, 4, len(scans), C.byref(self.p), self.lut.ctypes.data)
        if dtype == np.uint16:
            name += "_u16"
            args += (_lib.QUANT_EPSILON,)
        return getattr(self.lib, name)(*args, out.ctypes.data), out

    def single(self, scan, d_out, stream):
        """nsc_pipeline_encode_scan: returns before the row is written on `stream`."""
        return self.lib.nsc_pipeline_encode_scan(self.h, scan.ctypes.data, 4, len(scan), C.byref(self.p),
                                                 self.lut.ctypes.data, d_out.data_ptr(), stream.cuda_stream)


@pytest.fixture(scope="module")
def tiny(enc):
    scans = make_scans(TINY, 300, 24)
    assert max(len(scans[i]) + len(scans[i + 1]) for i in range(23)) <= CHUNK
    assert min(len(scans[i]) + len(scans[i + 1]) + len(scans[i + 2]) for i in range(22)) > CHUNK
    return scans, {dt: reference(enc, scans, dt) for dt in (np.float32, np.uint16)}


def test_entry_points_mixed_on_one_pipeline(lib, enc, tiny):
    """Single scans left running on a side stream hold every slot; a one-chunk batch call (one slot),
    a list call (every slot) and more single scans follow on the same pipeline without a sync."""
    scans, ref = tiny
    ref = ref[np.float32]
    pl = Pipeline(lib, enc, CHUNK, 3)
    side = torch.cuda.Stream()
    rows = torch.full((len(scans), enc.output_dim), SENTINEL, device="cuda")
    side.wait_stream(torch.cuda.current_stream())
    try:
        for i in range(6):                                # two rounds over the three slots
            assert pl.single(scans[i], rows[i], side) == 0
        st, one = pl.batch(scans[6:8], "buffer")          # one chunk
        assert st == 0 and same_bits(one, ref[6:8])
        st, many = pl.batch(scans[8:20], "list")          # six chunks
        assert st == 0 and same_bits(many, ref[8:20])
        for i in range(20, 24):
            assert pl.single(scans[i], rows[i], side) == 0
    finally:
        side.synchronize()
        pl.close()
    got = rows.cpu().numpy()
    assert same_bits(got[:6], ref[:6]) and same_bits(got[20:], ref[20:])


@pytest.mark.parametrize("dtype", [np.float32, np.uint16], ids=["float32", "uint16"])
@pytest.mark.parametrize("form", ["buffer", "list"])
@pytest.mark.parametrize("n_buffers", [1, 2, 3, 4])
def test_every_slot_count(lib, enc, tiny, n_buffers, form, dtype):
    """24 scans in 12 chunks of two: every slot is reused (three rounds over four slots)."""
    scans, ref = tiny
    pl = Pipeline(lib, enc, CHUNK, n_buffers)
    try:
        st, out = pl.batch(scans, form, dtype)
    finally:
        pl.close()
    assert st == 0 and same_bits(out, ref[dtype])


def test_chunks_of_1024_scans(lib, enc):
    """2500 scans of ~40 points, every seventh empty: chunks of 1024, 1024 and 452 scans."""
    scans = make_scans(SPECK, 0, 2500)
    for i in range(0, 2500, 7):
        scans[i] = scans[i][:0]
    ref = reference(enc, scans, np.float32)
    pl = Pipeline(lib, enc, 1 << 20, 2)
    try:
        for form in ("buffer", "list"):
            st, out = pl.batch(scans, form)
            assert st == 0 and same_bits(out, ref), form
    finally:
        pl.close()


def test_oversized_scan_is_refused_before_any_copy(lib, enc, tiny):
    """A scan larger than max_chunk_points after one that fits: NSC_ERR_WORKSPACE, h_out untouched."""
    scans, _ = tiny
    big = np.concatenate(scans[1:3])
    assert len(scans[0]) <= 4000 < len(big)
    pl = Pipeline(lib, enc, 4000, 2)
    try:
        for form in ("buffer", "list"):
            st, out = pl.batch([scans[0], big], form)
            assert st == -6 and (out == SENTINEL).all(), form
    finally:
        pl.close()
