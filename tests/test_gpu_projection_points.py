"""The projection checked one point at a time on the device.

Dense clouds hide misplaced points: a pixel shows only its closest point, so in a full HDL-64
scan 95 % of the points could land in the wrong pixel without changing the range image. Here the
points of the sets in point_sets.py are dealt into sparse scans in which no two kept points can
meet in one pixel -- not even an excused point that takes the pixel across its edge -- and dropped
points (out of range, ulps around the range limits, NaN / Inf, overflowing squares) are mixed in
at random positions, so both lanes of the packed pair path get every kind of point. Then, per
batch of nsc_project_batch (interpolate=False):

  * every kept point that is not within 1e-5 rad of an edge: the pixel the oracle assigns holds
    exactly its float32 range (bits); points on the axes (signed zeros) are held to this too,
    although they sit on column edges;
  * every excused point: its range is at its oracle pixel or at the pixel across the nearest
    edge(s) (columns wrap, rows clamp);
  * every scan: as many non-empty pixels as kept points, so nothing else was written.

Together these mean the whole image equals the oracle's, up to the excuse. The batch shapes are
those of test_gpu_encode_outputs.py, so every point kernel runs: cluster (2 scans),
warp-specialised (2 x SMs scans, stride 4), the same with the last wave split (2 x SMs + 5) and
the generic kernel (2 x SMs + 5 scans, stride 3).
"""
import functools
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import point_sets as ps
from conftest import ROOT
from oracle import nsc_oracle as orc

pytestmark = pytest.mark.gpu

SHAPES = ["cluster", "ws", "ws_split", "stride3"]
# name -> (elevation range in degrees, rows, min_range, max_range, row rule: 0 polynomial, 1 search)
CONFIGS = {
    "default": ((-24.8, 2.0), 16, 1.0, 80.0, 0),
    "fov15_e16": ((-15.0, 15.0), 16, 1.0, 80.0, 0),
    "fov60_e32": ((-60.0, 60.0), 32, 1.0, 80.0, 1),
    "fov89_e64": ((-89.0, 89.0), 64, 1.0, 80.0, 1),
    "e1": ((-24.8, 2.0), 1, 1.0, 80.0, 0),
    "e2": ((-24.8, 2.0), 2, 1.0, 80.0, 0),
    "e8": ((-24.8, 2.0), 8, 1.0, 80.0, 0),
    "e40": ((-24.8, 2.0), 40, 1.0, 80.0, 0),
    "e64": ((-24.8, 2.0), 64, 1.0, 80.0, 0),
    "r05_120": ((-24.8, 2.0), 16, 0.5, 120.0, 0),
    "r2_50": ((-30.0, 10.0), 16, 2.0, 50.0, 0),
    "r0_30": ((-24.8, 2.0), 16, 0.0, 30.0, 0),
}
INTENSITIES = np.array([-1.5, -0.0, 0.0, 1e-45, 1e-40, -1e-40, np.nan, -np.nan, np.inf, -np.inf, 0.25, 3e38],
                       np.float32)
EXCUSE = 1e-5
DEV = "cuda"


def oracle_config(name, n_azimuth=360):
    er, rows, lo, hi, _ = CONFIGS[name]
    return orc.OracleConfig(n_elevation=rows, n_azimuth=n_azimuth, elevation_range=er, min_range=lo, max_range=hi)


def projector(name, n_azimuth=360):
    from neural_spectral_codec_b200.encoder import RangeImageProjector
    er, rows, lo, hi, _ = CONFIGS[name]
    return RangeImageProjector(n_elevation=rows, n_azimuth=n_azimuth, elevation_range=er, min_range=lo,
                               max_range=hi, device="cuda")


def deal(cand, clear, excused, n_pix, rng):
    """Kept points -> scans, no two of which claim a common pixel within one scan. A point claims
    its candidate pixels (one if clear, up to four if excused). Clear points are dealt by their
    rank among the points of their pixel; excused points go to scans of their own, a greedy
    independent set per scan (the first point in the list always joins, so every pass makes progress)."""
    scans = []
    idx = rng.permutation(np.flatnonzero(clear))
    order = idx[np.argsort(cand[idx, 0], kind="stable")]
    pix = cand[order, 0]
    start = np.flatnonzero(np.r_[True, pix[1:] != pix[:-1]])
    rank = np.arange(len(order)) - np.repeat(start, np.diff(np.r_[start, len(order)]))
    by_rank = np.argsort(rank, kind="stable")
    bounds = np.searchsorted(rank[by_rank], np.arange(rank.max() + 2 if len(rank) else 1))
    scans += [order[by_rank[bounds[r]:bounds[r + 1]]] for r in range(len(bounds) - 1)]
    remaining = rng.permutation(np.flatnonzero(excused))
    while remaining.size:                         # a point joins if it is the first to claim each of its pixels
        c = cand[remaining]
        first = np.full(n_pix, len(remaining))
        np.minimum.at(first, c.reshape(-1), np.repeat(np.arange(len(remaining)), 4))
        ok = (first[c] == np.arange(len(remaining))[:, None]).all(1)
        scans.append(remaining[ok])
        remaining = remaining[~ok]
    return scans


class Pool:
    """The points of one configuration, what the oracle says about each, and their scans."""

    def __init__(self, name, n_azimuth=360, seed=0, scale=1.0):
        cfg = self.cfg = oracle_config(name, n_azimuth)
        rng = np.random.default_rng(seed)
        n = lambda k: int(k * scale)
        strict_set = ps.signed_zeros(cfg)
        sets = [strict_set, ps.uniform_sphere(rng, n(200_000)), ps.edge_points(rng, cfg, n(150_000)),
                ps.octant_lines(rng, n(6_000), cfg), ps.near_axis(rng, n(20_000), cfg),
                ps.adversarial(rng, 60, cfg), ps.range_limits(rng, cfg)]
        pts = np.concatenate(sets)
        strict = np.zeros(len(pts), bool)
        strict[:len(strict_set)] = True
        # min_range 0 keeps points whose float32 range is 0 (all squares underflow); a pixel holding
        # 0 reads as empty, so no image can show where they went: leave them out
        kept, _, _, r, _, _ = ps.oracle_pixels(pts, cfg)
        visible = ~(kept & (r == 0))
        pts = self.pts = np.ascontiguousarray(pts[visible])
        strict = strict[visible]
        self.intensity = rng.choice(INTENSITIES, len(pts))
        self.pts4 = np.ascontiguousarray(np.concatenate([pts, self.intensity[:, None]], 1))
        kept, row, col, self.range, d_az, d_el = ps.oracle_pixels(pts, cfg)
        ex_az, ex_el = kept & ~strict & (d_az <= EXCUSE), kept & ~strict & (d_el <= EXCUSE)
        row_x, col_x = ps.across_edges(pts, cfg, row, col)
        W = cfg.n_azimuth
        self.cand = np.stack([row * W + col, row * W + np.where(ex_az, col_x, col),
                              np.where(ex_el, row_x, row) * W + col,
                              np.where(ex_el, row_x, row) * W + np.where(ex_az, col_x, col)], 1)
        self.kept, self.excused = kept, ex_az | ex_el
        self.clear = kept & ~self.excused
        kept_scans = deal(self.cand, self.clear, self.excused, cfg.n_elevation * W, rng)
        # dropped points: every scan gets at least two, the rest at random; then a random order
        dropped = np.flatnonzero(~kept)
        extra = np.array_split(rng.permutation(dropped), len(kept_scans))
        self.scans = [rng.permutation(np.concatenate([k, e, rng.choice(dropped, 2)]))
                      for k, e in zip(kept_scans, extra)]
        self.filler = [rng.choice(dropped, 3) for _ in range(1000)]     # dropped-only scans
        assert self.excused.sum() > 1000 and self.clear.sum() > 100_000 * scale

    def batches(self, n_per_batch):
        """Scans padded with dropped-only scans to whole batches of n_per_batch."""
        scans = list(self.scans)
        pad = -len(scans) % n_per_batch
        scans += self.filler[:pad]
        return [scans[i:i + n_per_batch] for i in range(0, len(scans), n_per_batch)]


@functools.lru_cache(maxsize=None)
def pool(name, n_azimuth=360):
    return Pool(name, n_azimuth, seed=sorted(CONFIGS).index(name) * 1000 + n_azimuth)


def device_batch(pool, scans, stride):
    host = pool.pts4[np.concatenate(scans), :stride]
    offs = np.zeros(len(scans) + 1, np.int64)
    np.cumsum([len(s) for s in scans], out=offs[1:])
    return torch.from_numpy(np.ascontiguousarray(host)).to(DEV), torch.from_numpy(offs)


def check_images(pool, scans, images, intensity=None):
    """images: (len(scans), E, W) on the device; intensity: the same for the intensity images."""
    E, W = pool.cfg.n_elevation, pool.cfg.n_azimuth
    scan_of = np.concatenate([np.full(len(s), i) for i, s in enumerate(scans)])
    idx = np.concatenate(scans)
    k = pool.kept[idx]
    idx, scan_of = idx[k], scan_of[k]
    flat = images.reshape(-1).view(torch.int32)
    lin = torch.from_numpy(scan_of[:, None] * (E * W) + pool.cand[idx]).to(DEV)
    got = flat[lin].cpu().numpy()                                   # (n, 4) bits at the candidates
    want = pool.range[idx].view(np.int32)
    clear = pool.clear[idx]
    bad = clear & (got[:, 0] != want)
    assert not bad.any(), f"{bad.sum()} of {clear.sum()} clear points not at their oracle pixel, e.g. " \
        f"{pool.pts[idx[bad][:4]].tolist()} range bits {want[bad][:4]} found {got[bad][:4, 0]}"
    hit = got == want[:, None]
    assert hit.any(1).all(), f"{(~hit.any(1)).sum()} excused points at none of their candidate pixels, e.g. " \
        f"{pool.pts[idx[~hit.any(1)][:4]].tolist()}"
    count = (images != 0).sum((1, 2)).cpu().numpy()
    want_count = np.bincount(scan_of, minlength=len(scans))
    assert np.array_equal(count, want_count), f"{(count != want_count).sum()} scans with stray pixels"
    if intensity is not None:
        first = hit.argmax(1)                                        # where the range was found
        gi = intensity.reshape(-1)[lin[torch.arange(len(idx), device=DEV), torch.from_numpy(first).to(DEV)]]
        gi = gi.cpu().numpy()
        i = pool.intensity[idx]
        wi = np.where(i > 0, i, np.float32(0))
        nan = np.isnan(i)
        assert np.isnan(gi[nan]).all()
        assert np.array_equal(gi[~nan].view(np.int32), wi[~nan].view(np.int32))
    return int(clear.sum()), int((~clear).sum())


def n_per_batch(shape):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    return {"cluster": 2, "ws": 2 * sms, "ws_split": 2 * sms + 5, "stride3": 2 * sms + 5}[shape]


def run_case(name, shape):
    import ctypes as C
    from neural_spectral_codec_b200 import _lib
    p = pool(name)
    proj = projector(name)
    assert _lib.load().nsc_test_row_mode(C.byref(proj._params())) == CONFIGS[name][4]
    stride = 3 if shape == "stride3" else 4
    batches = p.batches(n_per_batch(shape))
    images = []
    for scans in batches:
        pts, offs = device_batch(p, scans, stride)
        images.append(proj.project_batch(pts, offs, interpolate=False))
    return check_images(p, [s for b in batches for s in b], torch.cat(images))


@pytest.mark.parametrize("shape", SHAPES)
@pytest.mark.parametrize("name", list(CONFIGS))
def test_every_point_lands_in_its_oracle_pixel(name, shape):
    n_clear, n_excused = run_case(name, shape)
    assert n_clear > 100_000 and n_excused > 1000


def test_every_point_through_the_generic_kernel():
    """The tuning build (the only one that reads NSC_WS) with the warp-specialised kernel off:
    the large batches run the generic persistent kernel."""
    from neural_spectral_codec_b200 import _lib
    code = f"""
import sys
sys.path[:0] = [{ROOT!r}, {os.path.join(ROOT, "tests")!r}]
import test_gpu_projection_points as t
for shape in ("ws", "ws_split"):
    t.run_case("default", shape)
print("same")
"""
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True,
                       env=dict(os.environ, NSC_LIB=_lib.TUNE_LIB_PATH, NSC_WS="0"), timeout=600)
    assert r.returncode == 0 and "same" in r.stdout, r.stderr[-3000:]


@pytest.mark.parametrize("name", ["default", "fov60_e32", "e64"])
def test_intensity_images_point_by_point(name):
    """project_intensity_batch: the range image as above, and at each kept point's pixel the
    intensity max(0, i) -- negative values and -0 give +0, subnormals and +Inf stay, NaN passes."""
    p = pool(name)
    proj = projector(name)
    batches = p.batches(n_per_batch("ws"))
    rng_imgs, int_imgs = [], []
    for scans in batches:
        pts, offs = device_batch(p, scans, 4)
        r, i = proj.project_intensity_batch(pts, offs)
        rng_imgs.append(r)
        int_imgs.append(i)
    check_images(p, [s for b in batches for s in b], torch.cat(rng_imgs), torch.cat(int_imgs))


@pytest.mark.parametrize("width", [77, 180, 500, 1024])
def test_other_widths_point_by_point(width):
    """Widths other than 360 run the general kernel (atan2f, the reference's operation order)."""
    p = pool("default", width)
    proj = projector("default", width)
    batches = p.batches(n_per_batch("ws"))
    images = []
    for scans in batches:
        pts, offs = device_batch(p, scans, 4)
        images.append(proj.project_batch(pts, offs, interpolate=False))
    n_clear, n_excused = check_images(p, [s for b in batches for s in b], torch.cat(images))
    assert n_clear > 100_000 and n_excused > 1000
