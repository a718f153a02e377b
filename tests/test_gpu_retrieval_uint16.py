"""uint16 retrieval database (WassersteinRetriever(database_dtype=torch.uint16),
nsc_wasserstein_cdf_u16 / nsc_wasserstein_query_u16) against the integer CDF computed in NumPy, the
oracle's distances over the dequantised rows and the float32 database.

Tolerances are those of tests/test_gpu_retrieval.py. Rows that sum to 65535 (wire rows) and all-zero
rows are stored exactly; any other uint16 row is rounded to 1/65535 per CDF element, so its distances
may differ from the dequantised float path by up to n_bins / 131070 more.
"""
import numpy as np
import pytest
import torch

from oracle import quantization_oracle as qo
from oracle import retrieval_oracle as ro
from test_gpu_retrieval import ATOL, RTOL, check_topk

pytestmark = pytest.mark.gpu


def retriever(dtype=torch.uint16):
    from neural_spectral_codec_b200.retrieval import WassersteinRetriever
    return WassersteinRetriever(device="cuda", database_dtype=dtype)


def same(a, b):
    """Bit equality of two tensors (uint16 ones compared as their int16 bits)."""
    if a.dtype == torch.uint16:
        a, b = a.view(torch.int16), b.view(torch.int16)
    return a.dtype == b.dtype and torch.equal(a, b)


def wire_rows(rng, n, n_bins):
    h = rng.gamma(0.5, 1.0, (n, n_bins)).astype(np.float32)
    h[np.arange(n), rng.integers(0, n_bins, n)] += 5.0 * rng.random(n).astype(np.float32)     # spikes
    return np.stack([qo.quantize(r) for r in h])


def dequantize(rows):
    return np.stack([qo.dequantize(r) for r in rows])


def integer_cdf(rows):
    """The stored CDF rows, computed with NumPy integers."""
    s = np.cumsum(rows.astype(np.int64), axis=1)
    t = s[:, -1:]
    num = 65535 * s
    q = num // np.maximum(t, 1)
    rem = num - q * np.maximum(t, 1)
    q += (2 * rem > t) | ((2 * rem == t) & (q % 2 == 1))
    out = np.where(t == 65535, s, np.where(t == 0, 0, q))
    return out.astype(np.uint16)


def odd_rows(rng, n_bins):
    """uint16 rows that do not sum to 65535: small, huge and odd totals."""
    rows = [np.zeros(n_bins, np.uint16) for _ in range(4)]
    rows[0][rng.integers(0, n_bins)] = 1
    rows[1][[0, n_bins - 1]] = 3
    rows[2][:] = 65535
    rows[3][:] = rng.integers(0, 9, n_bins)
    rows += list(rng.integers(0, 65536, (3, n_bins)).astype(np.uint16))
    rows += list(rng.integers(0, 200, (3, n_bins)).astype(np.uint16))
    r = np.stack(rows)
    assert ((r.astype(np.int64).sum(1) % 2) == 1).any() and (r.astype(np.int64).sum(1) > 65535).any()
    return r


@pytest.mark.parametrize("n_bins", [7, 50, 100, 800, 801, 1024])
def test_cdf_rows_equal_the_integer_computation(n_bins):
    rng = np.random.default_rng(n_bins)
    rows = np.concatenate([wire_rows(rng, 300, n_bins), np.zeros((5, n_bins), np.uint16), odd_rows(rng, n_bins)])
    rows = rows[rng.permutation(len(rows))]
    r = retriever()
    r.add_to_database(rows)
    assert r.database_hists.dtype == torch.uint16 and r.database_cdfs.dtype == torch.uint16
    np.testing.assert_array_equal(r.database_hists.cpu().numpy(), rows)
    np.testing.assert_array_equal(r.database_cdfs.cpu().numpy(), integer_cdf(rows))


@pytest.mark.parametrize("n_bins", [7, 50, 100, 800, 801, 1024])
def test_distances_against_the_oracle_on_dequantised_rows(n_bins):
    """Wire rows and zero rows; Q = 1, 8 and 11 (two query groups); every lane-padding case."""
    rng = np.random.default_rng(100 + n_bins)
    rows = wire_rows(rng, 2000, n_bins)
    rows[rng.choice(len(rows), 20, replace=False)] = 0
    deq = dequantize(rows)
    qs = deq[rng.integers(0, len(rows), 11)] + (rng.random((11, n_bins)) / n_bins).astype(np.float32)
    qs[3] = rng.gamma(0.5, 1.0, n_bins)
    r = retriever()
    r.add_to_database(rows)
    refs = [ro.wasserstein_distance_batch(torch.from_numpy(q), torch.from_numpy(deq)).numpy() for q in qs]
    for nq in (1, 8, 11):
        idx, top, cnt, dist = r.query_batch(qs[:nq], top_k=10, return_distances=True)
        assert cnt.cpu().tolist() == [10] * nq
        for i in range(nq):
            np.testing.assert_allclose(dist[i].cpu().numpy(), refs[i], rtol=RTOL, atol=ATOL)
            check_topk(idx[i].cpu().numpy(), top[i].cpu().numpy(), refs[i], 10)


@pytest.mark.parametrize("n_bins", [7, 800, 801])
def test_rows_that_do_not_sum_to_65535(n_bins):
    rng = np.random.default_rng(200 + n_bins)
    rows = np.concatenate([odd_rows(rng, n_bins), wire_rows(rng, 50, n_bins)])
    deq = dequantize(rows)
    qs = rng.gamma(0.5, 1.0, (3, n_bins)).astype(np.float32)
    r = retriever()
    r.add_to_database(rows)
    dist = r.query_batch(qs, top_k=0, return_distances=True)[3].cpu().numpy()
    for i in range(3):
        ref = ro.wasserstein_distance_batch(torch.from_numpy(qs[i]), torch.from_numpy(deq)).numpy()
        np.testing.assert_allclose(dist[i], ref, rtol=RTOL, atol=ATOL + n_bins / 131070)


def test_top_k_on_every_selection_path():
    """k <= 128 (many-CTA select), 128 < k <= 1024 (one CTA per query), k > 1024 (device sort)."""
    rng = np.random.default_rng(5)
    rows = wire_rows(rng, 3000, 800)
    deq = dequantize(rows)
    qs = deq[[3, 1700]] * np.float32(3.0)
    r = retriever()
    r.add_to_database(rows)
    refs = [ro.wasserstein_distance_batch(torch.from_numpy(q), torch.from_numpy(deq)).numpy() for q in qs]
    for k in (1, 10, 128, 300, 1024, 1500, 3000):
        idx, top, cnt = r.query_batch(qs, top_k=k)
        assert cnt.cpu().tolist() == [k, k]
        for i in range(2):
            check_topk(idx[i].cpu().numpy(), top[i].cpu().numpy(), refs[i], k)
    assert r.query_batch(qs, top_k=10)[0][:, 0].cpu().tolist() == [3, 1700]


def test_duplicates_tie_by_lower_index_and_the_spatial_filter():
    rng = np.random.default_rng(1)
    base = wire_rows(rng, 40, 800)
    rows = np.concatenate([base, base, base[:10]])
    xyz = np.stack([np.arange(len(rows)) * 10.0, np.zeros(len(rows)), np.zeros(len(rows))], 1)
    q = dequantize(base[5:6])
    r = retriever()
    r.add_to_database(rows, positions=xyz)
    idx, top, cnt = r.query_batch(q, top_k=3)
    assert idx[0].cpu().tolist() == [5, 45, 85] and float(top[0, 0]) == float(top[0, 1]) == float(top[0, 2])
    # the spatial filter excludes the same rows as on the float32 database of the dequantised rows
    f = retriever(torch.float32)
    f.add_to_database(dequantize(rows), positions=xyz)
    for k, radius in ((3, 50.0), (8, 420.0), (len(rows), 100.0)):
        got = r.query_batch(q, top_k=k, query_positions=xyz[45:46], spatial_filter_distance=radius)
        want = f.query_batch(q, top_k=k, query_positions=xyz[45:46], spatial_filter_distance=radius)
        n_valid = int((np.abs(np.arange(len(rows)) - 45) * 10.0 >= radius).sum())
        c = min(k, n_valid)
        assert got[2].item() == want[2].item() == c
        assert (got[0][0, c:] == -1).all() and torch.isinf(got[1][0, c:]).all()
        assert all(abs(i - 45) * 10.0 >= radius for i in got[0][0, :c].cpu().tolist())
        if k == len(rows):
            assert set(got[0][0, :c].cpu().tolist()) == set(want[0][0, :c].cpu().tolist())
        np.testing.assert_allclose(got[1][0, :c].cpu().numpy(), want[1][0, :c].cpu().numpy(), rtol=RTOL, atol=ATOL)


def test_many_identical_rows_take_the_radix_fallback():
    rng = np.random.default_rng(2)
    row = wire_rows(rng, 1, 800)[0]
    far = wire_rows(rng, 40, 800)
    rows = np.concatenate([np.tile(row, (3000, 1)), far, np.tile(row, (50, 1))])
    q = dequantize(row[None])[0] * np.float32(1.5)
    r = retriever()
    r.add_to_database(rows)
    for k in (20, 200):                 # select_kernel and topk_kernel, both past their candidate lists
        idx, top, cnt = r.query_batch(q, top_k=k)
        assert idx[0].cpu().tolist() == list(range(k))
        assert float(top[0].max()) == float(top[0].min())


def test_mixed_inserts_equal_converting_first():
    from neural_spectral_codec_b200.quantization import HistogramQuantizer
    rng = np.random.default_rng(3)
    h = rng.gamma(0.5, 1.0, (2600, 800)).astype(np.float32)
    hq = HistogramQuantizer(n_bins=800)
    q16 = hq.quantize(torch.from_numpy(h).cuda())
    deq = hq.dequantize(q16)
    queries = h[[7, 2000, 2500]]
    xyz = rng.random((len(h), 3)) * 100

    # float rows into a uint16 database, in chunks across the capacity steps (1024, 2048)
    a, b = retriever(), retriever()
    for lo, hi in ((0, 700), (700, 1100), (1100, 1101), (1101, 2600)):
        a.add_to_database(h[lo:hi], positions=xyz[lo:hi])
    b.add_to_database(q16, positions=xyz)
    assert a.database_size == b.database_size == len(h)
    assert same(a.database_hists, b.database_hists) and same(a.database_cdfs, b.database_cdfs)
    assert torch.equal(a._xyz[:len(h)], b._xyz[:len(h)])
    ra = a.query_batch(queries, top_k=10, return_distances=True)
    rb = b.query_batch(queries, top_k=10, return_distances=True)
    assert all(same(x, y) for x, y in zip(ra, rb))

    # uint16 rows into a float32 database
    c, d = retriever(torch.float32), retriever(torch.float32)
    c.add_to_database(q16[:1500])
    c.add_to_database(q16[1500:].cpu().numpy())
    d.add_to_database(deq)
    assert same(c.database_hists, d.database_hists) and same(c.database_cdfs, d.database_cdfs)
    rc, rd = c.query_batch(queries, top_k=10), d.query_batch(queries, top_k=10)
    assert all(same(x, y) for x, y in zip(rc, rd))

    # uint16 queries are their dequantised rows, on either database
    qq = torch.from_numpy(q16.cpu().numpy()[[7, 2000, 2500]]).cuda()
    for db in (b, d):
        got = db.query_batch(qq, top_k=10, return_distances=True)
        want = db.query_batch(hq.dequantize(qq), top_k=10, return_distances=True)
        assert all(same(x, y) for x, y in zip(got, want))
    qi, qd = b.query(qq[0].cpu().numpy(), top_k=5)
    assert qi[0] == 7 and qi.dtype == np.int64 and qd.dtype == np.float32


def test_uint16_encoder_output_feeds_the_retriever():
    """encode_points_batch(..., dtype=torch.uint16) into a uint16 database: the scans retrieve
    themselves; encode_scans(..., dtype=np.uint16) rows go into either database."""
    from neural_spectral_codec_b200 import SpectralEncoder, synth
    small = synth.SensorShape("s", 64, -24.8, 2.0, 600)
    pts, offs = synth.make_batch(small, 0, 64, device="cuda")
    enc = SpectralEncoder(n_elevation=16, target_elevation_bins=16).to("cuda")
    desc = enc.encode_points_batch(pts, offs, dtype=torch.uint16)
    r = retriever()
    r.add_to_database(desc)
    assert same(r.database_hists, desc)
    idx, top, cnt = r.query_batch(desc[:8], top_k=1)
    assert idx[:, 0].cpu().tolist() == list(range(8))
    scans = [synth.make_scan(small, i).numpy() for i in range(12)]
    rows = enc.encode_scans(scans, dtype=np.uint16)
    for dt in (torch.uint16, torch.float32):
        db = retriever(dt)
        db.add_to_database(rows)
        assert db.query_batch(rows[:8], top_k=1)[0][:, 0].cpu().tolist() == list(range(8))
