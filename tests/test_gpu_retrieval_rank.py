"""nsc_wasserstein_rank / nsc_wasserstein_rank_u16 (top_k of any size) against NumPy's stable argsort
of the distances they return, and against nsc_wasserstein_query where both apply (top_k <= 1024).

The order is that of the key (distance bits as uint32, row): ties go to the lower row, +inf and NaN
last; the count is min(top_k, finite distances), and entries at or past it are -1 / +inf. Every
comparison is bit for bit."""
import numpy as np
import pytest
import torch

from neural_spectral_codec_b200 import _lib

pytestmark = pytest.mark.gpu
N_BINS = 800
INF_BITS = 0x7F800000


def database(dtype, n_db, seed):
    """A retriever over n_db rows drawn from n_db // 20 + 1 distinct ones (heavy ties). The float32
    database also gets CDF rows holding NaN and +inf, whose distances are NaN and +inf."""
    from neural_spectral_codec_b200.retrieval import WassersteinRetriever
    rng = np.random.default_rng(seed)
    base = rng.gamma(0.5, 1.0, (n_db // 20 + 1, N_BINS)).astype(np.float32)
    rows = base[rng.integers(0, len(base), n_db)]
    r = WassersteinRetriever(device="cuda", database_dtype=dtype)
    r.add_to_database(rows)         # float rows into a uint16 database are quantised on the device
    if dtype == torch.float32 and n_db >= 4:
        bad = rng.choice(n_db, max(2, n_db // 100), replace=False)
        r._cdfs[torch.from_numpy(bad[0::2]).cuda(), 7] = float("nan")
        r._cdfs[torch.from_numpy(bad[1::2]).cuda(), 3] = float("inf")
    return r, rows


def queries(rows, n, seed):
    """Copies of database rows (distance ~0 to their duplicates), scaled ones, and a query with a
    NaN bin (every distance NaN: count 0)."""
    rng = np.random.default_rng(seed)
    q = rows[rng.integers(0, len(rows), n)] * (1 + 0.05 * rng.random((n, N_BINS))).astype(np.float32)
    q[0] = rows[len(rows) // 2]
    if n > 2:
        q[2, 11] = np.nan
    return torch.from_numpy(q).cuda()


def outputs(nq, n_db, k):
    return (torch.empty((nq, n_db), dtype=torch.float32, device="cuda"),
            torch.empty((nq, k), dtype=torch.int64, device="cuda"),
            torch.empty((nq, k), dtype=torch.float32, device="cuda"),
            torch.empty((nq,), dtype=torch.int32, device="cuda"))


def rank(r, q, k, xyz=None, qxyz=None, radius=0.0, ws=None, stream=None):
    lib = _lib.load()
    nq, n = q.shape[0], r.database_size
    dist, idx, top, cnt = outputs(nq, n, k)
    if ws is None:
        ws = torch.empty(int(lib.nsc_wasserstein_rank_workspace_bytes(nq, n)), dtype=torch.uint8, device="cuda")
    name = "nsc_wasserstein_rank_u16" if r.database_dtype == torch.uint16 else "nsc_wasserstein_rank"
    s = stream if stream is not None else torch.cuda.current_stream()
    s.wait_stream(torch.cuda.current_stream())          # the inputs and the filled workspace are ready
    with torch.cuda.stream(s):
        st = getattr(lib, name)(q.data_ptr(), nq, r._cdfs.data_ptr(), n, N_BINS, r.epsilon,
                                None if xyz is None else xyz.data_ptr(), None if qxyz is None else qxyz.data_ptr(),
                                radius, dist.data_ptr(), k, idx.data_ptr(), top.data_ptr(), cnt.data_ptr(),
                                ws.data_ptr(), ws.numel(), s.cuda_stream)
    _lib.check(st, name)
    s.synchronize()
    return dist, idx, top, cnt


def query(r, q, k, xyz=None, qxyz=None, radius=0.0):
    """nsc_wasserstein_query[_u16] on the same inputs (k <= 1024), with its zeroed selection workspace."""
    lib = _lib.load()
    nq, n = q.shape[0], r.database_size
    dist, idx, top, cnt = outputs(nq, n, k)
    ws = torch.zeros(int(lib.nsc_wasserstein_workspace_bytes(nq)), dtype=torch.uint8, device="cuda")
    name = "nsc_wasserstein_query_u16" if r.database_dtype == torch.uint16 else "nsc_wasserstein_query"
    st = getattr(lib, name)(q.data_ptr(), nq, r._cdfs.data_ptr(), n, N_BINS, r.epsilon,
                            None if xyz is None else xyz.data_ptr(), None if qxyz is None else qxyz.data_ptr(),
                            radius, dist.data_ptr(), k, idx.data_ptr(), top.data_ptr(), cnt.data_ptr(),
                            ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream)
    _lib.check(st, name)
    torch.cuda.synchronize()
    return dist, idx, top, cnt


def bits(t):
    return t.cpu().numpy().view(np.uint32) if t.dtype == torch.float32 else t.cpu().numpy()


def expected(dist, k):
    """NumPy's stable argsort of the distance bits, with the count and padding rule."""
    d = dist.cpu().numpy()
    key = d.view(np.uint32)
    order = np.argsort(key, axis=1, kind="stable")
    count = np.minimum(k, (key < INF_BITS).sum(1)).astype(np.int32)
    idx = np.full((len(d), k), -1, np.int64)
    top = np.full((len(d), k), np.inf, np.float32)
    for q, c in enumerate(count):
        idx[q, :c] = order[q, :c]
        top[q, :c] = d[q, order[q, :c]]
    return idx, top, count


def check(got, k):
    dist, idx, top, cnt = got
    want_idx, want_top, want_cnt = expected(dist, k)
    np.testing.assert_array_equal(bits(cnt), want_cnt)
    np.testing.assert_array_equal(bits(idx), want_idx)
    np.testing.assert_array_equal(bits(top), want_top.view(np.uint32))


def same(a, b):
    return all(np.array_equal(bits(x), bits(y)) for x, y in zip(a, b))


@pytest.mark.parametrize("dtype", [torch.float32, torch.uint16], ids=["f32", "u16"])
@pytest.mark.parametrize("n_db", [1, 2, 1000, 4097, 100000])
def test_rank_is_the_stable_order_of_the_distances(dtype, n_db):
    r, rows = database(dtype, n_db, seed=n_db)
    qs = queries(rows, 11, seed=n_db + 1)
    for nq in (1, 3, 8, 11):
        for k in sorted({1, 10, 1024, 1025, 4096, n_db, n_db + 5}):
            got = rank(r, qs[:nq], k)
            check(got, k)
            if k <= 1024:
                assert same(got, query(r, qs[:nq], k)), (nq, k)
    if n_db >= 1000:        # the ties, the NaN query and the NaN / inf rows are there
        d = rank(r, qs, 1)[0].cpu().numpy()
        assert np.isnan(d[2]).all()
        assert (np.diff(np.sort(d[0][np.isfinite(d[0])])) == 0).sum() > n_db // 4
        if dtype == torch.float32:
            assert np.isnan(d[0]).any() and np.isposinf(d[0]).any()


@pytest.mark.parametrize("dtype", [torch.float32, torch.uint16], ids=["f32", "u16"])
@pytest.mark.parametrize("n_db", [2, 4097, 100000])
def test_spatial_filter_that_excludes_most_or_all_rows(dtype, n_db):
    r, rows = database(dtype, n_db, seed=7 * n_db)
    xyz = torch.zeros((n_db, 3), dtype=torch.float64, device="cuda")
    xyz[:, 0] = torch.arange(n_db, dtype=torch.float64)
    qs = queries(rows, 8, seed=3)
    qxyz = torch.zeros((8, 3), dtype=torch.float64, device="cuda")
    qxyz[:, 0] = torch.linspace(0, n_db - 1, 8, dtype=torch.float64)
    for radius in (0.95 * n_db, 2.0 * n_db):           # most rows excluded, then all of them
        for k in sorted({1, 10, 1024, 1025, n_db, n_db + 5}):
            got = rank(r, qs, k, xyz, qxyz, radius)
            check(got, k)
            if k <= 1024:
                assert same(got, query(r, qs, k, xyz, qxyz, radius))
        if radius > n_db:
            assert (got[3] == 0).all() and (got[1] == -1).all()


@pytest.mark.parametrize("dtype", [torch.float32, torch.uint16], ids=["f32", "u16"])
def test_workspace_needs_no_initialisation_and_any_stream_works(dtype):
    r, rows = database(dtype, 100000, seed=11)
    qs = queries(rows, 11, seed=12)
    lib = _lib.load()
    for k in (5, 1025, 100000):
        first = rank(r, qs, k)
        check(first, k)
        ws = torch.full((int(lib.nsc_wasserstein_rank_workspace_bytes(11, 100000)),), 0xFF, dtype=torch.uint8,
                        device="cuda")
        s = torch.cuda.Stream()
        assert same(first, rank(r, qs, k, ws=ws, stream=s))
        for _ in range(3):                              # the workspace now holds the last call's data
            assert same(first, rank(r, qs, k, ws=ws, stream=s))
            assert same(first, rank(r, qs, k, ws=ws))


def test_no_rows_and_top_k_zero():
    from neural_spectral_codec_b200.retrieval import WassersteinRetriever
    lib = _lib.load()
    r, rows = database(torch.float32, 1000, seed=5)
    qs = queries(rows, 3, seed=6)
    dist, idx, top, cnt = outputs(3, 1000, 0)
    st = lib.nsc_wasserstein_rank(qs.data_ptr(), 3, r._cdfs.data_ptr(), 1000, N_BINS, r.epsilon, None, None, 0.0,
                                  dist.data_ptr(), 0, None, None, None, None, 0, None)
    assert st == 0                                      # distances only: no workspace, no outputs
    torch.cuda.synchronize()
    assert same((dist,), (query(r, qs, 0)[0],))
    empty = WassersteinRetriever(device="cuda")
    dist, idx, top, cnt = outputs(3, 1, 7)                # d_distances must not be NULL, even for no rows
    ws = torch.empty(int(lib.nsc_wasserstein_rank_workspace_bytes(3, 0)), dtype=torch.uint8, device="cuda")
    st = lib.nsc_wasserstein_rank(qs.data_ptr(), 3, None, 0, N_BINS, 1e-8, None, None, 0.0, dist.data_ptr(), 7,
                                  idx.data_ptr(), top.data_ptr(), cnt.data_ptr(), ws.data_ptr(), ws.numel(), None)
    assert st == 0 and empty.database_size == 0
    torch.cuda.synchronize()
    assert (cnt == 0).all() and (idx == -1).all() and torch.isinf(top).all()


@pytest.mark.parametrize("dtype", [torch.float32, torch.uint16], ids=["f32", "u16"])
def test_query_batch_beyond_1024_ranks_the_whole_database(dtype):
    """query_batch(top_k > 1024) goes through the rank: the same bits as the entry point, and
    query(top_k=n) lists every finite row."""
    r, rows = database(dtype, 4097, seed=21)
    qs = queries(rows, 3, seed=22)
    for k in (1025, 4097, 10 ** 6):
        idx, top, cnt, dist = r.query_batch(qs, top_k=k, return_distances=True)
        kk = min(k, 4097)
        assert idx.shape == (3, kk) and top.shape == (3, kk) and cnt.dtype == torch.int32
        assert same((dist, idx, top, cnt), rank(r, qs, kk))
    qi, qd = r.query(qs[0].cpu().numpy(), top_k=4097)
    d0 = dist[0].cpu().numpy()
    assert len(qi) == np.isfinite(d0).sum() and qi.dtype == np.int64 and qd.dtype == np.float32
