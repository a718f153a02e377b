"""Device-free checks of the rank entry points (nsc_wasserstein_rank, nsc_wasserstein_rank_u16,
nsc_wasserstein_rank_workspace_bytes): argument validation happens before any CUDA call, in the order
and with the status codes of nsc_wasserstein_query, and the workspace check comes after it."""
import ctypes as C
import os

import pytest

from neural_spectral_codec_b200 import _lib

P = 256      # a non-null device address; validation never dereferences it
SIZE_MAX = 2 ** 64 - 1


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.load()


def ptr(on):
    return C.c_void_p(P) if on else None


def test_rank_validates_like_the_query_entry(lib):
    def both(nq=1, n_db=10, bins=800, k=10, q=True, db=True, dist=True, idx=True, top=True, cnt=True,
             db_xyz=False, q_xyz=False, ws=True, ws_bytes=None):
        if ws_bytes is None:
            ws_bytes = lib.nsc_wasserstein_rank_workspace_bytes(max(nq, 0), max(n_db, 0))
        args = lambda: (ptr(q), nq, ptr(db), n_db, bins, 1e-8, ptr(db_xyz), ptr(q_xyz), 0.0, ptr(dist), k,
                        ptr(idx), ptr(top), ptr(cnt), ptr(ws), ws_bytes, None)
        f = lib.nsc_wasserstein_rank(*args())
        u = lib.nsc_wasserstein_rank_u16(*args())
        assert f == u, (nq, n_db, bins, k)
        if u not in (0, -6) and 0 <= k <= 1024 and n_db < (1 << 32):
            # the query entry defines the same case and refuses it with the same code (only refused
            # cases are passed on: the addresses here are not real)
            want = lib.nsc_wasserstein_query(ptr(q), nq, ptr(db), n_db, bins, 1e-8, ptr(db_xyz), ptr(q_xyz), 0.0,
                                             ptr(dist), k, ptr(idx), ptr(top), ptr(cnt), None, 0, None)
            assert u == want, (nq, n_db, bins, k, u, want)
        return u

    assert both(nq=-1) == -3 and both(n_db=-1) == -3 and both(k=-1) == -3
    assert both(n_db=1 << 32) == -3 and both(n_db=(1 << 32) + 5, bins=0) == -3
    assert both(nq=-1, bins=0, q=False) == -3              # counts before widths before pointers
    assert both(k=-1, bins=0, ws=False) == -3
    assert both(bins=0) == -4 and both(bins=1025) == -4
    assert both(bins=1025, q=False) == -4 and both(bins=0, ws=False) == -4
    assert both(nq=0, q=False, dist=False, ws=False) == 0  # no queries: a no-op
    assert both(q=False) == -1 and both(dist=False) == -1 and both(db=False) == -1
    for missing in ("idx", "top", "cnt"):
        assert both(**{missing: False}) == -1
        assert both(k=5000, **{missing: False}) == -1
    assert both(k=0, idx=False, top=False, cnt=False, db=False) == -1     # rows still needed
    assert both(db_xyz=True) == -1 and both(q_xyz=True) == -1             # one of the positions only
    assert both(q=False, ws=False) == -1                                  # pointers before the workspace


def test_a_missing_or_small_workspace_is_refused(lib):
    def both(nq, n_db, k, ws, ws_bytes):
        args = (ptr(True), nq, ptr(True), n_db, 800, 1e-8, None, None, 0.0, ptr(True), k,
                ptr(True), ptr(True), ptr(True), ptr(ws), ws_bytes, None)
        f, u = lib.nsc_wasserstein_rank(*args), lib.nsc_wasserstein_rank_u16(*args)
        assert f == u
        return u

    for nq, n_db in ((1, 1), (3, 1000), (8, 100000), (11, 4097), (2, 0)):
        need = lib.nsc_wasserstein_rank_workspace_bytes(nq, n_db)
        assert need > 0
        for k in (1, 1024, 1025, n_db + 5):
            assert both(nq, n_db, k, False, need) == -6
            assert both(nq, n_db, k, True, need - 1) == -6
            assert both(nq, n_db, k, True, 0) == -6
            assert both(nq, n_db, k, False, 0) == -6


def test_workspace_size_is_monotone_and_zero_for_invalid_arguments(lib):
    ws = lib.nsc_wasserstein_rank_workspace_bytes
    assert ws(-1, 10) == 0 and ws(1, -1) == 0 and ws(-5, -5) == 0
    assert ws(1, 1 << 32) == 0 and ws(1, (1 << 32) + 1) == 0
    assert ws(0, 100) == 0 and ws(1, (1 << 32) - 1) > 16 * ((1 << 32) - 1)
    assert ws(2 ** 31 - 1, (1 << 32) - 1) >= ws(1, (1 << 32) - 1)
    ns = [0, 1, 2, 255, 256, 4095, 4096, 4097, 8192, 100000, 10 ** 6, 10 ** 9, (1 << 32) - 1]
    qs = [1, 2, 3, 8, 11, 1000, 65535, 65536, 2 ** 31 - 1]
    for q in qs:
        sizes = [ws(q, n) for n in ns]
        assert sizes == sorted(sizes), q
        assert all(s >= min(16 * q * n, SIZE_MAX) for s, n in zip(sizes, ns))   # two key and two row buffers
    for n in ns:
        sizes = [ws(q, n) for q in qs]
        assert sizes == sorted(sizes), n
    assert ws(2 ** 31 - 1, (1 << 32) - 1) == SIZE_MAX           # does not fit a size_t
