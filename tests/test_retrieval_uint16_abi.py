"""Device-free checks of the uint16 retrieval entry points (nsc_wasserstein_cdf_u16,
nsc_wasserstein_query_u16): argument validation happens before any CUDA call, in the order and with
the status codes of nsc_wasserstein_cdf and nsc_wasserstein_query."""
import ctypes as C
import os

import pytest
import torch

from neural_spectral_codec_b200 import _lib

P = 256      # a non-null device address; validation never dereferences it


@pytest.fixture(scope="module")
def lib():
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.load()


def ptr(on):
    return C.c_void_p(P) if on else None


def test_cdf_u16_validates_like_the_float_entry(lib):
    def both(n=1, bins=800, rows=True, out=True):
        f = lib.nsc_wasserstein_cdf(ptr(rows), n, bins, 1e-8, ptr(out), None)
        u = lib.nsc_wasserstein_cdf_u16(ptr(rows), n, bins, ptr(out), None)
        assert f == u, (n, bins, rows, out)
        return u

    assert both(n=-1) == -3
    assert both(n=-1, bins=0, rows=False) == -3           # the count is checked first
    assert both(bins=0) == -4 and both(bins=1025) == -4
    assert both(bins=0, rows=False, out=False) == -4      # then the width
    assert both(n=0, rows=False, out=False) == 0          # no rows: a no-op, pointers unused
    assert both(rows=False) == -1 and both(out=False) == -1


def test_query_u16_validates_like_the_float_entry(lib):
    def both(nq=1, n_db=10, bins=800, k=10, q=True, db=True, dist=True, idx=True, top=True, cnt=True,
             db_xyz=False, q_xyz=False):
        args = lambda: (ptr(q), nq, ptr(db), n_db, bins, 1e-8, ptr(db_xyz), ptr(q_xyz), 0.0, ptr(dist), k,
                        ptr(idx), ptr(top), ptr(cnt), None, 0, None)
        f = lib.nsc_wasserstein_query(*args())
        u = lib.nsc_wasserstein_query_u16(*args())
        assert f == u
        return u

    assert both(nq=-1) == -3 and both(n_db=-1) == -3 and both(k=-1) == -3
    assert both(nq=-1, bins=0, q=False) == -3             # counts before widths before pointers
    assert both(bins=0) == -4 and both(bins=1025) == -4 and both(k=1025) == -4
    assert both(bins=1025, q=False) == -4
    assert both(n_db=1 << 32) == -3
    assert both(nq=0, q=False, dist=False) == 0           # no queries: a no-op
    assert both(q=False) == -1 and both(dist=False) == -1
    assert both(db=False) == -1
    for missing in ("idx", "top", "cnt"):
        assert both(**{missing: False}) == -1
    assert both(k=0, idx=False, top=False, cnt=False, db=False) == -1     # rows still needed
    assert both(db_xyz=True) == -1 and both(q_xyz=True) == -1             # one of the positions only


def test_retriever_refuses_other_database_dtypes(lib):
    from neural_spectral_codec_b200.retrieval import WassersteinRetriever
    for dt in (torch.float16, torch.int16, torch.float64):
        with pytest.raises(ValueError, match="database_dtype"):
            WassersteinRetriever(device="cuda", database_dtype=dt)
    with pytest.raises(RuntimeError, match="no CPU implementation"):
        WassersteinRetriever(device="cpu", database_dtype=torch.uint16)
