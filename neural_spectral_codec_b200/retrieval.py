"""Stage-1 retrieval on the GPU: 1-D Wasserstein top-K over the descriptor database.

``WassersteinRetriever`` mirrors the reference class of the same name
(reference ``src/retrieval/wasserstein.py:276-389``: ``add_to_database``, ``query``,
``clear_database``, attributes ``database_hists`` / ``database_size``). Differences that do
not change results: the database keeps, next to the histograms, their normalised CDF rows
(computed once per insert instead of on every query), and storage grows geometrically instead
of by one ``torch.cat`` per keyframe. ``query_batch`` answers many queries in one pass over
the database and takes the spatial exclusion of ``TwoStageRetrieval._global_retrieval``
(``src/retrieval/two_stage_retrieval.py:145-202``) as optional positions.

``database_dtype=torch.uint16`` keeps the database in the ``HistogramQuantizer`` wire format
instead: the rows as uint16 and their CDFs as uint16 in units of 1/65535
(``nsc_wasserstein_cdf_u16`` / ``nsc_wasserstein_query_u16``), a quarter of the float32
database's memory. Its distances are those of the float32 database of the dequantised rows. The
default stays float32, which keeps the unquantised distances. Rows and queries of either dtype go
into either database: uint16 rows are dequantised on the device, float rows going into a uint16
database are quantised on the device, both with the retriever's ``epsilon``.

``query_batch`` accepts any ``top_k``, as the reference's ``query`` does: up to ``MAX_TOP_K`` = 1024
the selection kernels of ``nsc_wasserstein_query`` pick the nearest rows; beyond that
``nsc_wasserstein_rank`` orders the whole database with a stable radix sort on the device (the
reference's ``_global_retrieval`` asks for every keyframe). Both give the order of (distance, lower
row first).

All arithmetic runs in ``libnsc_b200.so`` (``nsc_wasserstein_cdf`` / ``nsc_wasserstein_query`` /
``nsc_wasserstein_rank``); there is no CPU path.
"""
from __future__ import annotations

from typing import Optional, Tuple, Union

import numpy as np
import torch

from . import _lib

MAX_TOP_K = 1024


class WassersteinRetriever:
    def __init__(self, use_torch: bool = True, device: str = "cuda", epsilon: float = 1e-8,
                 database_dtype: torch.dtype = torch.float32):
        if database_dtype not in (torch.float32, torch.uint16):
            raise ValueError("database_dtype must be torch.float32 or torch.uint16")
        dev = torch.device(device)
        if dev.type != "cuda":
            raise RuntimeError("WassersteinRetriever: no CPU implementation; pass a CUDA device")
        _lib.load()
        self.use_torch = use_torch      # kept for signature compatibility; always the CUDA path
        self.device = dev
        self.epsilon = float(epsilon)
        self.database_dtype = database_dtype
        self._hists: Optional[torch.Tensor] = None      # capacity x n_bins
        self._cdfs: Optional[torch.Tensor] = None
        self._xyz: Optional[torch.Tensor] = None        # capacity x 3 float64 (NaN = unknown)
        self._ws: Optional[torch.Tensor] = None         # selection workspace (zero between calls)
        self._rank_ws: Optional[torch.Tensor] = None    # rank workspace (k > MAX_TOP_K; needs no zeroing)
        self.database_size = 0

    # -- database ---------------------------------------------------------------------------
    @property
    def database_hists(self) -> Optional[torch.Tensor]:
        return None if self._hists is None else self._hists[: self.database_size]

    @property
    def database_cdfs(self) -> Optional[torch.Tensor]:
        return None if self._cdfs is None else self._cdfs[: self.database_size]

    def _reserve(self, rows: int, n_bins: int) -> None:
        if self._hists is not None and self._hists.shape[1] != n_bins:
            raise ValueError("all histograms of one database must have the same number of bins")
        cap = 0 if self._hists is None else self._hists.shape[0]
        if rows <= cap:
            return
        new_cap = max(rows, 2 * cap, 1024)
        hists = torch.empty((new_cap, n_bins), dtype=self.database_dtype, device=self.device)
        cdfs = torch.empty((new_cap, n_bins), dtype=self.database_dtype, device=self.device)
        xyz = torch.full((new_cap, 3), float("nan"), dtype=torch.float64, device=self.device)
        if self.database_size:
            hists[: self.database_size] = self._hists[: self.database_size]
            cdfs[: self.database_size] = self._cdfs[: self.database_size]
            xyz[: self.database_size] = self._xyz[: self.database_size]
        self._hists, self._cdfs, self._xyz = hists, cdfs, xyz

    def _rows(self, x: Union[np.ndarray, torch.Tensor], what: str) -> torch.Tensor:
        """``(n, n_bins)`` rows on the device: uint16 rows stay uint16, anything else is float32."""
        if isinstance(x, np.ndarray):
            x = torch.from_numpy(np.ascontiguousarray(x, np.uint16 if x.dtype == np.uint16 else np.float32))
        h = x.detach().to(self.device, torch.uint16 if x.dtype == torch.uint16 else torch.float32)
        if h.dim() == 1:
            h = h.unsqueeze(0)
        if h.dim() != 2:
            raise ValueError(f"{what} must have shape (n, n_bins)")
        return h

    def _convert(self, rows: torch.Tensor, out: torch.Tensor) -> torch.Tensor:
        """float32 rows -> uint16 ``out`` (quantise) or uint16 rows -> float32 ``out`` (dequantise)."""
        lib = _lib.load()
        rows = rows.contiguous()
        name = "nsc_quantize_histograms" if out.dtype == torch.uint16 else "nsc_dequantize_histograms"
        with torch.cuda.device(self.device):
            st = getattr(lib, name)(rows.data_ptr(), rows.shape[0], rows.shape[1], self.epsilon, out.data_ptr(),
                                    torch.cuda.current_stream(self.device).cuda_stream)
        _lib.check(st, name)
        return out

    def add_to_database(self, histograms: Union[np.ndarray, torch.Tensor],
                        positions: Union[np.ndarray, torch.Tensor, None] = None) -> None:
        """Append ``(n, n_bins)`` histograms (reference :300-326); ``positions`` are optional
        ``(n, 3)`` keyframe positions (``pose[:3, 3]``) for the spatial filter of ``query_batch``.
        float rows or uint16 wire rows; they are converted to the database's dtype."""
        lib = _lib.load()
        h = self._rows(histograms, "histograms")
        n, n_bins = h.shape
        if n == 0:
            return
        lo = self.database_size
        self._reserve(lo + n, n_bins)
        if h.dtype == self.database_dtype:
            self._hists[lo: lo + n] = h
        elif h.dtype == torch.uint16:
            self._hists[lo: lo + n] = self._convert(h, torch.empty(h.shape, dtype=torch.float32, device=self.device))
        else:
            self._convert(h, self._hists[lo: lo + n])
        if positions is not None:
            p = torch.as_tensor(positions, dtype=torch.float64).reshape(n, 3)
            self._xyz[lo: lo + n] = p.to(self.device)
        stream = torch.cuda.current_stream(self.device).cuda_stream
        with torch.cuda.device(self.device):
            if self.database_dtype == torch.uint16:
                name = "nsc_wasserstein_cdf_u16"
                st = lib.nsc_wasserstein_cdf_u16(self._hists[lo: lo + n].data_ptr(), n, n_bins,
                                                 self._cdfs[lo: lo + n].data_ptr(), stream)
            else:
                name = "nsc_wasserstein_cdf"
                st = lib.nsc_wasserstein_cdf(self._hists[lo: lo + n].data_ptr(), n, n_bins, self.epsilon,
                                             self._cdfs[lo: lo + n].data_ptr(), stream)
        _lib.check(st, name)
        self.database_size = lo + n

    def clear_database(self) -> None:
        self._hists = self._cdfs = self._xyz = None
        self.database_size = 0

    # -- queries ----------------------------------------------------------------------------
    def query_batch(self, query_hists: Union[np.ndarray, torch.Tensor], top_k: int = 10,
                    query_positions: Union[np.ndarray, torch.Tensor, None] = None,
                    spatial_filter_distance: float = 0.0, return_distances: bool = False):
        """``(Q, n_bins)`` queries -> ``(indices (Q, k) int64, distances (Q, k) float32,
        counts (Q,) int32)`` on the device, ``k = min(top_k, database_size)``; rows are sorted by
        ascending distance and padded with -1 / +inf beyond ``counts[q]`` (only when the spatial
        filter leaves fewer than ``k`` candidates). With ``return_distances`` the full
        ``(Q, database_size)`` distance matrix is returned as a fourth element. Queries are float
        rows or uint16 wire rows (dequantised on the device first)."""
        lib = _lib.load()
        q = self._rows(query_hists, "queries")
        nq = q.shape[0]
        n = self.database_size
        if n and q.shape[1] != self._hists.shape[1]:
            raise ValueError("query and database bin counts differ")
        if q.dtype == torch.uint16:
            q = self._convert(q, torch.empty(q.shape, dtype=torch.float32, device=self.device))
        q = q.contiguous()
        k = min(int(top_k), n)
        dist = torch.empty((nq, n), dtype=torch.float32, device=self.device)
        idx = torch.empty((nq, k), dtype=torch.int64, device=self.device)
        top = torch.empty((nq, k), dtype=torch.float32, device=self.device)
        # every call below writes the counts, except the empty cases
        cnt = (torch.empty if (n and nq and k) else torch.zeros)((nq,), dtype=torch.int32, device=self.device)
        if n and nq:
            use_xyz = query_positions is not None and spatial_filter_distance > 0
            qp = None
            if use_xyz:
                qp = torch.as_tensor(query_positions, dtype=torch.float64).reshape(nq, 3).to(self.device).contiguous()
            u16 = "_u16" if self.database_dtype == torch.uint16 else ""
            if k <= MAX_TOP_K:
                need = int(lib.nsc_wasserstein_workspace_bytes(nq))
                if self._ws is None or self._ws.numel() < need:
                    self._ws = torch.zeros(need, dtype=torch.uint8, device=self.device)
                name, ws = "nsc_wasserstein_query" + u16, self._ws
            else:
                # the selection kernels hold k <= 1024 candidates per query; larger k (the reference's
                # _global_retrieval asks for every keyframe) ranks the whole database
                need = int(lib.nsc_wasserstein_rank_workspace_bytes(nq, n))
                if self._rank_ws is None or self._rank_ws.numel() < need:
                    self._rank_ws = torch.empty(need, dtype=torch.uint8, device=self.device)
                name, ws = "nsc_wasserstein_rank" + u16, self._rank_ws
            with torch.cuda.device(self.device):
                st = getattr(lib, name)(
                    q.data_ptr(), nq, self._cdfs.data_ptr(), n, q.shape[1], self.epsilon,
                    self._xyz.data_ptr() if use_xyz else None, qp.data_ptr() if use_xyz else None,
                    float(spatial_filter_distance), dist.data_ptr(), k,
                    idx.data_ptr() if k else None, top.data_ptr() if k else None,
                    cnt.data_ptr() if k else None, ws.data_ptr(), ws.numel(),
                    torch.cuda.current_stream(self.device).cuda_stream)
            _lib.check(st, name)
        if return_distances:
            return idx, top, cnt, dist
        return idx, top, cnt

    def query(self, query_hist: Union[np.ndarray, torch.Tensor], top_k: int = 10) -> Tuple[np.ndarray, np.ndarray]:
        """One query -> ``(indices, distances)`` as numpy, ascending (reference :328-384)."""
        if self.database_size == 0:
            return np.array([]), np.array([])
        idx, top, cnt = self.query_batch(query_hist, top_k=top_k)
        c = int(cnt[0].item())
        return idx[0, :c].cpu().numpy(), top[0, :c].cpu().numpy()


def wasserstein_distance_batch(query_hist: torch.Tensor, database_hists: torch.Tensor,
                               epsilon: float = 1e-8) -> torch.Tensor:
    """``wasserstein_distance_batch_torch`` (wasserstein.py:134-172) on CUDA tensors: ``(n_db,)``."""
    r = WassersteinRetriever(device=database_hists.device, epsilon=epsilon)
    r.add_to_database(database_hists)
    return r.query_batch(query_hist, top_k=0, return_distances=True)[3][0]
