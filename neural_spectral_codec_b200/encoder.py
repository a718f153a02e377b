"""Host-side mirror of the reference encoder interface, bound to the CUDA library.

``SpectralEncoder`` keeps the constructor, attributes and method names of the reference class
(reference ``src/encoding/spectral_encoder.py:24-261``) and ``RangeImageProjector`` those of
the reference projector (``src/encoding/range_image.py:92-232``), so the reference's callers
(``src/pipeline.py:66-73,245,351``, ``train_multi_dataset.py:264-271,182``) work unchanged:

    enc = SpectralEncoder(n_elevation=16, n_azimuth=360, n_bins=50, alpha=2.0,
                          learnable_alpha=True, target_elevation_bins=16).to("cuda")
    desc = enc.encode_points(points).detach().cpu().numpy()        # (800,) float32

All arithmetic runs in ``libnsc_b200.so`` (hand-written sm_100a kernels behind the C ABI of
``include/nsc_b200.h``). There is no CPU path: the module must live on a CUDA device and the
shared library must be present, otherwise the calls raise.

Beyond the reference surface:
  * ``encode_points_batch(points, offsets)`` -- device-resident concatenated scans in, one
    fused kernel launch, ``(B, 800)`` out (the batched entry of ``BASELINE.json``);
  * ``encode_scans(scans)`` -- host buffers in, host descriptors out, H2D / encode / D2H
    overlapped on rotating streams inside the library (the end-to-end path);
  * ``dtype=torch.uint16`` / ``dtype=np.uint16`` on both -- the descriptors in the wire format of
    ``HistogramQuantizer.quantize`` (the same integers), quantised in the encode kernel's epilogue.
"""
from __future__ import annotations

import ctypes as C
from typing import Optional, Sequence, Tuple, Union

import numpy as np
import torch
import torch.nn as nn

from . import _lib


def _no_cpu(what: str) -> RuntimeError:
    return RuntimeError(
        f"{what}: this encoder has no CPU implementation. Move it to a CUDA device first "
        "(`encoder.to('cuda')`); the reference CPU encoder is not bundled.")


class RangeImageProjector:
    """Spherical projection to an ``n_elevation x 360`` min-range image on the GPU.

    Mirrors ``RangeImageProjector`` (reference range_image.py:92-127 constructor,
    :129-232 ``project``). The encoder's path uses the geometry branch
    (``keep_intensity=False``, spectral_encoder.py:217); the intensity image is a separate kernel.
    """

    def __init__(self, n_elevation: int = 64, n_azimuth: int = 360,
                 elevation_range: Tuple[float, float] = (-24.8, 2.0),
                 max_range: float = 80.0, min_range: float = 1.0, device=None):
        if not 2 <= int(n_azimuth) <= 4096:
            raise ValueError("n_azimuth must be in [2, 4096]")
        self.n_elevation = n_elevation
        self.n_azimuth = n_azimuth
        self.max_range = max_range
        self.min_range = min_range
        self.elevation_min = np.deg2rad(elevation_range[0])   # np.float64, as the reference
        self.elevation_max = np.deg2rad(elevation_range[1])
        self.device = torch.device(device) if device is not None else None

    # -- helpers shared with SpectralEncoder ------------------------------------------------
    def _fill_params(self, p: _lib.NscParams) -> None:
        p.flags = _lib.FLAG_TALL_IMAGES       # this package handles images of up to 128 rows
        p.n_elevation = int(self.n_elevation)
        p.n_azimuth = int(self.n_azimuth)
        p.min_range = float(self.min_range)
        p.max_range = float(self.max_range)
        p.el_min_rad = float(self.elevation_min)
        p.el_max_rad = float(self.elevation_max)

    def _params(self) -> _lib.NscParams:
        p = _lib.NscParams()
        _lib.load().nsc_default_params(C.byref(p))
        self._fill_params(p)
        p.n_bins, p.target_rows = 1, 1        # the projector has no spectrum; keeps any width valid
        return p

    def project_batch(self, points: torch.Tensor, offsets: torch.Tensor,
                      interpolate: bool = False) -> torch.Tensor:
        """Concatenated device scans -> ``(B, n_elevation, 360)`` range images (optionally after
        ``interpolate_range_image``)."""
        lib = _lib.load()
        points, offsets, n_scans, stride = _check_batch(points, offsets)
        dev = points.device
        out = torch.empty((n_scans, self.n_elevation, self.n_azimuth), dtype=torch.float32, device=dev)
        p = self._params()
        if self.n_azimuth != _lib.N_AZIMUTH:
            _anywidth_points(points, offsets, n_scans, stride, p, None, None, out,
                             _lib.STAGE_INTERPOLATED if interpolate else _lib.STAGE_PROJECTED)
            return out
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            ws = _workspace(dev, stream, p, n_scans)
            st = lib.nsc_project_batch(
                points.data_ptr(), stride, offsets.data_ptr(), 0, n_scans, C.byref(p),
                _lib.STAGE_INTERPOLATED if interpolate else _lib.STAGE_PROJECTED,
                out.data_ptr(), ws.data_ptr(), ws.numel() * 4, stream)
        _lib.check(st, "nsc_project_batch")
        return out

    def project_intensity_batch(self, points: torch.Tensor, offsets: torch.Tensor):
        """Concatenated ``(sum N, 4)`` device scans -> ``(range images, intensity images)``, both
        ``(B, n_elevation, 360)`` (reference range_image.py:216-230 for the second)."""
        lib = _lib.load()
        points, offsets, n_scans, stride = _check_batch(points, offsets)
        if stride != 4:
            raise ValueError("the intensity image needs (N, 4) points")
        if self.n_azimuth != _lib.N_AZIMUTH:
            raise NotImplementedError("the intensity image (off the encoding path) is built for n_azimuth = 360 only")
        dev = points.device
        shape = (n_scans, self.n_elevation, self.n_azimuth)
        rng = torch.empty(shape, dtype=torch.float32, device=dev)
        inten = torch.empty(shape, dtype=torch.float32, device=dev)
        p = self._params()
        with torch.cuda.device(dev):
            st = lib.nsc_project_intensity_batch(points.data_ptr(), offsets.data_ptr(), 0, n_scans,
                                                 C.byref(p), rng.data_ptr(), inten.data_ptr(),
                                                 torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(st, "nsc_project_intensity_batch")
        return rng, inten

    def project(self, points: np.ndarray, keep_intensity: bool = True):
        """``project(points, keep_intensity) -> (range_image, intensity_image | None)`` as numpy,
        like the reference (range_image.py:129-232): the intensity image exists only for 4-column
        input with ``keep_intensity=True``."""
        if self.device is None or self.device.type != "cuda":
            raise _no_cpu("RangeImageProjector.project")
        a = _as_f32_points(points)
        pts, offs = _host_scan_to_device(a, self.device)
        if keep_intensity and a.shape[1] == 4:
            rng, inten = self.project_intensity_batch(pts, offs)
            return rng[0].cpu().numpy(), inten[0].cpu().numpy()
        img = self.project_batch(pts, offs)[0]
        return img.cpu().numpy(), None


_WORKSPACES = {}


def _workspace(dev: torch.device, stream: int, p: "_lib.NscParams", n_scans: int) -> torch.Tensor:
    """Device workspace of the encode kernels (``nsc_workspace_bytes``: the work counter plus room
    to split the scans of the grid's last wave), one per (device, stream): launches on one
    stream are ordered, so they can share it."""
    need = int(_lib.load().nsc_workspace_bytes(n_scans, C.byref(p)))
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), stream)
    ws = _WORKSPACES.get(key)
    if ws is None or ws.numel() * 4 < need:
        ws = torch.empty((need + 3) // 4, dtype=torch.int32, device=dev)
        _WORKSPACES[key] = ws
    return ws


def _anywidth_need(p: "_lib.NscParams", n: int, rows: int) -> int:
    """Workspace bytes of the kernels for widths other than 360; ValueError outside their envelope."""
    need = int(_lib.load().nsc_anywidth_workspace_bytes(n, rows, C.byref(p)))
    if need == 0:
        raise ValueError("encoder geometry outside the supported envelope (rows <= 128, 2 <= n_azimuth <= 4096, "
                         "n_bins <= n_azimuth // 2 + 1)")
    return need


def _anywidth_workspace(dev: torch.device, stream: int, p: "_lib.NscParams", n: int, rows: int) -> torch.Tensor:
    need = _anywidth_need(p, n, rows)
    key = (dev.index if dev.index is not None else torch.cuda.current_device(), stream, "anywidth")
    ws = _WORKSPACES.get(key)
    if ws is None or ws.numel() * 4 < need:
        ws = torch.empty((need + 3) // 4, dtype=torch.int32, device=dev)
        _WORKSPACES[key] = ws
    return ws


def _anywidth_points(points, offsets, n_scans, stride, p, lut, out, images, stage):
    """Widths other than 360 (``nsc_anywidth_points``): the fused shared-memory kernel for
    descriptors at widths whose prime factors are at most 13 and images that fit one block's
    shared memory, the general kernel otherwise (and for images alone). A uint16 ``out`` takes
    ``nsc_anywidth_points_u16`` (same kernel, quantised in its epilogue; no images)."""
    dev = points.device
    u16 = out is not None and out.dtype == torch.uint16
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        ws = _anywidth_workspace(dev, stream, p, n_scans, p.n_elevation)
        if u16:
            st = _lib.load().nsc_anywidth_points_u16(
                points.data_ptr(), stride, offsets.data_ptr(), 0, n_scans, C.byref(p), lut.ctypes.data,
                _lib.QUANT_EPSILON, out.data_ptr(), ws.data_ptr(), ws.numel() * 4, stream)
        else:
            st = _lib.load().nsc_anywidth_points(
                points.data_ptr(), stride, offsets.data_ptr(), 0, n_scans, C.byref(p),
                lut.ctypes.data if lut is not None else None, out.data_ptr() if out is not None else None,
                images.data_ptr() if images is not None else None, stage, ws.data_ptr(), ws.numel() * 4, stream)
    _lib.check(st, "nsc_anywidth_points_u16" if u16 else "nsc_anywidth_points")


def _anywidth_images(x, p, lut, method, out, images_out):
    dev = x.device
    with torch.cuda.device(dev):
        stream = torch.cuda.current_stream(dev).cuda_stream
        ws = _anywidth_workspace(dev, stream, p, x.shape[0], x.shape[1])
        st = _lib.load().nsc_anywidth_images(
            x.data_ptr(), x.shape[0], x.shape[1], C.byref(p), lut.ctypes.data if lut is not None else None, method,
            out.data_ptr() if out is not None else None, images_out.data_ptr() if images_out is not None else None,
            ws.data_ptr(), ws.numel() * 4, stream)
    _lib.check(st, "nsc_anywidth_images")


def _check_batch(points: torch.Tensor, offsets: torch.Tensor):
    if not isinstance(points, torch.Tensor) or not points.is_cuda:
        raise _no_cpu("points must be a CUDA tensor")
    if points.dtype != torch.float32 or points.dim() != 2 or points.shape[1] not in (3, 4):
        raise ValueError("points must be float32 of shape (sum N, 3) or (sum N, 4)")
    points = points.contiguous()
    offsets = torch.as_tensor(offsets)
    if offsets.dim() != 1 or offsets.numel() < 1:
        raise ValueError("offsets must be a 1-D tensor of B+1 point offsets")
    if not offsets.is_cuda:   # host offsets are cheap to validate; device offsets are the caller's contract
        o = offsets.to(torch.int64)
        if int(o[0]) < 0 or int(o[-1]) > points.shape[0] or bool((o[1:] < o[:-1]).any()):
            raise ValueError("offsets must be non-decreasing, start at >= 0 and end at <= len(points)")
    offsets = offsets.to(device=points.device, dtype=torch.int64).contiguous()
    return points, offsets, offsets.numel() - 1, points.shape[1]


def _as_f32_points(points) -> np.ndarray:
    """What the reference's ``points[:, 0..2]`` indexing accepts, as contiguous float32."""
    a = np.asarray(points)
    if a.ndim != 2 or a.shape[1] < 3:
        raise ValueError("points must have shape (N, 3) or (N, 4)")
    if a.shape[1] > 4:
        a = a[:, :3]
    return np.ascontiguousarray(a, dtype=np.float32)


def _host_scan_to_device(points, device) -> Tuple[torch.Tensor, torch.Tensor]:
    a = _as_f32_points(points)
    pts = torch.from_numpy(a).to(device)
    offs = torch.tensor([0, a.shape[0]], dtype=torch.int64).to(device)
    return pts, offs


class SpectralEncoder(nn.Module):
    """Per-elevation spectral histogram encoder (``target_elevation_bins * n_bins`` = 800-D).

    Constructor arguments are the reference's (spectral_encoder.py:35-47).
    """

    def __init__(self, n_elevation: int = 64, n_azimuth: int = 360, n_bins: int = 50,
                 alpha: float = 2.0, learnable_alpha: bool = True, epsilon: float = 1e-8,
                 target_elevation_bins: int = 16, interpolate_empty: bool = True,
                 elevation_range: tuple = (-24.8, 2.0), device: str = "cpu"):
        super().__init__()
        _lib.load()   # fail at construction if the CUDA library is absent
        self.n_elevation = n_elevation
        self.n_azimuth = n_azimuth
        self.n_bins = n_bins
        self.epsilon = epsilon
        self.target_elevation_bins = target_elevation_bins
        self.interpolate_empty = interpolate_empty
        self._device = device   # stored and unused, like the reference (:71); .to() decides
        if learnable_alpha:
            self.alpha = nn.Parameter(torch.tensor(alpha, dtype=torch.float32))
        else:
            self.register_buffer("alpha", torch.tensor(alpha, dtype=torch.float32))
        self.projector = RangeImageProjector(n_elevation=n_elevation, n_azimuth=n_azimuth,
                                             elevation_range=elevation_range)
        self.n_freqs = n_azimuth // 2 + 1
        self.output_dim = target_elevation_bins * n_bins
        self._lut_key = None
        self._lut = None
        self._pipelines = {}    # name -> (nsc_pipeline handle, (device, chunk, n_buffers))

    # ------------------------------------------------------------------ constants
    def _compute_bin_edges(self, alpha: torch.Tensor) -> torch.Tensor:
        """Exponential bin edges, the reference's formula with the reference's torch calls
        (spectral_encoder.py:107-114) evaluated on the host in float32."""
        a = alpha.detach().to("cpu", torch.float32)
        t = torch.linspace(0, 1, self.n_bins + 1)
        edges = (torch.exp(a * t) - 1) / (torch.exp(a) - 1 + self.epsilon)
        return edges * self.n_freqs

    def freq_to_bin(self) -> np.ndarray:
        """int32 ``(181,)`` frequency -> bin table (spectral_encoder.py:136-145). Recomputed
        only when ``alpha`` is modified (tensor version counter)."""
        key = (self.alpha._version, self.alpha.data_ptr(), self.n_bins, self.epsilon)
        if key != self._lut_key:
            edges = self._compute_bin_edges(self.alpha)
            k = torch.arange(self.n_freqs, dtype=torch.float32)
            b = torch.clamp(torch.searchsorted(edges, k, right=True) - 1, 0, self.n_bins - 1)
            self._lut = np.ascontiguousarray(b.numpy().astype(np.int32))
            self._lut_key = key
        return self._lut

    def _params(self) -> _lib.NscParams:
        p = _lib.NscParams()
        _lib.load().nsc_default_params(C.byref(p))
        self.projector._fill_params(p)
        p.n_bins = int(self.n_bins)
        p.target_rows = int(self.target_elevation_bins)
        p.interpolate_empty = 1 if self.interpolate_empty else 0
        p.epsilon = float(self.epsilon)
        return p

    def _cuda_device(self, what: str) -> torch.device:
        dev = self.alpha.device
        if dev.type != "cuda":
            raise _no_cpu(what)
        self.projector.device = dev
        return dev

    def _apply(self, fn, *a, **k):   # keep the projector's device in step with .to()/.cuda()
        out = super()._apply(fn, *a, **k)
        self.projector.device = self.alpha.device
        return out

    # ------------------------------------------------------------------ points in
    def encode_points_batch(self, points: torch.Tensor, offsets: torch.Tensor,
                            out: Optional[torch.Tensor] = None, dtype: torch.dtype = torch.float32) -> torch.Tensor:
        """``B`` scans concatenated on the device -> ``(B, output_dim)`` float32 on the device.

        points: float32 ``(sum N, 3|4)`` CUDA tensor, rows xyz[i] as the reference loaders give
        them; offsets: int64 ``(B+1,)`` point offsets. One fused kernel launch on the current
        stream; nothing synchronises.

        ``dtype=torch.uint16`` returns the rows in the wire format instead: the integers
        ``HistogramQuantizer(output_dim).quantize`` gives for the float32 rows (epsilon 1e-8, each
        row summing to 65535), quantised in the same kernel launch at every image width. ``out``, if
        given, has ``dtype``.
        """
        lib = _lib.load()
        if dtype not in (torch.float32, torch.uint16):
            raise ValueError("dtype must be torch.float32 or torch.uint16")
        points, offsets, n_scans, stride = _check_batch(points, offsets)
        dev = points.device
        if out is None:
            out = torch.empty((n_scans, self.output_dim), dtype=dtype, device=dev)
        elif (out.shape != (n_scans, self.output_dim) or out.dtype != dtype
              or not out.is_contiguous() or out.device != dev):
            raise ValueError(f"out must be a contiguous {str(dtype)[6:]} (B, output_dim) tensor on the same device")
        p = self._params()
        lut = self.freq_to_bin()
        if self.n_azimuth != _lib.N_AZIMUTH:
            _anywidth_points(points, offsets, n_scans, stride, p, lut, out, None, _lib.STAGE_INTERPOLATED)
            return out
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            ws = _workspace(dev, stream, p, n_scans)
            if dtype == torch.uint16:
                st = lib.nsc_encode_batch_u16(points.data_ptr(), stride, offsets.data_ptr(), 0, n_scans,
                                              C.byref(p), lut.ctypes.data, _lib.QUANT_EPSILON, out.data_ptr(),
                                              ws.data_ptr(), ws.numel() * 4, stream)
                _lib.check(st, "nsc_encode_batch_u16")
                return out
            st = lib.nsc_encode_batch(points.data_ptr(), stride, offsets.data_ptr(), 0, n_scans,
                                      C.byref(p), lut.ctypes.data, out.data_ptr(), ws.data_ptr(),
                                      ws.numel() * 4, stream)
        _lib.check(st, "nsc_encode_batch")
        return out

    def encode_points(self, points: np.ndarray) -> torch.Tensor:
        """One scan ``(N, 3|4)`` -> ``(output_dim,)`` on ``alpha.device``
        (spectral_encoder.py:206-229)."""
        dev = self._cuda_device("encode_points")
        if isinstance(points, torch.Tensor):
            pts = points.to(dev, torch.float32)
            if pts.dim() != 2 or pts.shape[1] < 3:
                raise ValueError("points must have shape (N, 3) or (N, 4)")
            if pts.shape[1] > 4:
                pts = pts[:, :3]
            offs = torch.tensor([0, pts.shape[0]], dtype=torch.int64).to(dev)
            return self.encode_points_batch(pts, offs)[0]
        return self._encode_host_scan(_as_f32_points(points), dev)

    def _encode_host_scan(self, a: np.ndarray, dev: torch.device) -> torch.Tensor:
        """One pageable numpy scan -> descriptor on the device through ``nsc_pipeline_encode_scan``
        (pinned staging in pieces overlapped with their DMA, kernel on the current stream)."""
        index = dev.index if dev.index is not None else torch.cuda.current_device()
        cap = max(1 << 18, int(a.shape[0]))
        pl = self._cached_pipeline("scan", (index, cap, 3), lambda k: k[0] == index and k[1] >= cap)
        out = torch.empty((self.output_dim,), dtype=torch.float32, device=dev)
        p = self._params()
        if self.n_azimuth != _lib.N_AZIMUTH:
            _anywidth_need(p, 1, p.n_elevation)
        lut = self.freq_to_bin()
        st = _lib.load().nsc_pipeline_encode_scan(pl, a.ctypes.data, a.shape[1], a.shape[0], C.byref(p),
                                                  lut.ctypes.data, out.data_ptr(),
                                                  torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(st, "nsc_pipeline_encode_scan")
        return out

    def encode_scans(self, scans: Union[Sequence[np.ndarray], Tuple[np.ndarray, np.ndarray]],
                     out: Optional[np.ndarray] = None, max_chunk_points: int = 4_000_000,
                     n_buffers: int = 3, dtype=np.float32) -> np.ndarray:
        """Host scans in, host descriptors out: ``(B, output_dim)`` float32 numpy.

        ``scans`` is a list of ``(N_i, 4)`` (or all ``(N_i, 3)``) float32 arrays, or a tuple
        ``(points, offsets)`` of an already concatenated host buffer (pinned memory gives the
        full PCIe rate). Copies and the fused kernel overlap on ``n_buffers`` streams inside
        ``nsc_pipeline_encode``; the call returns when ``out`` is complete.

        ``dtype=np.uint16`` returns the wire format of ``encode_points_batch(..., dtype=torch.uint16)``
        (``*_u16`` pipeline entry points: half the bytes cross PCIe, no float32 rows on the host);
        ``out``, if given, has ``dtype``.
        """
        lib = _lib.load()
        dtype = np.dtype(dtype)
        if dtype not in (np.float32, np.uint16):
            raise ValueError("dtype must be np.float32 or np.uint16")
        u16 = dtype == np.uint16
        dev = self._cuda_device("encode_scans")
        arrs = None
        if isinstance(scans, tuple) and len(scans) == 2 and np.ndim(scans[1]) == 1:
            pts = scans[0]
            if isinstance(pts, torch.Tensor):
                pts = pts.numpy()
            offs = scans[1].numpy() if isinstance(scans[1], torch.Tensor) else np.asarray(scans[1])
            if pts.dtype != np.float32 or pts.ndim != 2 or pts.shape[1] not in (3, 4) \
                    or not pts.flags.c_contiguous:
                raise ValueError("points must be contiguous float32 (sum N, 3|4)")
            offs = np.ascontiguousarray(offs, dtype=np.int64)
            if offs.ndim != 1 or offs.shape[0] < 1 or offs[0] < 0 or offs[-1] > pts.shape[0] \
                    or (np.diff(offs) < 0).any():
                raise ValueError("offsets must be non-decreasing, start at >= 0 and end at <= len(points)")
        else:
            arrs = [_as_f32_points(s) for s in scans]
            widths = {a.shape[1] for a in arrs}
            if len(widths) > 1:
                arrs = [np.ascontiguousarray(a[:, :3]) for a in arrs]
            offs = np.zeros(len(arrs) + 1, np.int64)
            np.cumsum([a.shape[0] for a in arrs], out=offs[1:])
        n_scans = offs.shape[0] - 1
        if out is None:
            out = np.empty((n_scans, self.output_dim), dtype)
        elif out.shape != (n_scans, self.output_dim) or out.dtype != dtype or not out.flags.c_contiguous:
            raise ValueError(f"out must be contiguous {dtype.name} (B, output_dim)")
        if n_scans == 0:
            return out
        biggest = int(np.diff(offs).max())
        chunk = max(int(max_chunk_points), biggest)
        key = (dev.index if dev.index is not None else torch.cuda.current_device(), chunk, n_buffers)
        pl = self._cached_pipeline("batch", key, key.__eq__)
        p = self._params()
        if self.n_azimuth != _lib.N_AZIMUTH:
            _anywidth_need(p, 1, p.n_elevation)
        lut = self.freq_to_bin()
        if arrs is not None:   # separate host arrays: gathered into pinned staging inside the library
            ptrs = (C.c_void_p * n_scans)(*[a.ctypes.data for a in arrs])
            counts = np.diff(offs)
            name = "nsc_pipeline_encode_scans"
            args = (pl, ptrs, counts.ctypes.data, arrs[0].shape[1], n_scans, C.byref(p), lut.ctypes.data)
        else:
            name = "nsc_pipeline_encode"
            args = (pl, pts.ctypes.data, pts.shape[1], pts.shape[0], offs.ctypes.data, n_scans, C.byref(p),
                    lut.ctypes.data)
        if u16:
            name += "_u16"
            args += (_lib.QUANT_EPSILON,)
        _lib.check(getattr(lib, name)(*args, out.ctypes.data), name)
        return out

    def _cached_pipeline(self, name: str, key: Tuple[int, int, int], keep) -> C.c_void_p:
        """The pipeline cached as ``name``, kept while ``keep(its key)`` holds and otherwise replaced
        by ``nsc_pipeline_create(chunk, n_buffers, device)`` for ``key = (device, chunk, n_buffers)``."""
        cached = self._pipelines.get(name)
        if cached is not None and keep(cached[1]):
            return cached[0]
        lib = _lib.load()
        if cached is not None:
            del self._pipelines[name]
            lib.nsc_pipeline_destroy(cached[0])
        h = C.c_void_p()
        _lib.check(lib.nsc_pipeline_create(key[1], key[2], key[0], C.byref(h)), "nsc_pipeline_create")
        self._pipelines[name] = (h, key)
        return h

    def _close_pipeline(self) -> None:
        pipelines = getattr(self, "_pipelines", {})
        while pipelines:
            _lib.load().nsc_pipeline_destroy(pipelines.popitem()[1][0])

    def __del__(self):
        try:
            self._close_pipeline()
        except Exception:
            pass

    # ------------------------------------------------------------------ range images in
    def forward(self, x: torch.Tensor) -> torch.Tensor:
        """``(B, rows, 360)`` range images -> ``(B, output_dim)``; no projection and no
        interpolation, rows average-pooled to ``target_elevation_bins`` when they differ
        (spectral_encoder.py:231-249, :171-176)."""
        lib = _lib.load()
        dev = self._cuda_device("forward")
        if x.dim() != 3 or x.shape[2] != self.n_azimuth:
            raise ValueError("expected (batch, n_elevation, n_azimuth) range images")
        if x.requires_grad and torch.is_grad_enabled():
            # the reference's forward is differentiable w.r.t. the range image; this kernel is
            # forward-only (no caller of the reference backpropagates through the encoder:
            # gnn/trainer.py:115-119 optimises the GNN only, and every call site detaches)
            raise RuntimeError("SpectralEncoder.forward is forward-only on this backend: call it under "
                               "torch.no_grad() or pass range_images.detach()")
        x = x.detach().to(dev, torch.float32).contiguous()
        out = torch.empty((x.shape[0], self.output_dim), dtype=torch.float32, device=dev)
        p = self._params()
        lut = self.freq_to_bin()
        if self.n_azimuth != _lib.N_AZIMUTH:
            if x.shape[0]:
                _anywidth_images(x, p, lut, -1, out, None)
            return out
        with torch.cuda.device(dev):
            st = lib.nsc_encode_range_images(x.data_ptr(), x.shape[0], x.shape[1], C.byref(p),
                                             lut.ctypes.data, out.data_ptr(),
                                             torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(st, "nsc_encode_range_images")
        return out

    def encode_batch(self, range_images: torch.Tensor) -> torch.Tensor:
        return self.forward(range_images)

    def encode_range_image(self, range_image: torch.Tensor) -> torch.Tensor:
        """``(rows, 360)`` -> ``(output_dim,)`` (spectral_encoder.py:160-204)."""
        return self.forward(range_image.unsqueeze(0))[0]


def interpolate_range_image(range_image: Union[np.ndarray, torch.Tensor], method: str = "linear",
                            device="cuda"):
    """``interpolate_range_image`` of the reference (range_image.py:15-89) on the GPU. Accepts a
    ``(rows, width)`` image or a ``(B, rows, width)`` batch; numpy in -> numpy out."""
    if method not in ("linear", "nearest"):
        # the reference silently leaves the holes of partly filled rows for any other string
        raise ValueError("method must be 'linear' or 'nearest'")
    lib = _lib.load()
    is_np = isinstance(range_image, np.ndarray)
    x = torch.from_numpy(np.ascontiguousarray(range_image, np.float32)) if is_np else range_image
    single = x.dim() == 2
    if single:
        x = x.unsqueeze(0)
    if not x.is_cuda:
        x = x.to(device)
    x = x.to(torch.float32).contiguous()
    out = torch.empty_like(x)
    if x.shape[2] != _lib.N_AZIMUTH:             # other widths: the general kernel (images only)
        p = _lib.NscParams()
        lib.nsc_default_params(C.byref(p))
        p.n_azimuth, p.n_elevation, p.target_rows, p.n_bins = int(x.shape[2]), int(x.shape[1]), 1, 1
        p.flags = _lib.FLAG_TALL_IMAGES
        if x.shape[0]:
            _anywidth_images(x, p, None, 1 if method == "nearest" else 0, None, out)
        if single:
            out = out[0]
        return out.cpu().numpy() if is_np else out
    with torch.cuda.device(x.device):
        st = lib.nsc_interpolate_range_images(x.data_ptr(), x.shape[0], x.shape[1],
                                              1 if method == "nearest" else 0, out.data_ptr(),
                                              torch.cuda.current_stream(x.device).cuda_stream)
    _lib.check(st, "nsc_interpolate_range_images")
    if single:
        out = out[0]
    return out.cpu().numpy() if is_np else out


def test_rotation_invariance(encoder: SpectralEncoder, points: np.ndarray, n_rotations: int = 8) -> float:
    """Max |difference| between descriptors of yaw-rotated copies of one cloud -- the only
    property the reference states for this path (spectral_encoder.py:365-415)."""
    descs = []
    for k in range(n_rotations):
        a = 2 * np.pi * k / n_rotations
        rot = np.array([[np.cos(a), -np.sin(a), 0], [np.sin(a), np.cos(a), 0], [0, 0, 1]])
        p = np.array(points, dtype=np.float32, copy=True)
        p[:, :3] = points[:, :3] @ rot.T
        descs.append(encoder.encode_points(p).detach().cpu().numpy())
    d = np.stack(descs)
    return float(max(np.abs(d[i] - d[j]).max() for i in range(len(d)) for j in range(i + 1, len(d))))


test_rotation_invariance.__test__ = False   # a helper taking arguments, not a pytest test
