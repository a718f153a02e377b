#!/usr/bin/env python
"""Per-phase cycle counts of the persistent encode kernel (tuning build:
make -C neural_spectral_codec_b200/csrc VARIANT=phase DEFS=-DNSC_PHASE_TIMING, NSC_LIB=...).

    python tools/phase_timing.py [shape] [n_elevation]      (default: hdl64 16)

The generic and the tall kernels count phases; the warp-specialised one does not, so at 16 rows
run it with the tuning variant's NSC_WS=0. For images of more than 64 rows the in-place pooling
counts as part of "load signals"."""
import ctypes as C
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from neural_spectral_codec_b200 import SpectralEncoder, _lib, synth  # noqa: E402

shape = synth.SHAPES[sys.argv[1] if len(sys.argv) > 1 else "hdl64"]
rows = int(sys.argv[2]) if len(sys.argv) > 2 else 16
n = 1184                      # 4 scans per CTA
enc = SpectralEncoder(n_elevation=rows, target_elevation_bins=16,
                      elevation_range=(shape.el_lo_deg, shape.el_hi_deg) if rows > 16 else (-24.8, 2.0)).to("cuda")
pts, offs = synth.make_batch(shape, 0, n, device="cuda")
out = torch.empty((n, 800), device="cuda")
ws = torch.zeros(64, dtype=torch.int32, device="cuda")
lib = _lib.load()
p, lut = enc._params(), enc.freq_to_bin()
for _ in range(3):
    st = lib.nsc_encode_batch(pts.data_ptr(), 4, offs.data_ptr(), 0, n, C.byref(p), lut.ctypes.data,
                              out.data_ptr(), ws.data_ptr(), 256, None)
    assert st == 0
torch.cuda.synchronize()
c = ws.view(torch.int64)[2:12].cpu().tolist()      # counter + 2 + phase, 64-bit slots
names = ["scan fetch + init image", "point pass", "keys->ranges, masks, interpolation", "  bin sums (rest of spectrum)",
         "normalise + store", "  load signals (pooling, row indirection)", "  FFT pass radix 8", "  FFT pass radix 9",
         "  FFT pass radix 5", "  magnitudes"]
tot = sum(c)
for k, v in zip(names, c):
    print(f"{k:38s} {v / n:10.0f} cycles per scan  {100 * v / tot:5.1f} %")
