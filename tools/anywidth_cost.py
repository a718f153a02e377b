#!/usr/bin/env python
"""What do image widths other than 360 cost? A device-resident batch of HDL-64-shaped scans (far
larger than the 126 MB L2) is encoded by nsc_anywidth_points at n_azimuth = 512, 1024, 2048 and
180 (16 rows, 16 target rows, 50 bins), by both kernels of csrc/nsc_anywidth.cu:

    fused     the product library (image, FFT and histogram in shared memory)
    general   the tuning build with NSC_ANYWIDTH=0 (image and spectrum in a global scratch,
              direct float64 DFT)

launch by launch alternating, each launch timed with CUDA events. Bytes moved per launch: 16 per
point plus 4 * D per descriptor; the share given is of the 6547.8 GB/s copy peak the project
measures shares against (profiles/README.md). The GPU name and power limit are read in the same
run. The two kernels' descriptors of the timed batch must meet the suite's bars (allclose rtol
1e-4 / atol 1e-7, relative L2 <= 1e-5 per row), or the run fails.

    python tools/anywidth_cost.py [--scans 2048] [--launches 30] [--widths 512,1024,2048,180]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import numpy as np
import torch

os.environ["NSC_ANYWIDTH"] = "0"          # read by the tuning build only: its general kernel
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from neural_spectral_codec_b200 import SpectralEncoder, _lib, synth  # noqa: E402

COPY_PEAK_GBS = 6547.8


def gpu_state():
    q = "name,power.limit,clocks.sm,clocks.max.sm,temperature.gpu"
    r = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip() or r.stderr.strip()


def load_variant(path):
    lib = C.CDLL(os.path.abspath(path))
    for name, (res, args) in _lib.SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    return lib


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scans", type=int, default=2048)
    ap.add_argument("--launches", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--widths", default="512,1024,2048,180")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda")
    state0 = gpu_state()
    points, offsets = synth.make_batch_resident(synth.HDL64, 0, a.scans, dev)
    n, n_points = a.scans, int(offsets[-1])
    stream = torch.cuda.current_stream(dev).cuda_stream
    libs = {"fused": _lib.load(), "general": load_variant(_lib.TUNE_LIB_PATH)}
    runs = {}
    for W in (int(w) for w in a.widths.split(",")):
        enc = SpectralEncoder(n_elevation=16, n_azimuth=W, n_bins=50, target_elevation_bins=16).to(dev)
        p = enc._params()
        for lname, lib in libs.items():
            path = lib.nsc_test_anywidth_path(C.byref(p), 16, 1)
            assert path == (1 if lname == "fused" else 0), (lname, W, path)
            nbytes = int(lib.nsc_anywidth_workspace_bytes(n, 16, C.byref(p)))
            ws = torch.empty((nbytes + 3) // 4, dtype=torch.int32, device=dev)
            out = torch.empty((n, enc.output_dim), dtype=torch.float32, device=dev)
            runs[f"W{W}_{lname}"] = (lib, p, enc.freq_to_bin(), enc.output_dim, ws, out)

    def launch(k):
        lib, p, lut, D, ws, out = runs[k]
        _lib.check(lib.nsc_anywidth_points(points.data_ptr(), 4, offsets.data_ptr(), 0, n, C.byref(p),
                                           lut.ctypes.data, out.data_ptr(), None, _lib.STAGE_INTERPOLATED,
                                           ws.data_ptr(), ws.numel() * 4, stream), k)

    for k in runs:
        for _ in range(a.warmup):
            launch(k)
    torch.cuda.synchronize()
    times = {k: [] for k in runs}
    ev = {k: (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for k in runs}
    for _ in range(a.launches):
        for k in runs:
            ev[k][0].record()
            launch(k)
            ev[k][1].record()
        torch.cuda.synchronize()
        for k in runs:
            times[k].append(ev[k][0].elapsed_time(ev[k][1]))
    state1 = gpu_state()
    print(f"# {n} HDL-64 scans, {n_points} points ({16 * n_points / 1e9:.2f} GB), 16 rows, target_rows 16, "
          f"50 bins, {a.launches} launches each, alternating")
    print(f"# gpu before: {state0}")
    print(f"# gpu after:  {state1}")
    rec = {"gpu": state0, "scans": n, "points": n_points, "launches": a.launches, "runs": {}, "agree": {}}
    ok = True
    for k in runs:
        D = runs[k][3]
        s = sorted(times[k])
        med = statistics.median(s)
        nbytes = 16 * n_points + 4 * D * n
        r = {"median_ms": med, "p10_ms": s[len(s) // 10], "p90_ms": s[(9 * len(s)) // 10],
             "scans_per_s": n / (med * 1e-3), "GB_per_s": nbytes / (med * 1e-3) / 1e9,
             "share_of_copy_peak": nbytes / (med * 1e-3) / 1e9 / COPY_PEAK_GBS}
        rec["runs"][k] = r
        print(f"{k:14s} median {med:9.3f} ms  p10 {r['p10_ms']:9.3f}  p90 {r['p90_ms']:9.3f}  "
              f"{r['scans_per_s']:10.0f} scans/s  {r['GB_per_s']:7.1f} GB/s  "
              f"{100 * r['share_of_copy_peak']:5.1f} % of copy peak")
    for W in (int(w) for w in a.widths.split(",")):
        got = runs[f"W{W}_fused"][5].cpu().numpy().astype(np.float64)
        ref = runs[f"W{W}_general"][5].cpu().numpy().astype(np.float64)
        close = bool(np.all(np.abs(got - ref) <= 1e-7 + 1e-4 * np.abs(ref)))
        l2 = float((np.linalg.norm(got - ref, axis=1) / np.linalg.norm(ref, axis=1)).max())
        speedup = rec["runs"][f"W{W}_fused"]["scans_per_s"] / rec["runs"][f"W{W}_general"]["scans_per_s"]
        rec["agree"][W] = {"allclose": close, "max_rel_l2": l2, "max_abs": float(np.abs(got - ref).max()),
                           "speedup": speedup}
        ok = ok and close and l2 <= 1e-5
        print(f"W={W:5d} fused / general {speedup:7.1f} x scans/s; descriptors allclose {close}, "
              f"max relative L2 {l2:.2e}, max |diff| {rec['agree'][W]['max_abs']:.2e}")
    print(json.dumps(rec))
    if not ok:
        raise SystemExit("the fused kernel's descriptors miss the bars against the general kernel")


if __name__ == "__main__":
    main()
