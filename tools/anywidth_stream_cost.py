#!/usr/bin/env python
"""What does a host-memory encode cost at image widths other than 360? Measured on one GPU:

  end to end  encode_scans of HDL-64-shaped scans (far larger than the 126 MB L2) at 1024 x 16,
              2048 x 16 (fused kernel) and 64 x 1024 (general kernel), from a pinned concatenated
              buffer and from a list of pageable arrays, float32 and uint16 rows:
                old   the earlier path of encode_scans at these widths, reproduced here: concatenate
                      on the host, one torch copy, one device batch, one copy back
                new   encode_scans: the host-buffer pipeline (nsc_pipeline_encode[_scans][_u16])
                h2d   the bare pinned host-to-device copy of the same point bytes (the ceiling)
              plus the peak torch-allocated device memory of each call (the pipeline's own buffers
              are allocated by the library, outside torch: their size is printed beside it);
  device u16  nsc_anywidth_points_u16 against nsc_anywidth_points + nsc_quantize_histograms on a
              device-resident batch at 1024 x 16, launches alternating, CUDA events;
  per scan    encode_points(numpy) at 1024 columns: old (a pageable torch copy, then a one-scan
              batch) against new (nsc_pipeline_encode_scan), each call ending in a synchronise.

Old and new alternate call by call; medians of --reps repetitions are reported. Old and new
outputs must be equal bit for bit on every timed input, or the run fails. The GPU name and power
limit are read in the same run.

    python tools/anywidth_stream_cost.py [--scans 1024] [--reps 10] [--device-scans 2048] [--launches 30]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from neural_spectral_codec_b200 import SpectralEncoder, _lib, synth  # noqa: E402


def gpu_state():
    q = "name,power.limit,clocks.sm,clocks.max.sm,temperature.gpu"
    r = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip() or r.stderr.strip()


def encoder(rows, W):
    return SpectralEncoder(n_elevation=rows, n_azimuth=W, n_bins=50, target_elevation_bins=16).to("cuda")


def host_scans(n, distinct=64):
    """n HDL-64 scans (distinct different ones, repeated), as a list of pageable arrays."""
    base = [synth.make_scan(synth.HDL64, 1000 + i).numpy() for i in range(distinct)]
    return [base[i % distinct].copy() for i in range(n)]


def old_encode_scans(enc, scans, u16):
    """encode_scans at widths other than 360 before the pipeline took them."""
    if isinstance(scans, tuple):
        host, offs = scans
    else:
        host = np.concatenate(scans)
        offs = np.zeros(len(scans) + 1, np.int64)
        np.cumsum([len(s) for s in scans], out=offs[1:])
    d = enc.encode_points_batch(torch.from_numpy(np.ascontiguousarray(host)).to("cuda"), torch.from_numpy(offs),
                                dtype=torch.uint16 if u16 else torch.float32)
    return d.cpu().numpy()


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    r = fn()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, r


def end_to_end(rows, W, scans, pinned, reps):
    enc = encoder(rows, W)
    n = len(scans)
    offs = np.zeros(n + 1, np.int64)
    np.cumsum([len(s) for s in scans], out=offs[1:])
    point_bytes = int(offs[-1]) * 16
    dev_buf = torch.empty(pinned.shape, dtype=torch.float32, device="cuda")
    pinned_np = pinned.numpy()
    res = []
    for form, arg in (("pinned", (pinned_np, offs)), ("list", scans)):
        for u16 in (False, True):
            t = {"old": [], "new": [], "h2d": []}
            peak = {}
            for r in range(reps + 1):                              # the first round warms up
                for name in ("old", "new", "h2d"):
                    torch.cuda.reset_peak_memory_stats()
                    base = torch.cuda.memory_allocated()
                    if name == "old":
                        dt, out = timed(lambda: old_encode_scans(enc, arg, u16))
                        ref = out
                    elif name == "new":
                        dt, out = timed(lambda: enc.encode_scans(arg, dtype=np.uint16 if u16 else np.float32))
                        if not np.array_equal(out, ref):
                            raise SystemExit(f"{rows}x{W} {form} u16={u16}: old and new rows differ")
                    else:
                        dt, _ = timed(lambda: dev_buf.copy_(pinned, non_blocking=True))
                    peak[name] = torch.cuda.max_memory_allocated() - base
                    if r:
                        t[name].append(dt)
            med = {k: statistics.median(v) for k, v in t.items()}
            row = {"config": f"{rows}x{W}", "input": form, "rows": "uint16" if u16 else "float32", "scans": n,
                   "point_GB": round(point_bytes / 1e9, 3),
                   "old_ms": round(med["old"] * 1e3, 2), "new_ms": round(med["new"] * 1e3, 2),
                   "h2d_ms": round(med["h2d"] * 1e3, 2),
                   "new_share_of_h2d": round(med["h2d"] / med["new"], 3), "speedup": round(med["old"] / med["new"], 2),
                   "old_peak_torch_MB": round(peak["old"] / 2**20, 1), "new_peak_torch_MB": round(peak["new"] / 2**20, 1),
                   "old_min_ms": round(min(t["old"]) * 1e3, 2), "new_min_ms": round(min(t["new"]) * 1e3, 2)}
            res.append(row)
            print(json.dumps(row), flush=True)
    enc._close_pipeline()
    return res


def device_u16(n_scans, launches):
    lib = _lib.load()
    enc = encoder(16, 1024)
    p, lut = enc._params(), enc.freq_to_bin()
    pts, offs = synth.make_batch(synth.HDL64, 3000, n_scans, device="cuda")
    pts = pts.contiguous()
    D = enc.output_dim
    nbytes = int(lib.nsc_anywidth_workspace_bytes(n_scans, 16, C.byref(p)))
    ws = torch.empty((nbytes + 3) // 4, dtype=torch.int32, device="cuda")
    f32 = torch.empty((n_scans, D), device="cuda")
    q_two = torch.empty((n_scans, D), dtype=torch.int16, device="cuda")
    q_one = torch.empty((n_scans, D), dtype=torch.int16, device="cuda")
    s = torch.cuda.current_stream().cuda_stream

    def two():
        assert lib.nsc_anywidth_points(pts.data_ptr(), 4, offs.data_ptr(), 0, n_scans, C.byref(p), lut.ctypes.data,
                                       f32.data_ptr(), None, _lib.STAGE_INTERPOLATED, ws.data_ptr(), nbytes, s) == 0
        assert lib.nsc_quantize_histograms(f32.data_ptr(), n_scans, D, _lib.QUANT_EPSILON, q_two.data_ptr(), s) == 0

    def one():
        assert lib.nsc_anywidth_points_u16(pts.data_ptr(), 4, offs.data_ptr(), 0, n_scans, C.byref(p),
                                           lut.ctypes.data, _lib.QUANT_EPSILON, q_one.data_ptr(), ws.data_ptr(),
                                           nbytes, s) == 0
    t = {"two": [], "one": []}
    for i in range(launches + 2):
        for name, fn in (("two", two), ("one", one)):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            fn()
            b.record()
            torch.cuda.synchronize()
            if i >= 2:
                t[name].append(a.elapsed_time(b))
    if not torch.equal(q_one, q_two):
        raise SystemExit("device uint16: one launch and two launches differ")
    row = {"device_u16": "16x1024", "scans": n_scans, "two_launch_ms": round(statistics.median(t["two"]), 4),
           "one_launch_ms": round(statistics.median(t["one"]), 4),
           "speedup": round(statistics.median(t["two"]) / statistics.median(t["one"]), 3)}
    print(json.dumps(row), flush=True)
    return row


def per_scan(scans, reps):
    enc = encoder(16, 1024)

    def old(a):
        pts = torch.from_numpy(a).to("cuda")
        offs = torch.tensor([0, a.shape[0]], dtype=torch.int64).to("cuda")
        return enc.encode_points_batch(pts, offs)[0]
    t = {"old": [], "new": []}
    for r in range(reps + 1):
        for a in scans:
            dt_old, d_old = timed(lambda: old(a))
            dt_new, d_new = timed(lambda: enc.encode_points(a))
            if not torch.equal(d_old, d_new):
                raise SystemExit("encode_points: old and new differ")
            if r:
                t["old"].append(dt_old)
                t["new"].append(dt_new)
    row = {"per_scan": "16x1024", "calls": len(t["new"]), "old_us": round(statistics.median(t["old"]) * 1e6, 1),
           "new_us": round(statistics.median(t["new"]) * 1e6, 1),
           "speedup": round(statistics.median(t["old"]) / statistics.median(t["new"]), 2)}
    print(json.dumps(row), flush=True)
    enc._close_pipeline()
    return row


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scans", type=int, default=1024)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--device-scans", type=int, default=2048)
    ap.add_argument("--launches", type=int, default=30)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    print("gpu:", gpu_state(), flush=True)
    scans = host_scans(args.scans)
    pinned = torch.from_numpy(np.concatenate(scans)).pin_memory()
    for rows, W in ((16, 1024), (16, 2048), (64, 1024)):
        end_to_end(rows, W, scans, pinned, args.reps)
    device_u16(args.device_scans, args.launches)
    per_scan(scans[:50], args.reps)
    print("gpu:", gpu_state(), flush=True)


if __name__ == "__main__":
    main()
