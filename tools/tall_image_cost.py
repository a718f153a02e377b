#!/usr/bin/env python
"""What do images of more than 64 rows cost? A device-resident batch of BEAM128-shaped scans (128
beams x 2200 azimuth steps, far larger than the 126 MB L2) is encoded at n_elevation = 16, 64 and
128 (target_rows = 16), the row counts alternating launch by launch in one process, each timed
with CUDA events:

    E = 16    the warp-specialised kernel (TMA ring, two images per SM)
    E = 64    the generic kernel (cp.async ring, one image per SM)
    E = 128   the tall kernel (points straight into registers, one 128-row image per SM)

and, for every --variant NAME=PATH (a build of the library with another tall feed, e.g.
-DNSC_TALL_PTS=4), E = 128 through that build, whose rows must equal the product build's.
Bytes moved per launch: 16 per point plus 4 * D per descriptor; the share given is of the
6547.8 GB/s copy peak the project measures shares against (profiles/README.md). The GPU name and power limit
are read in the same run.

    python tools/tall_image_cost.py [--scans 2048] [--launches 30] [--variant tall4=path.so]
"""
import argparse
import ctypes as C
import json
import os
import statistics
import subprocess
import sys

import torch

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
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--variant", action="append", default=[], metavar="NAME=PATH")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    dev = torch.device("cuda")
    state0 = gpu_state()
    points, offsets = synth.make_batch_resident(synth.BEAM128, 0, a.scans, dev)
    n, n_points = a.scans, int(offsets[-1])
    stream = torch.cuda.current_stream(dev).cuda_stream
    libs = {"product": _lib.load()}
    for v in a.variant:
        name, path = v.split("=", 1)
        libs[name] = load_variant(path)
    runs = {}
    for rows in (16, 64, 128):
        enc = SpectralEncoder(n_elevation=rows, target_elevation_bins=16, elevation_range=(-25.0, 15.0)).to(dev)
        for lname in (libs if rows == 128 else ["product"]):
            runs[f"E{rows}_{lname}"] = (libs[lname], enc._params(), enc.freq_to_bin(), enc.output_dim)
    state = {}
    for k, (lib, p, lut, D) in runs.items():
        ws = torch.empty((int(lib.nsc_workspace_bytes(n, C.byref(p))) + 3) // 4, dtype=torch.int32, device=dev)
        out = torch.empty((n, D), dtype=torch.float32, device=dev)
        state[k] = (ws, out)

    def launch(k):
        lib, p, lut, D = runs[k]
        ws, out = state[k]
        _lib.check(lib.nsc_encode_batch(points.data_ptr(), 4, offsets.data_ptr(), 0, n, C.byref(p), lut.ctypes.data,
                                        out.data_ptr(), ws.data_ptr(), ws.numel() * 4, stream), k)

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
    same = {k: torch.equal(state[k][1], state["E128_product"][1]) for k in runs if k.startswith("E128_")}
    print(f"# {n} BEAM128 scans, {n_points} points ({16 * n_points / 1e9:.2f} GB), target_rows 16, "
          f"{a.launches} launches each, alternating")
    print(f"# gpu before: {state0}")
    print(f"# gpu after:  {state1}")
    rec = {"gpu": state0, "scans": n, "points": n_points, "launches": a.launches, "runs": {}}
    for k in runs:
        D = runs[k][3]
        s = sorted(times[k])
        med = statistics.median(s)
        nbytes = 16 * n_points + 4 * D * n
        r = {"median_ms": med, "p10_ms": s[len(s) // 10], "p90_ms": s[(9 * len(s)) // 10],
             "scans_per_s": n / (med * 1e-3), "GB_per_s": nbytes / (med * 1e-3) / 1e9,
             "share_of_copy_peak": nbytes / (med * 1e-3) / 1e9 / COPY_PEAK_GBS}
        if k in same:
            r["rows_equal_product"] = same[k]
        rec["runs"][k] = r
        print(f"{k:16s} median {med:8.3f} ms  p10 {r['p10_ms']:8.3f}  p90 {r['p90_ms']:8.3f}  "
              f"{r['scans_per_s']:10.0f} scans/s  {r['GB_per_s']:7.1f} GB/s  "
              f"{100 * r['share_of_copy_peak']:5.1f} % of copy peak" + (f"  rows equal: {same[k]}" if k in same else ""))
    print(json.dumps(rec))
    if not all(same.values()):
        raise SystemExit("a variant's rows differ from the product build's")


if __name__ == "__main__":
    main()
