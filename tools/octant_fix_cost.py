#!/usr/bin/env python
"""What does the scale-invariant octant reduction of the column (nsc_point.h: min and max scaled by
2^32 before the reciprocal) cost the encode kernels? Two library builds in one process, the base
(given by path, e.g. one built from the parent commit) and the product library, on the bench.py
default workload (4541 HDL-64-shaped scans resident in HBM), timed per launch with CUDA events and
alternating launch by launch:

    stride 4   the warp-specialised kernel (what bench.py times)
    stride 3   the same points as (N, 3): the generic kernel, which bench.py has no option for

For each stride the product library runs twice per round (A and A'), so |A - A'| shows the spread.
After timing, both libraries' descriptors must be equal bit for bit (no point of this workload is
near the vertical axis). The GPU name, power limit and SM clocks are read in the same run.

    python tools/octant_fix_cost.py --base neural_spectral_codec_b200/libnsc_b200_parent.so [--launches 30]
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


def gpu_state():
    q = "name,power.limit,clocks.sm,clocks.max.sm,temperature.gpu"
    r = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip() or r.stderr.strip()


def load_as(path):
    lib = C.CDLL(os.path.abspath(path))
    for name, (res, args) in _lib.SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype = res
        fn.argtypes = args
    return lib


def summary(ms):
    s = sorted(ms)
    return {"median_ms": statistics.median(s), "min_ms": s[0], "max_ms": s[-1],
            "p10_ms": s[len(s) // 10], "p90_ms": s[(9 * len(s)) // 10], "n": len(s)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--base", required=True, help="path of the library to compare against")
    ap.add_argument("--scans", type=int, default=4541)
    ap.add_argument("--launches", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    a = ap.parse_args()
    if a.launches < 20:
        raise SystemExit("--launches must be >= 20")
    dev = torch.device("cuda")
    libs = {"base": load_as(a.base), "fixed": _lib.load()}
    state0 = gpu_state()
    enc = SpectralEncoder(n_elevation=16, target_elevation_bins=16).to(dev)
    p4, offsets = synth.make_batch_resident(synth.HDL64, 0, a.scans, dev)
    p3 = p4[:, :3].contiguous()
    n, D = a.scans, enc.output_dim
    p, lut = enc._params(), enc.freq_to_bin()
    stream = torch.cuda.current_stream(dev).cuda_stream
    ws = torch.empty((int(libs["fixed"].nsc_workspace_bytes(n, C.byref(p))) + 3) // 4, dtype=torch.int32,
                     device=dev)
    outs = {}

    def launcher(lib_name, stride, tag):
        lib, pts = libs[lib_name], (p4 if stride == 4 else p3)
        out = outs.setdefault(tag, torch.empty((n, D), dtype=torch.float32, device=dev))

        def run():
            _lib.check(lib.nsc_encode_batch(pts.data_ptr(), stride, offsets.data_ptr(), 0, n, C.byref(p),
                                            lut.ctypes.data, out.data_ptr(), ws.data_ptr(), ws.numel() * 4,
                                            stream), "nsc_encode_batch")
        return run

    variants = {}
    for stride in (4, 3):
        variants[f"s{stride}_base"] = launcher("base", stride, f"s{stride}_base")
        variants[f"s{stride}_fixed"] = launcher("fixed", stride, f"s{stride}_fixed")
        variants[f"s{stride}_fixed_again"] = launcher("fixed", stride, f"s{stride}_fixed_again")
    for fn in variants.values():
        for _ in range(a.warmup):
            fn()
    torch.cuda.synchronize()
    times = {k: [] for k in variants}
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in variants]
    for _ in range(a.launches):
        for (k, fn), (e0, e1) in zip(variants.items(), ev):
            e0.record()
            fn()
            e1.record()
        torch.cuda.synchronize()
        for k, (e0, e1) in zip(variants, ev):
            times[k].append(e0.elapsed_time(e1))
    state1 = gpu_state()
    same = {f"s{s}": torch.equal(outs[f"s{s}_base"].view(torch.int32), outs[f"s{s}_fixed"].view(torch.int32))
            for s in (4, 3)}
    res = {"gpu_before": state0, "gpu_after": state1, "scans": n, "input_gb": round(p4.numel() * 4 / 1e9, 2),
           "launches_per_variant": a.launches, "kernel": {k: summary(v) for k, v in times.items()},
           "descriptors_equal_to_base": same}
    med = {k: v["median_ms"] for k, v in res["kernel"].items()}
    print(f"GPU: {state0}  (after: {state1})")
    print(f"{n} scans, {res['input_gb']} GB of points, {a.launches} launches per variant, alternating")
    for k, v in res["kernel"].items():
        print(f"  {k:18s} median {v['median_ms']:.4f} ms  p10 {v['p10_ms']:.4f}  p90 {v['p90_ms']:.4f}  "
              f"min {v['min_ms']:.4f}  max {v['max_ms']:.4f}")
    for s in (4, 3):
        d = med[f"s{s}_fixed"] - med[f"s{s}_base"]
        spread = abs(med[f"s{s}_fixed"] - med[f"s{s}_fixed_again"])
        print(f"  stride {s}: fixed - base = {d:+.4f} ms ({100 * d / med[f's{s}_base']:+.2f} %)   "
              f"|A - A'| = {spread:.4f} ms   descriptors equal: {same[f's{s}']}")
    print(json.dumps(res))
    if not all(same.values()):
        raise SystemExit("descriptors differ from the base library's")


if __name__ == "__main__":
    main()
