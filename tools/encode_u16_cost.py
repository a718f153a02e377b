#!/usr/bin/env python
"""What does the uint16 epilogue of the encode kernels cost? The bench.py default workload (4541
HDL-64-shaped scans resident in HBM, 8.7 GB, far larger than the 126 MB L2), timed per launch with
CUDA events, the variants alternating launch by launch in one process:

    A   nsc_encode_batch                                  float32 rows
    A'  nsc_encode_batch again                            the spread of A against itself
    B   nsc_encode_batch_u16                              uint16 rows from the epilogue
    C   nsc_encode_batch + nsc_quantize_histograms        the two-pass route it replaces

and end to end, host scans in / host rows out through encode_scans (pinned buffers), float32
against uint16. After timing, B's output must equal quantize(A's output) and C's output. The GPU
name, power limit and SM clocks are read in the same run.

    python tools/encode_u16_cost.py [--scans 4541] [--launches 30] [--e2e-scans 1024] [--e2e-reps 5]
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


def summary(ms):
    s = sorted(ms)
    return {"median_ms": statistics.median(s), "min_ms": s[0], "max_ms": s[-1],
            "p10_ms": s[len(s) // 10], "p90_ms": s[(9 * len(s)) // 10], "n": len(s)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scans", type=int, default=4541)
    ap.add_argument("--launches", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--e2e-scans", type=int, default=1024)
    ap.add_argument("--e2e-reps", type=int, default=5)
    a = ap.parse_args()
    if a.launches < 20:
        raise SystemExit("--launches must be >= 20")
    dev = torch.device("cuda")
    lib = _lib.load()
    state0 = gpu_state()
    enc = SpectralEncoder(n_elevation=16, target_elevation_bins=16).to(dev)
    points, offsets = synth.make_batch_resident(synth.HDL64, 0, a.scans, dev)
    n, D = a.scans, enc.output_dim
    p, lut = enc._params(), enc.freq_to_bin()
    stream = torch.cuda.current_stream(dev).cuda_stream
    ws = torch.empty((int(lib.nsc_workspace_bytes(n, C.byref(p))) + 3) // 4, dtype=torch.int32, device=dev)
    out_a = torch.empty((n, D), dtype=torch.float32, device=dev)
    out_a2 = torch.empty_like(out_a)
    out_b = torch.empty((n, D), dtype=torch.uint16, device=dev)
    out_c = torch.empty_like(out_b)
    eps = _lib.QUANT_EPSILON

    def enc_f32(out):
        _lib.check(lib.nsc_encode_batch(points.data_ptr(), 4, offsets.data_ptr(), 0, n, C.byref(p), lut.ctypes.data,
                                        out.data_ptr(), ws.data_ptr(), ws.numel() * 4, stream), "nsc_encode_batch")

    def enc_u16():
        _lib.check(lib.nsc_encode_batch_u16(points.data_ptr(), 4, offsets.data_ptr(), 0, n, C.byref(p),
                                            lut.ctypes.data, eps, out_b.data_ptr(), ws.data_ptr(), ws.numel() * 4,
                                            stream), "nsc_encode_batch_u16")

    def two_pass():
        enc_f32(out_a2)
        _lib.check(lib.nsc_quantize_histograms(out_a2.data_ptr(), n, D, eps, out_c.data_ptr(), stream),
                   "nsc_quantize_histograms")

    variants = {"A_encode_f32": lambda: enc_f32(out_a), "A2_encode_f32_again": lambda: enc_f32(out_a2),
                "B_encode_u16": enc_u16, "C_encode_f32_then_quantize": two_pass}
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

    # the timed outputs: B is quantize(A) and the two-pass route's result, every row
    with torch.cuda.device(dev):
        want = torch.empty_like(out_b)
        _lib.check(lib.nsc_quantize_histograms(out_a.data_ptr(), n, D, eps, want.data_ptr(), stream), "quantize")
    torch.cuda.synchronize()
    same_q = torch.equal(out_b.view(torch.int16), want.view(torch.int16))
    same_c = torch.equal(out_b.view(torch.int16), out_c.view(torch.int16))
    sums = out_b.view(torch.int16).to(torch.int32).bitwise_and(0xffff).sum(1)
    rows_65535 = int((sums == 65535).sum())

    # end to end: host scans in, host rows out
    m = min(a.e2e_scans, n)
    host_pts = points[: int(offsets[m])].cpu().pin_memory()
    host_offs = offsets[: m + 1].cpu().numpy()
    f_out = torch.empty((m, D), dtype=torch.float32).pin_memory().numpy()
    q_out = torch.empty((m, D), dtype=torch.uint16).pin_memory().numpy()
    e2e = {"float32": [], "uint16": []}
    for rep in range(a.e2e_reps + 1):
        for k, out, dt in (("float32", f_out, np.float32), ("uint16", q_out, np.uint16)):
            t0 = time.perf_counter()
            enc.encode_scans((host_pts.numpy(), host_offs), out=out, dtype=dt)
            t1 = time.perf_counter()
            if rep:                                    # the first round warms the pipeline up
                e2e[k].append((t1 - t0) * 1e3)
    e2e_same = bool(np.array_equal(q_out, want[:m].cpu().numpy()))

    res = {"gpu_before": state0, "gpu_after": state1, "scans": n, "descriptor": D,
           "input_gb": round(points.numel() * 4 / 1e9, 2), "launches_per_variant": a.launches,
           "kernel": {k: summary(v) for k, v in times.items()},
           "checks": {"u16_equals_quantize_of_f32_timed_outputs": same_q, "u16_equals_two_pass": same_c,
                      "rows_summing_to_65535": f"{rows_65535}/{n}"},
           "end_to_end": {"scans": m, "input_gb": round(host_pts.numel() * 4 / 1e9, 2),
                          **{k: summary(v) for k, v in e2e.items()}, "u16_equals_quantize": e2e_same}}
    med = {k: v["median_ms"] for k, v in res["kernel"].items()}
    a_spread = abs(med["A_encode_f32"] - med["A2_encode_f32_again"])
    print(f"GPU: {state0}  (after: {state1})")
    print(f"{n} scans, {res['input_gb']} GB of points, {a.launches} launches per variant, alternating")
    for k, v in res["kernel"].items():
        print(f"  {k:28s} median {v['median_ms']:.4f} ms  p10 {v['p10_ms']:.4f}  p90 {v['p90_ms']:.4f}  "
              f"min {v['min_ms']:.4f}  max {v['max_ms']:.4f}")
    print(f"  B - A  = {med['B_encode_u16'] - med['A_encode_f32']:+.4f} ms   |A - A'| = {a_spread:.4f} ms   "
          f"C - B = {med['C_encode_f32_then_quantize'] - med['B_encode_u16']:+.4f} ms")
    print(f"  B == quantize(A) on the timed outputs: {same_q};  B == C: {same_c};  rows summing to 65535: "
          f"{rows_65535}/{n}")
    ee = res["end_to_end"]
    print(f"end to end, encode_scans of {m} scans ({ee['input_gb']} GB pinned): float32 median "
          f"{ee['float32']['median_ms']:.2f} ms, uint16 median {ee['uint16']['median_ms']:.2f} ms "
          f"(min {ee['float32']['min_ms']:.2f} / {ee['uint16']['min_ms']:.2f}); uint16 == quantize: {e2e_same}")
    print(json.dumps(res))
    if not (same_q and same_c and e2e_same):
        raise SystemExit("uint16 rows differ from the quantised float32 rows")


if __name__ == "__main__":
    main()
