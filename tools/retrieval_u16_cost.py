#!/usr/bin/env python
"""What does a uint16 retrieval database save? The bench.py --workload retrieval database (100 k x 800
rows from the same seeded generator: 320 MB of float32 CDF rows, 160 MB of uint16 ones, both larger
than the 126 MB L2), Q = 1 and Q = 8 queries, the variants alternating launch by launch in one
process:

    A   float32 database                 nsc_wasserstein_query
    A'  float32 database again           the spread of A against itself
    B   uint16 database of the           nsc_wasserstein_query_u16
        quantised rows

each as the distance pass alone (top_k = 0) and as the whole call (top-10, many-CTA selection).
Device time per call with CUDA events; a spin kernel ahead of each timed call keeps the host's launch
work out of the window. The GPU name, power limit and SM clocks are read in the same run.

Also reported, not gated on: the top-10 agreement between the float32 database of the original rows
and the uint16 database of their quantised rows (float32 queries), on that database and on encoder
descriptors of synth HDL-64 scans -- the cost of the wire format.

    python tools/retrieval_u16_cost.py [--db 100000] [--launches 50]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from neural_spectral_codec_b200 import SpectralEncoder, _lib, synth  # noqa: E402
from neural_spectral_codec_b200.retrieval import WassersteinRetriever  # noqa: E402


def gpu_state():
    q = "name,power.limit,clocks.sm,clocks.max.sm,temperature.gpu"
    r = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip() or r.stderr.strip()


def summary(ms):
    s = sorted(ms)
    return {"median_us": 1e3 * statistics.median(s), "min_us": 1e3 * s[0], "max_us": 1e3 * s[-1],
            "p10_us": 1e3 * s[len(s) // 10], "p90_us": 1e3 * s[(9 * len(s)) // 10], "n": len(s)}


def bench_workload(n_db, nq, dev):
    """bench.py run_retrieval's inputs: the same generator, seed and draws."""
    g = torch.Generator(device=dev).manual_seed(7)
    db = torch.rand((n_db, 800), generator=g, device=dev) ** 4
    db /= db.sum(1, keepdim=True)
    q = db[torch.randint(0, n_db, (nq,), device=dev)] * (1 + 0.05 * torch.rand((nq, 800), device=dev))
    return db, q


def agreement(f32, u16, queries, k=10):
    """Mean share of the float32 top-k found in the uint16 top-k, and the share of identical lists."""
    a = f32.query_batch(queries, top_k=k)[0].cpu()
    b = u16.query_batch(queries, top_k=k)[0].cpu()
    shared = [len(set(x.tolist()) & set(y.tolist())) / k for x, y in zip(a, b)]
    return {"queries": len(a), "top_k": k, "mean_overlap": sum(shared) / len(shared),
            "identical_lists": float((a == b).all(1).float().mean())}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--db", type=int, default=100000)
    ap.add_argument("--launches", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--scans", type=int, default=4096, help="encoder descriptors for the agreement figure")
    a = ap.parse_args()
    if a.launches < 30:
        raise SystemExit("--launches must be >= 30")
    dev = torch.device("cuda")
    lib = _lib.load()
    state0 = gpu_state()
    stream = torch.cuda.current_stream(dev).cuda_stream
    db, _ = bench_workload(a.db, 8, dev)
    f32 = WassersteinRetriever(device=dev)
    f32.add_to_database(db)
    u16 = WassersteinRetriever(device=dev, database_dtype=torch.uint16)
    u16.add_to_database(db)                                   # quantised on the device
    n = a.db
    ws = torch.zeros(int(lib.nsc_wasserstein_workspace_bytes(8)), dtype=torch.uint8, device=dev)

    def call(fn, cdfs, q, dist, k, idx, top, cnt):
        _lib.check(fn(q.data_ptr(), q.shape[0], cdfs.data_ptr(), n, 800, 1e-8, None, None, 0.0, dist.data_ptr(), k,
                      idx.data_ptr() if k else None, top.data_ptr() if k else None, cnt.data_ptr() if k else None,
                      ws.data_ptr(), ws.numel(), stream), "query")

    res = {"gpu_before": state0, "db_rows": n, "n_bins": 800,
           "db_bytes": {"float32_cdf": n * 800 * 4, "uint16_cdf": n * 800 * 2}, "launches_per_variant": a.launches,
           "timing": "device time per call: CUDA events, each call queued behind a spin kernel", "cases": {}}
    for nq in (1, 8):
        _, q = bench_workload(a.db, nq, dev)
        dist = torch.empty((nq, n), dtype=torch.float32, device=dev)
        idx = torch.empty((nq, 10), dtype=torch.int64, device=dev)
        top = torch.empty((nq, 10), dtype=torch.float32, device=dev)
        cnt = torch.empty((nq,), dtype=torch.int32, device=dev)
        outs = {}
        variants = {}
        for k, tag in ((0, "distances"), (10, "top10")):
            for name, fn, cdfs in (("A_f32", lib.nsc_wasserstein_query, f32._cdfs),
                                   ("A2_f32_again", lib.nsc_wasserstein_query, f32._cdfs),
                                   ("B_u16", lib.nsc_wasserstein_query_u16, u16._cdfs)):
                variants[f"{tag}_{name}"] = (lambda fn=fn, cdfs=cdfs, k=k: call(fn, cdfs, q, dist, k, idx, top, cnt))
        for fn in variants.values():
            for _ in range(a.warmup):
                fn()
        torch.cuda.synchronize()
        times = {v: [] for v in variants}
        ev = {v: (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for v in variants}
        for _ in range(a.launches):
            for v, fn in variants.items():
                torch.cuda._sleep(1_000_000)                 # the GPU is busy while the call is queued
                ev[v][0].record()
                fn()
                ev[v][1].record()
            torch.cuda.synchronize()
            for v in variants:
                times[v].append(ev[v][0].elapsed_time(ev[v][1]))
        # the distances of the two databases on these queries
        for name, fn, cdfs in (("f32", lib.nsc_wasserstein_query, f32._cdfs),
                               ("u16", lib.nsc_wasserstein_query_u16, u16._cdfs)):
            call(fn, cdfs, q, dist, 0, idx, top, cnt)
            outs[name] = dist.clone()
        torch.cuda.synchronize()
        d = (outs["u16"] - outs["f32"]).abs()
        case = {v: summary(t) for v, t in times.items()}
        med = {v: s["median_us"] for v, s in case.items()}
        for tag in ("distances", "top10"):
            case[f"{tag}_B_minus_A_us"] = med[f"{tag}_B_u16"] - med[f"{tag}_A_f32"]
            case[f"{tag}_A_spread_us"] = abs(med[f"{tag}_A_f32"] - med[f"{tag}_A2_f32_again"])
        case["distance_pass_f32_TBps"] = n * 800 * 4 / (med["distances_A_f32"] * 1e-6) / 1e12
        case["distance_pass_u16_TBps"] = n * 800 * 2 / (med["distances_B_u16"] * 1e-6) / 1e12
        case["max_abs_distance_difference_u16_vs_f32"] = float(d.max())
        case["distance_range"] = [float(outs["f32"].min()), float(outs["f32"].max())]
        res["cases"][f"Q{nq}"] = case
    res["gpu_after"] = gpu_state()

    # what the wire format costs in neighbours: float32 queries, float32 rows against their quantised rows
    _, qa = bench_workload(a.db, 64, dev)
    res["agreement_bench_db"] = agreement(f32, u16, qa)
    enc = SpectralEncoder(n_elevation=16, target_elevation_bins=16).to(dev)
    pts, offs = synth.make_batch_resident(synth.HDL64, 0, a.scans, dev)
    desc = enc.encode_points_batch(pts, offs)
    desc16 = enc.encode_points_batch(pts, offs, dtype=torch.uint16)     # == quantize(desc)
    del pts, offs
    qpts, qoffs = synth.make_batch_resident(synth.HDL64, 50000, 256, dev)
    qdesc = enc.encode_points_batch(qpts, qoffs)
    ef, eu = WassersteinRetriever(device=dev), WassersteinRetriever(device=dev, database_dtype=torch.uint16)
    ef.add_to_database(desc)
    eu.add_to_database(desc16)
    res["agreement_synth_descriptors"] = {"db_scans": a.scans, **agreement(ef, eu, qdesc)}

    print(f"GPU: {state0}  (after: {res['gpu_after']})")
    print(f"{n} x 800 database: float32 CDF rows {n * 800 * 4 / 1e6:.0f} MB, uint16 {n * 800 * 2 / 1e6:.0f} MB; "
          f"{a.launches} launches per variant, alternating; device time per call")
    for cname, case in res["cases"].items():
        print(f"{cname}:")
        for v, s in case.items():
            if isinstance(s, dict):
                print(f"  {v:24s} median {s['median_us']:8.2f} us  p10 {s['p10_us']:8.2f}  p90 {s['p90_us']:8.2f}  "
                      f"min {s['min_us']:8.2f}  max {s['max_us']:8.2f}")
        for tag in ("distances", "top10"):
            print(f"  {tag}: B - A = {case[f'{tag}_B_minus_A_us']:+.2f} us   |A - A'| = {case[f'{tag}_A_spread_us']:.2f} us")
        print(f"  distance pass: float32 {case['distance_pass_f32_TBps']:.2f} TB/s, uint16 "
              f"{case['distance_pass_u16_TBps']:.2f} TB/s of CDF rows; max |d_u16 - d_f32| = "
              f"{case['max_abs_distance_difference_u16_vs_f32']:.3g} on distances in "
              f"[{case['distance_range'][0]:.3g}, {case['distance_range'][1]:.3g}]")
    for key in ("agreement_bench_db", "agreement_synth_descriptors"):
        g = res[key]
        print(f"top-10 agreement, float32 rows vs their uint16 rows ({key[10:]}): mean overlap "
              f"{g['mean_overlap']:.4f}, identical lists {g['identical_lists']:.4f} over {g['queries']} queries")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
