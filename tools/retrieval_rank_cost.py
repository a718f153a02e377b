#!/usr/bin/env python
"""What does ranking the whole database cost? ``query_batch(top_k=n_db)`` -- the reference's
_global_retrieval asks for every keyframe -- on the device radix sort (nsc_wasserstein_rank) against
the torch path it replaced, which this script re-implements: the distance pass alone, then
torch.sort(stable=True), isfinite().sum(), clamp and two masked fills.

Databases of n_db in {4541, 100 000, 1 000 000} rows x 800 bins from bench.py's retrieval generator,
float32 and uint16, Q = 1 and Q = 8 queries. Variants, alternating call by call in one process:

    distances   nsc_wasserstein_query with top_k = 0 (the distance pass both paths share)
    rank        query_batch(top_k=n_db) (this library)
    torch       the replaced torch path
    rank_alt    (with --alt-lib) nsc_wasserstein_rank of another build of the library, e.g. the
                11-bit digit build (make VARIANT=rank11 DEFS=-DNSC_RANK_BITS=11)

Two timings per variant, CUDA events, median of --launches after --warmup calls: "queued" (each
call queued behind a spin kernel: device time without the host's launch gaps) and "direct" (after
a synchronise: what a caller waits for). The outputs of rank and torch are compared bit for bit. The
GPU name, power limit and SM clocks are read in the same run.

    python tools/retrieval_rank_cost.py [--alt-lib PATH] [--launches 30]
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
from neural_spectral_codec_b200 import _lib  # noqa: E402
from neural_spectral_codec_b200.retrieval import WassersteinRetriever  # noqa: E402


def gpu_state():
    q = "name,power.limit,clocks.sm,clocks.max.sm,temperature.gpu"
    r = subprocess.run(["nvidia-smi", "-i", "0", f"--query-gpu={q}", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return r.stdout.strip() or r.stderr.strip()


def bench_workload(n_db, nq, dev):
    """bench.py run_retrieval's inputs: the same generator, seed and draws."""
    g = torch.Generator(device=dev).manual_seed(7)
    db = torch.rand((n_db, 800), generator=g, device=dev) ** 4
    db /= db.sum(1, keepdim=True)
    q = db[torch.randint(0, n_db, (nq,), device=dev)] * (1 + 0.05 * torch.rand((nq, 800), device=dev))
    return db, q


def distances(lib, r, q):
    """The distance pass alone (top_k = 0), as both paths run it."""
    n, nq = r.database_size, q.shape[0]
    dist = torch.empty((nq, n), dtype=torch.float32, device=q.device)
    name = "nsc_wasserstein_query_u16" if r.database_dtype == torch.uint16 else "nsc_wasserstein_query"
    _lib.check(getattr(lib, name)(q.data_ptr(), nq, r._cdfs.data_ptr(), n, 800, r.epsilon, None, None, 0.0,
                                  dist.data_ptr(), 0, None, None, None, None, 0,
                                  torch.cuda.current_stream().cuda_stream), name)
    return dist


def torch_path(lib, r, q, k):
    """The replaced query_batch branch for k > 1024, with its allocations."""
    nq = q.shape[0]
    idx = torch.empty((nq, k), dtype=torch.int64, device=q.device)
    top = torch.empty((nq, k), dtype=torch.float32, device=q.device)
    cnt = torch.zeros((nq,), dtype=torch.int32, device=q.device)
    del idx, top, cnt
    dist = distances(lib, r, q)
    sd, si = torch.sort(dist, dim=1, stable=True)
    top, idx = sd[:, :k].contiguous(), si[:, :k].contiguous()
    cnt = torch.isfinite(dist).sum(1).clamp(max=k).to(torch.int32)
    beyond = torch.arange(k, device=q.device).unsqueeze(0) >= cnt.unsqueeze(1)
    idx[beyond] = -1
    top[beyond] = float("inf")
    return idx, top, cnt, dist


def rank_call(lib, r, q, k, ws):
    """nsc_wasserstein_rank[_u16] of `lib` straight through ctypes."""
    n, nq = r.database_size, q.shape[0]
    dist = torch.empty((nq, n), dtype=torch.float32, device=q.device)
    idx = torch.empty((nq, k), dtype=torch.int64, device=q.device)
    top = torch.empty((nq, k), dtype=torch.float32, device=q.device)
    cnt = torch.empty((nq,), dtype=torch.int32, device=q.device)
    name = "nsc_wasserstein_rank_u16" if r.database_dtype == torch.uint16 else "nsc_wasserstein_rank"
    _lib.check(getattr(lib, name)(q.data_ptr(), nq, r._cdfs.data_ptr(), n, 800, r.epsilon, None, None, 0.0,
                                  dist.data_ptr(), k, idx.data_ptr(), top.data_ptr(), cnt.data_ptr(),
                                  ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream), name)
    return idx, top, cnt, dist


def load_alt(path):
    lib = C.CDLL(path)
    for name, (res, args) in _lib.SYMBOLS.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    return lib


def median_us(ms):
    return 1e3 * statistics.median(ms)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--db", type=int, nargs="+", default=[4541, 100000, 1000000])
    ap.add_argument("--queries", type=int, nargs="+", default=[1, 8])
    ap.add_argument("--launches", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--alt-lib", help="another build of libnsc_b200.so whose nsc_wasserstein_rank is timed too")
    a = ap.parse_args()
    dev = torch.device("cuda")
    lib = _lib.load()
    alt = load_alt(a.alt_lib) if a.alt_lib else None
    res = {"gpu_before": gpu_state(), "launches": a.launches, "warmup": a.warmup, "alt_lib": a.alt_lib,
           "timing": "median device time per call, CUDA events; queued = behind a spin kernel, direct = after a "
                     "synchronise", "points": []}
    for n_db in a.db:
        db, _ = bench_workload(n_db, 8, dev)
        for dtype in (torch.float32, torch.uint16):
            r = WassersteinRetriever(device=dev, database_dtype=dtype)
            r.add_to_database(db)
            for nq in a.queries:
                _, q = bench_workload(n_db, nq, dev)
                need = max(int(x.nsc_wasserstein_rank_workspace_bytes(nq, n_db)) for x in (lib, alt) if x is not None)
                ws = torch.empty(need, dtype=torch.uint8, device=dev)      # the 11-bit build needs more
                variants = {"distances": lambda: distances(lib, r, q),
                            "rank": lambda: r.query_batch(q, top_k=n_db, return_distances=True),
                            "torch": lambda: torch_path(lib, r, q, n_db)}
                if alt is not None:
                    variants["rank_direct"] = lambda: rank_call(lib, r, q, n_db, ws)
                    variants["rank_alt"] = lambda: rank_call(alt, r, q, n_db, ws)
                for fn in variants.values():
                    for _ in range(a.warmup):
                        fn()
                torch.cuda.synchronize()
                times = {(v, m): [] for v in variants for m in ("queued", "direct")}
                for _ in range(a.launches):
                    for mode in ("queued", "direct"):
                        for v, fn in variants.items():
                            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                            torch.cuda.synchronize()
                            if mode == "queued":
                                torch.cuda._sleep(2_000_000)
                            e0.record()
                            fn()
                            e1.record()
                            e1.synchronize()
                            times[(v, mode)].append(e0.elapsed_time(e1))
                new, old = variants["rank"](), variants["torch"]()
                identical = all(torch.equal(x.view(torch.int32) if x.dtype == torch.float32 else x,
                                            y.view(torch.int32) if y.dtype == torch.float32 else y)
                                for x, y in zip(new, old))
                if alt is not None:
                    identical = identical and all(torch.equal(x, y) for x, y in zip(
                        rank_call(lib, r, q, n_db, ws), rank_call(alt, r, q, n_db, ws)))
                point = {"n_db": n_db, "dtype": str(dtype).replace("torch.", ""), "queries": nq,
                         "outputs_bit_identical": identical,
                         **{f"{v}_{m}_us": median_us(t) for (v, m), t in times.items()}}
                for m in ("queued", "direct"):
                    point[f"rank_over_torch_{m}"] = point[f"rank_{m}_us"] / point[f"torch_{m}_us"]
                    point[f"sort_{m}_us"] = point[f"rank_{m}_us"] - point[f"distances_{m}_us"]
                res["points"].append(point)
                print(f"n_db {n_db:8d} {point['dtype']:8s} Q {nq}: " + "  ".join(
                    f"{v} {point[f'{v}_queued_us']:9.1f}/{point[f'{v}_direct_us']:9.1f}" for v in variants) +
                    f"  us (queued/direct); rank/torch {point['rank_over_torch_queued']:.3f}/"
                    f"{point['rank_over_torch_direct']:.3f}; identical {identical}", flush=True)
            del r
        del db
        torch.cuda.empty_cache()
    res["gpu_after"] = gpu_state()
    print(f"GPU: {res['gpu_before']}  (after: {res['gpu_after']})")
    print(json.dumps(res))


if __name__ == "__main__":
    main()
