#!/usr/bin/env python
"""Benchmark of the spectral encoding front end (BASELINE.json metric: scans/s encoded to 800-D).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

A step = one pass of the fused encode kernel over this rank's batch of synthetic scans
(BASELINE.json configs[1]: 4541 HDL-64-shaped scans of ~120 k xyzi points, 8.7 GB, resident in
HBM before timing), followed for N > 1 by the gather of the 800-D descriptors into the database
replicated on every GPU. Weak scaling: every rank holds its own 4541 scans.

Prints ONE JSON line (rank 0):
  value         device-timed whole-job throughput (CUDA events, max over ranks)
  roofline      the fused kernel against the measured HBM peak (events around each launch)
  e2e           the same metric through ``SpectralEncoder.encode_scans`` with pinned HOST buffers
                (H2D + kernel + D2H inside the timed region), with the bare pinned-H2D rate of
                the same bytes beside it (``h2d_ceiling_gbs_per_gpu``), the reference's own call
                pattern (``per_scan``: one ``encode_points(numpy)`` per scan) and pageable lists
  checks        made AFTER the timed region on the timed output: rows of ``out`` against the CPU
                oracle, and for N > 1 the gathered database against an NCCL all-gather of the
                single-GPU encodes, on every rank. A failed check exits non-zero.
  configs       the other BASELINE.json shapes (HDL-32, 128-beam, shuffled order) at reduced step
                counts, each with its own roofline fraction and CPU baseline   (N = 1)
  c5            BASELINE.json configs[4]: 100 000 scans sharded over the ranks        (N > 1)
  cpu_baseline  the reference's CPU encoder on all host cores (``kind: "reference"`` when the
                git-ignored copy made by oracle/make_ref.py is present, else the oracle port)

``--impl reference`` times that same CPU encoder as the reference arm, honouring --steps/--warmup.

``--dump-outputs DIR`` writes, after the timed steps, what the timed path returned in its last step
as ``DIR/<name>.npy`` (float32 / float64; integer outputs converted exactly), so that two builds can
be compared output for output: the inputs depend on the arguments only (seeded). Outputs above
64 MB in all are cut to a fixed, seeded sample of rows, listed in ``DIR/rows.npy``.

Secondary lines (not the BASELINE.json metric, same JSON shape): ``--workload retrieval`` (stage-1
Wasserstein top-K over a 100 k x 800 database), ``--workload keyframe`` (voxel IoU of the keyframe
gate), ``--workload quantize`` (uint16 wire format).
"""
import argparse
import json
import multiprocessing as mp
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "scans_per_sec_encoded_to_800d"
UNIT = "scans/s"
N_SCANS = 4541            # KITTI sequence 00 length (BASELINE.json configs[1])
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md, used only without MEASURED_PEAKS.json
ENCODER_DESC = "n_elevation=16 n_azimuth=360 n_bins=50 alpha=2.0 target_rows=16"

SHAPE_DESC = {"hdl64": "HDL-64-shaped scans x ~120k xyzi points", "hdl32": "NCLT HDL-32-shaped scans x ~70k xyzi points",
              "beam128": "128-beam dense scans x ~260k xyzi points"}
SHAPE_GB = {"hdl64": 1.93e-3, "hdl32": 1.13e-3, "beam128": 4.15e-3}   # GB per scan, for the config text


def workload_name(n, shape="hdl64", shuffle=False):
    head = "synthetic KITTI seq-00-length batch" if shape == "hdl64" else "synthetic batch"
    return f"{head}: {n} {SHAPE_DESC[shape]} per GPU" + (" (shuffled point order)" if shuffle else "")


def make_config(args, world):
    """The ``config`` object; identical for the GPU arm and the reference arm of one invocation."""
    return {"workload": workload_name(args.scans, args.shape, args.shuffle), "scans_per_gpu": args.scans,
            "l2": f"inputs (~{args.scans * SHAPE_GB[args.shape]:.1f} GB per GPU) larger than the 126 MB L2, no flush needed",
            "gather": ("none (single GPU)" if world == 1 else gather_name(args)), "encoder": ENCODER_DESC}


def gather_name(args):
    if args.gather == "fused" and args.gather_lag:
        return "fused, pipelined (the database of step s-1 is complete when step s is enqueued; all complete before the timed region ends)"
    return args.gather


# ----------------------------------------------------------------------------- CPU arm
def reference_src():
    """sys.path entry of the unmodified reference (oracle/make_ref.py), or None."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    try:
        import make_ref
        return make_ref.ref_src_path()
    except Exception:
        return None
    finally:
        sys.path.pop(0)


def make_cpu_encoder(kind):
    """``encode(points np (N,4)) -> descriptor`` of the reference's CPU path.
    kind "reference": the reference's own SpectralEncoder, constructed as its callers do
    (train_multi_dataset.py:264-271); kind "port": oracle/nsc_oracle.py."""
    if kind == "reference":
        src = reference_src()
        if src not in sys.path:
            sys.path.insert(0, src)
        from encoding.spectral_encoder import SpectralEncoder as RefEncoder
        enc = RefEncoder(n_elevation=16, n_azimuth=360, n_bins=50, alpha=2.0, learnable_alpha=True,
                         target_elevation_bins=16)
        return lambda pts: enc.encode_points(pts).detach().cpu().numpy()
    from oracle import nsc_oracle as orc
    cfg = orc.OracleConfig()
    return lambda pts: orc.encode_points(pts, cfg).numpy()


def _cpu_worker(job):
    """Encode ``count`` scans starting at seed ``first``; returns (count, seconds)."""
    first, count, shape, shuffle, kind = job
    import torch
    torch.set_num_threads(1)
    from neural_spectral_codec_b200 import synth
    encode = make_cpu_encoder(kind)
    scans = [synth.make_scan(synth.SHAPES[shape], first + i, shuffle=shuffle).numpy() for i in range(count)]
    t0 = time.perf_counter()
    for s in scans:
        encode(s)
    return count, time.perf_counter() - t0


def cpu_throughput(pool, scans_per_core, cores, kind, shape="hdl64", shuffle=False, first=100000):
    """All-cores throughput: each worker generates its own scans from seeds (not timed) and encodes
    them single-threaded; throughput = sum over workers of count / time."""
    jobs = [(first + w * scans_per_core, scans_per_core, shape, shuffle, kind) for w in range(cores)]
    res = pool.map(_cpu_worker, jobs, chunksize=1)
    return sum(c / t for c, t in res), sum(c for c, _ in res)


def cpu_kind():
    return "reference" if reference_src() else "port"


def cpu_kind_text(kind):
    return ("the reference's own SpectralEncoder.encode_points (verbatim copy of its Python files, oracle/make_ref.py)"
            if kind == "reference" else "oracle/nsc_oracle.py (port of the reference's Python encoder)")


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = int(os.environ.get("WORLD_SIZE", str(args.gpus)))
    cores = os.cpu_count() or 1
    kind = cpu_kind()
    # bounded sample per step: the whole --steps/--warmup run stays within ~2 minutes
    per_core = int(max(2, min(16, 120.0 / max(1, args.steps + args.warmup) / 0.03)))
    vals, ms = [], []
    with mp.get_context("spawn").Pool(cores) as pool:
        for _ in range(args.warmup):
            cpu_throughput(pool, per_core, cores, kind, args.shape, args.shuffle)
        for _ in range(args.steps):
            t0 = time.perf_counter()
            v, _n = cpu_throughput(pool, per_core, cores, kind, args.shape, args.shuffle)
            ms.append(1e3 * (time.perf_counter() - t0))
            vals.append(v)
    value = statistics.median(vals)
    sample = (f"{per_core} scans per core x {cores} cores per step; {cpu_kind_text(kind)}, one single-threaded "
              "process per core; scan generation is outside the timed part")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": statistics.median(ms), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": make_config(args, max(world, args.gpus)),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    emit(line)


# ----------------------------------------------------------------------------- clocks
class ClockSampler(threading.Thread):
    """Polls NVML for SM clock and throttle reasons while the timed region runs."""

    def __init__(self, index: int, period: float = 0.005):
        super().__init__(daemon=True)
        self.index, self.period = index, period
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop_evt = threading.Event()
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        names = {
            getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8): "hw_slowdown",
            getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40): "hw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20): "sw_thermal_slowdown",
            getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4): "sw_power_cap",
            getattr(nv, "nvmlClocksEventReasonHwPowerBrakeSlowdown", 0x80): "hw_power_brake",
        }
        while not self._stop_evt.is_set():
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in names.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(self.period)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=2)
        return {"sm_mhz": statistics.median(self.samples) if self.samples else None,
                "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ----------------------------------------------------------------------------- GPU arm helpers
def hbm_peak():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        return float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md)"


def time_encode(enc, points, offsets, out, steps, warmup):
    """CUDA-event time of ``steps`` launches of the fused kernel, each bracketed on the launching
    stream; returns (mean ms per launch, total ms first-to-last)."""
    import torch
    dev = points.device
    for _ in range(warmup):
        enc.encode_points_batch(points, offsets, out=out)
    torch.cuda.synchronize(dev)
    stream = torch.cuda.current_stream(dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * steps)]
    for k in range(steps):
        ev[2 * k].record(stream)
        enc.encode_points_batch(points, offsets, out=out)
        ev[2 * k + 1].record(stream)
    torch.cuda.synchronize(dev)
    ms = [ev[2 * k].elapsed_time(ev[2 * k + 1]) for k in range(steps)]
    return sum(ms) / len(ms), ev[0].elapsed_time(ev[-1])


def oracle_spot_check(enc, points, offsets_host, rows, scan_ids):
    """Rows of a timed output against the CPU oracle (the checker; never timed).

    For every scan id: (1) ``rows[i]`` vs the oracle on the same cloud -- max |diff| must stay
    below 1e-4 (points within 1e-5 rad of a pixel edge may land one pixel over, north star);
    (2) the cloud stripped of those edge points, encoded on the GPU, vs the oracle on the
    stripped cloud at the test-suite tolerances (rtol 1e-4 / atol 1e-7, relative L2 1e-5);
    (3) ``rows[i]`` bit-identical to a single-scan encode of the same cloud."""
    import numpy as np
    from oracle import nsc_oracle as orc
    cfg = orc.OracleConfig()
    max_abs, max_l2, ok, same_bits = 0.0, 0.0, True, True
    for i in scan_ids:
        s = points[int(offsets_host[i]):int(offsets_host[i + 1])].cpu().numpy()
        got = rows[i].cpu().numpy()
        ref = orc.encode_points(s, cfg).numpy()
        d = float(np.abs(got - ref).max())
        max_abs = max(max_abs, d)
        ok &= d < 1e-4
        same_bits &= bool(np.array_equal(enc.encode_points(s).cpu().numpy(), got))
        st = orc.strip_ambiguous(s, cfg)
        g2 = enc.encode_points(st).cpu().numpy()
        r2 = orc.encode_points(st, cfg).numpy()
        ok &= bool(np.allclose(g2, r2, rtol=1e-4, atol=1e-7))
        l2 = float(np.linalg.norm(g2 - r2) / max(np.linalg.norm(r2), 1e-30))
        max_l2 = max(max_l2, l2)
        ok &= l2 <= 1e-5
    return {"oracle_spot": len(scan_ids), "max_abs": max_abs, "stripped_rel_l2": max_l2,
            "rows_equal_single_scan_encode": same_bits, "ok": bool(ok and same_bits)}


def h2d_ceiling(h_points, dev, steps, barrier):
    """Bare pinned host -> device copy of the e2e step's bytes, nothing else in the stream: GB/s."""
    import torch
    d = torch.empty(h_points.shape, dtype=h_points.dtype, device=dev)
    d.copy_(h_points, non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        d.copy_(h_points, non_blocking=True)
    torch.cuda.synchronize(dev)
    dt = time.perf_counter() - t0
    del d
    return h_points.numel() * 4 * steps / dt / 1e9


def run_other_configs(enc, dev, pool, cores, kind, peak, steps):
    """BASELINE.json configs[2..3] and the shuffled-order variant, device-resident, at reduced
    step counts: scans/s, roofline fraction, and the CPU encoder on the same shape."""
    import torch
    from neural_spectral_codec_b200 import synth
    res = []
    for shape, n, shuffle in (("hdl32", 4096, False), ("beam128", 2048, False), ("hdl64", 2048, True)):
        points, offsets = synth.make_batch_resident(synth.SHAPES[shape], 0, n, dev, shuffle=shuffle)
        out = torch.empty((n, enc.output_dim), dtype=torch.float32, device=dev)
        ms, _ = time_encode(enc, points, offsets, out, steps, 3)
        total_points = int(points.shape[0])
        alg = 16 * total_points + 3200 * n
        chk = oracle_spot_check(enc, points, offsets.cpu().numpy(), out, [0, n // 2, n - 1])
        rec = {"workload": workload_name(n, shape, shuffle), "shape": shape, "shuffled": shuffle, "scans": n,
               "points": total_points, "steps": steps, "kernel_ms": ms, "value": n / (ms * 1e-3), "unit": UNIT,
               "frac": alg / (ms * 1e-3) / 1e9 / peak, "checks": chk}
        if pool is not None:
            v, cnt = cpu_throughput(pool, 8, cores, kind, shape, shuffle)
            rec["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
                                   "sample": f"{cnt} scans (8 per core)"}
        res.append(rec)
        del points, offsets, out
        torch.cuda.empty_cache()
    return res


def run_c5(enc, dev, rank, world, gather, lag, total_scans, steps):
    """BASELINE.json configs[4]: ``total_scans`` HDL-64 scans sharded over the ranks (strong
    scaling), descriptors gathered into the database replicated on every GPU; 256 oracle spot
    checks (every 391st scan) and a bit-comparison of every rank's database."""
    import numpy as np
    import torch
    import torch.distributed as dist
    from neural_spectral_codec_b200 import synth
    from neural_spectral_codec_b200.distributed import ShardedEncoder
    from oracle import nsc_oracle as orc
    lo, hi = synth.shard_range(total_scans, world, rank)
    points, offsets = synth.make_batch_resident(synth.HDL64, lo, hi - lo, dev)
    se = ShardedEncoder(enc, total_scans, mode=gather, lag=lag if gather == "fused" else 0)
    for _ in range(2):
        se.encode(points, offsets)
    se.flush()
    dist.barrier()
    torch.cuda.synchronize(dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        se.encode(points, offsets)
    db = se.flush()
    e1.record()
    dist.barrier()
    torch.cuda.synchronize(dev)
    ms = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=dev)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    # every rank's database vs an NCCL all-gather of plain single-GPU encodes of the same blocks
    local = torch.zeros((se.per, enc.output_dim), dtype=torch.float32, device=dev)
    enc.encode_points_batch(points, offsets, out=local[:hi - lo])
    want = torch.empty((world * se.per, enc.output_dim), dtype=torch.float32, device=dev)
    dist.all_gather_into_tensor(want, local)
    same = torch.tensor([1 if torch.equal(want[:total_scans], db) else 0], device=dev)
    dist.all_reduce(same, op=dist.ReduceOp.MIN)
    cfg = orc.OracleConfig()
    o = offsets.cpu().numpy()
    worst, checked = 0.0, 0
    for g in range(0, total_scans, 391):
        if lo <= g < hi:
            s = points[int(o[g - lo]):int(o[g - lo + 1])].cpu().numpy()
            worst = max(worst, float(np.abs(db[g].cpu().numpy() - orc.encode_points(s, cfg).numpy()).max()))
            checked += 1
    stats = torch.tensor([worst, float(checked)], dtype=torch.float64, device=dev)
    mx = stats.clone()
    dist.all_reduce(mx, op=dist.ReduceOp.MAX)
    dist.all_reduce(stats, op=dist.ReduceOp.SUM)
    rec = {"workload": f"{total_scans} HDL-64 scans sharded over {world} GPUs, descriptors gathered into the replicated database",
           "scaling": "strong", "scans": total_scans, "gather": gather, "gather_lag": lag if gather == "fused" else 0,
           "steps": steps,
           "ms_per_pass": float(ms.item()), "value": total_scans / (float(ms.item()) * 1e-3), "unit": UNIT,
           "points_per_gpu": int(points.shape[0]), "db_bytes": int(db.numel() * 4),
           "db_identical": bool(int(same.item()) == 1), "oracle_spot": int(stats[1].item()),
           "max_abs": float(mx[0].item())}
    rec["ok"] = rec["db_identical"] and rec["max_abs"] < 1e-4
    del points, offsets, se, db, want, local
    torch.cuda.empty_cache()
    return rec


# ----------------------------------------------------------------------------- GPU arm
def run_gpu_arm(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    from neural_spectral_codec_b200 import SpectralEncoder, synth
    from neural_spectral_codec_b200.distributed import ShardedEncoder

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit("--gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)")
        args.gpus = world
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # keep each rank (and the pinned host buffers it allocates) on the CPUs next to its GPU
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[local_rank]) if visible else local_rank
            pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(phys))
        except Exception:
            pass
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    # the CPU pool is spawned early (workers import torch while the GPU part runs)
    pool, cores, kind = None, os.cpu_count() or 1, cpu_kind()
    if rank == 0 and world == 1 and not args.no_cpu:
        pool = mp.get_context("spawn").Pool(cores)

    n_scans = args.scans
    enc = SpectralEncoder(n_elevation=16, n_azimuth=360, n_bins=50, alpha=2.0, learnable_alpha=True,
                          target_elevation_bins=16).to(dev)

    # synthetic scans of this rank, generated on the device from per-scan seeds
    first = rank * n_scans
    points, offsets = synth.make_batch_resident(synth.SHAPES[args.shape], first, n_scans, dev, shuffle=args.shuffle)
    offsets_host = offsets.cpu().numpy()
    total_points = int(points.shape[0])
    alg_bytes = 16 * total_points + 3200 * n_scans

    sharded = None
    if world > 1:
        try:
            sharded = ShardedEncoder(enc, world * n_scans, mode=args.gather,
                                     lag=args.gather_lag if args.gather == "fused" else 0)
        except Exception as exc:   # symmetric memory unavailable on this box: use the NCCL gather
            if args.gather != "fused":
                raise
            print(f"[bench] fused gather unavailable ({type(exc).__name__}: {exc}); using nccl", file=sys.stderr)
            ok = torch.tensor([0], device=dev)
        else:
            ok = torch.tensor([1], device=dev)
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)      # every rank must take the same path
        if int(ok.item()) == 0 and args.gather == "fused":
            args.gather = "nccl"
            sharded = ShardedEncoder(enc, world * n_scans, mode="nccl")
    out = torch.empty((n_scans, enc.output_dim), dtype=torch.float32, device=dev)

    def step():
        if sharded is None:
            enc.encode_points_batch(points, offsets, out=out)
        else:
            sharded.encode(points, offsets)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def flush():
        if sharded is not None:
            sharded.flush()

    for _ in range(args.warmup):
        step()
    flush()
    barrier()

    sampler = ClockSampler(torch.cuda.current_device() if "CUDA_VISIBLE_DEVICES" not in os.environ
                           else int(os.environ["CUDA_VISIBLE_DEVICES"].split(",")[local_rank]))
    sampler.start()
    stream = torch.cuda.current_stream(dev)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2 * args.steps)]
    end = torch.cuda.Event(enable_timing=True)
    barrier()
    for k in range(args.steps):
        ev[2 * k].record(stream)
        step()
        ev[2 * k + 1].record(stream)
    flush()                      # pipelined gather: the last step's database completes inside the timed region
    end.record(stream)
    barrier()
    clocks = sampler.stop()
    if args.dump_outputs and rank == 0:
        # one GPU: this batch's descriptors; N > 1: the gathered database, the same on every rank
        dump_outputs(args.dump_outputs, {"descriptors": out if sharded is None else sharded.flush()})
    total_ms = ev[0].elapsed_time(end)
    step_ms = [ev[2 * k].elapsed_time(ev[2 * k + 1]) for k in range(args.steps)]
    if world > 1:
        t = torch.tensor([total_ms], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    value = world * n_scans * args.steps / (total_ms * 1e-3)

    # the fused kernel alone (same launches, N=1 path) for the roofline; leaves the single-GPU
    # encode of this rank's block in `out`
    kern_avg_ms = sum(step_ms) / len(step_ms)
    breakdown = None
    if world > 1:
        kern_avg_ms, _ = time_encode(enc, points, offsets, out, args.steps, 0)
        # where the step time goes: every rank's plain kernel (GPUs of one box differ by a few %,
        # and a step ends when the slowest rank has stored), and the kernel with the peer stores
        # but without the signal-and-wait that ends a step
        def loop_ms(fn, n):
            barrier()
            e = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
            e[0].record(stream)
            for _ in range(n):
                fn()
            e[1].record(stream)
            barrier()
            return e[0].elapsed_time(e[1]) / n

        # interleaved rounds, so that drift of the box hits the three variants alike
        plain, fused, full = [], [], []
        n_loop = max(10, args.steps)
        for _ in range(2):
            plain.append(loop_ms(lambda: enc.encode_points_batch(points, offsets, out=out), n_loop))
            if args.gather == "fused":
                fused.append(loop_ms(lambda: sharded.encode(points, offsets, wait=False), n_loop))
                sharded.encode(points, offsets)      # a complete step again (flags and buffers in step)
                flush()
            full.append(loop_ms(lambda: sharded.encode(points, offsets), n_loop))
            flush()
        enc.encode_points_batch(points, offsets, out=out)
        barrier()
        med = lambda v: min(v) if v else None
        fused_ms = med(fused) if fused else med(plain)
        mine = torch.tensor([med(plain), fused_ms, med(full)], dtype=torch.float64, device=dev)
        allr = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allr, mine)
        breakdown = {"step_ms": total_ms / args.steps,
                     "how": f"after the timed region: 2 interleaved rounds of {n_loop} launches of each variant, best of the two, ms per launch",
                     "kernel_ms_per_rank": [float(t[0]) for t in allr],
                     "kernel_with_peer_stores_ms_per_rank": [float(t[1]) for t in allr],
                     "full_step_ms_per_rank": [float(t[2]) for t in allr],
                     "note": "step = slowest rank's kernel with peer stores + one signal-and-wait kernel; "
                             "weak-scaling efficiency against ONE GPU cannot exceed that GPU's kernel time / the "
                             "slowest rank's"}
    peak, peak_src = hbm_peak()
    achieved = alg_bytes / (kern_avg_ms * 1e-3) / 1e9
    traffic, traffic_src = None, "not captured for this shape (ncu --set full is a separate, profiler-run pass)"
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath):
        tj = json.load(open(tpath))
        if tj.get("scans") == n_scans and args.shape == "hdl64" and not args.shuffle:
            traffic = tj.get("dram_bytes_per_launch")
            traffic_src = ("constant read from profiles/traffic.json: dram__bytes_read.sum + dram__bytes_write.sum of one "
                           f"ncu --set full capture of this kernel on this workload ({tj.get('source', 'see profiles/')}); "
                           "NOT measured in this run")
    roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic, "traffic_source": traffic_src,
                "kernel": "encode_points_ws_kernel<0>", "kernel_ms": kern_avg_ms,
                "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src}

    # ---- checks on the timed output (outside every timed region) ----------------------------------
    checks = {}
    ids = sorted(set(int(x) for x in np.linspace(0, n_scans - 1, 8 if world == 1 else 4)))
    db = None
    if sharded is not None:
        db = sharded.flush()[:world * n_scans]
        rows = db[rank * sharded.per: rank * sharded.per + n_scans]      # the timed output, this rank's block
        want = torch.empty((world * sharded.per, enc.output_dim), dtype=torch.float32, device=dev)
        local = torch.zeros((sharded.per, enc.output_dim), dtype=torch.float32, device=dev)
        local[:n_scans] = out
        dist.all_gather_into_tensor(want, local)                         # plain NCCL gather of single-GPU encodes
        same = torch.tensor([1 if torch.equal(want[:world * n_scans], db) else 0], device=dev)
        dist.all_reduce(same, op=dist.ReduceOp.MIN)
        checks["db_identical"] = bool(int(same.item()) == 1)
        del want, local
    else:
        rows = out
        checks["db_identical"] = None
    spot = oracle_spot_check(enc, points, offsets_host, rows, ids)
    if world > 1:
        agg = torch.tensor([spot["max_abs"], spot["stripped_rel_l2"], 0.0 if spot["ok"] else 1.0],
                           dtype=torch.float64, device=dev)
        dist.all_reduce(agg, op=dist.ReduceOp.MAX)
        spot.update(max_abs=float(agg[0].item()), stripped_rel_l2=float(agg[1].item()), ok=bool(agg[2].item() == 0.0),
                    oracle_spot=spot["oracle_spot"] * world)
    checks.update(spot)
    checks["what"] = ("rows of the timed output vs the CPU oracle on the same clouds (max_abs < 1e-4), GPU vs oracle on the "
                      "clouds stripped of edge points (rtol 1e-4 / atol 1e-7, rel. L2 <= 1e-5), rows bit-identical to "
                      "single-scan encodes" + ("; gathered database on every rank bit-identical to an NCCL all-gather of "
                                               "single-GPU encodes" if world > 1 else ""))
    checks["ok"] = bool(checks["ok"] and checks["db_identical"] is not False)

    # ---- end to end: pinned host buffers -> descriptors on the host, through the public API -------
    n_e2e = min(n_scans, args.e2e_scans)
    e_off = offsets[: n_e2e + 1].cpu()
    h_points = torch.empty((int(e_off[-1]), 4), dtype=torch.float32).pin_memory()
    h_points.copy_(points[: int(e_off[-1])])
    h_out = torch.empty((n_e2e, enc.output_dim), dtype=torch.float32).pin_memory()
    hp, ho, hoff = h_points.numpy(), h_out.numpy(), e_off.numpy()
    enc.encode_scans((hp, hoff), out=ho)
    barrier()
    e2e_steps = max(2, min(args.steps, 5))
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        enc.encode_scans((hp, hoff), out=ho)     # synchronous: returns when ho is complete
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_same = bool(np.array_equal(ho, rows[:n_e2e].cpu().numpy()))
    h2d_bytes = int(hp.nbytes + hoff.nbytes)
    e2e = {"value": world * n_e2e * e2e_steps / e2e_s, "unit": UNIT,
           "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": int(ho.nbytes),
           "scans_per_step_per_gpu": n_e2e, "steps": e2e_steps,
           "api": "SpectralEncoder.encode_scans -> nsc_pipeline_encode (pinned host buffers)",
           "h2d_gbs_per_gpu": h2d_bytes * e2e_steps / e2e_s / 1e9,
           "equals_device_path": e2e_same}
    checks["ok"] = bool(checks["ok"] and e2e_same)
    if not args.no_extras:
        # the ceiling: the same pinned bytes through a bare host -> device copy on every rank at once
        ceil_gbs = h2d_ceiling(h_points, dev, e2e_steps, barrier)
        if world > 1:
            t = torch.tensor([ceil_gbs], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
            ceil_gbs = float(t.item())
        e2e["h2d_ceiling_gbs_per_gpu"] = ceil_gbs
        e2e["frac_of_h2d_ceiling"] = e2e["h2d_gbs_per_gpu"] / ceil_gbs
        e2e["ceiling_note"] = ("bare cudaMemcpyAsync of the step's pinned input, all ranks at once (slowest rank); the "
                               "end-to-end path cannot exceed it: 16 B per point have to cross PCIe")
    if not args.no_extras and rank == 0:
        # the reference's own call pattern (pipeline.py:336-354): one encode_points(numpy) per scan
        host_scans = [np.array(points[int(offsets_host[i]):int(offsets_host[i + 1])].cpu().numpy()) for i in range(64)]
        for s_ in host_scans[:4]:
            enc.encode_points(s_).detach().cpu().numpy()
        t0 = time.perf_counter()
        per = [enc.encode_points(s_).detach().cpu().numpy() for s_ in host_scans]
        dt = time.perf_counter() - t0
        same = all(np.array_equal(per[i], rows[i].cpu().numpy()) for i in range(len(per)))
        e2e["per_scan"] = {"value": len(host_scans) / dt, "unit": UNIT, "ms_per_scan": 1e3 * dt / len(host_scans),
                           "scans": len(host_scans), "equals_batch_path": bool(same),
                           "api": "encoder.encode_points(points_np).detach().cpu().numpy() per scan, pageable numpy "
                                  "input (the reference's loop, pipeline.py:336-354)"}
        enc.encode_scans(host_scans[:8])
        t0 = time.perf_counter()
        reps = 4
        for _ in range(reps):
            lst = enc.encode_scans(host_scans)
        dt = time.perf_counter() - t0
        e2e["pageable_list"] = {"value": reps * len(host_scans) / dt, "unit": UNIT, "scans": len(host_scans),
                                "equals_batch_path": bool(np.array_equal(lst, np.stack(per))),
                                "api": "encoder.encode_scans(list of pageable numpy scans)"}
        checks["ok"] = bool(checks["ok"] and same)
    del h_points, h_out

    # ---- other configs (N = 1) / the sharded 100 k-scan config (N > 1) ------------------------------
    other, c5 = None, None
    if not args.no_extras:
        del points, offsets, out, rows, db
        sharded = None
        torch.cuda.empty_cache()
        if world == 1:
            other = run_other_configs(enc, dev, pool, cores, kind, peak, max(3, min(args.steps, 10)))
            checks["ok"] = bool(checks["ok"] and all(c["checks"]["ok"] for c in other))
        else:
            c5 = run_c5(enc, dev, rank, world, args.gather, args.gather_lag, args.c5_scans, 3)
            checks["ok"] = bool(checks["ok"] and c5["ok"])

    cpu_baseline = None
    if pool is not None:
        per_core = 32
        v, n = cpu_throughput(pool, per_core, cores, kind)
        # the reference's native call pattern: one process looping encode_points (pipeline.py:336-354)
        encode = make_cpu_encoder(kind)
        single_scans = [synth.make_scan(synth.HDL64, 200000 + i).numpy() for i in range(12)]
        encode(single_scans[0])
        t0 = time.perf_counter()
        for s_ in single_scans:
            encode(s_)
        single = len(single_scans) / (time.perf_counter() - t0)
        cpu_baseline = {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
                        "sample": f"{n} HDL-64 scans ({per_core} per core), {cpu_kind_text(kind)}, "
                                  "one single-threaded process per core",
                        "single_process_value": single,
                        "single_process_sample": f"{len(single_scans)} scans in one process, torch threads = "
                                                 f"{torch.get_num_threads()} (the reference's per-scan loop)"}
        pool.close()
        pool.join()

    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": total_ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": make_config(args, world),
            "workload_stats": {"points_per_gpu": total_points, "input_bytes_per_gpu": 16 * total_points},
            "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "checks": checks,
            "gpu_launches": args.steps * (1 if world == 1 or args.gather != "fused" else 2), "clocks": clocks,
        }
        if breakdown is not None:
            line["scaling_breakdown"] = breakdown
        if other is not None:
            line["configs"] = other
        if c5 is not None:
            line["c5"] = c5
        emit(line)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if not checks["ok"] and not args.no_checks:
        print("[bench] CHECKS FAILED: " + json.dumps(checks), file=sys.stderr)
        raise SystemExit(1)


# ----------------------------------------------------------------------------- retrieval (secondary)
def run_retrieval(args):
    """Secondary workload (SURVEY.md 8(f) rank 1): Wasserstein top-K over a 100 k x 800 database.
    The reference's only stated target for this stage is 27 ms per query at 100 k descriptors
    (configs/training.yaml:99). Not the BASELINE.json metric; printed in the same JSON shape."""
    import torch

    from neural_spectral_codec_b200.retrieval import WassersteinRetriever
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(7)
    n_db, nq, k = args.db, args.queries, args.topk
    db = torch.rand((n_db, 800), generator=g, device=dev) ** 4
    db /= db.sum(1, keepdim=True)
    q = db[torch.randint(0, n_db, (nq,), device=dev)] * (1 + 0.05 * torch.rand((nq, 800), device=dev))
    r = WassersteinRetriever(device=dev)
    r.add_to_database(db)
    for _ in range(max(args.warmup, 3)):
        r.query_batch(q, top_k=k)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        res = r.query_batch(q, top_k=k)
    e1.record()
    torch.cuda.synchronize()
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dict(zip(("indices", "distances", "counts"), res)))
    ms = e0.elapsed_time(e1) / args.steps
    passes = -(-nq // 8)                                   # one pass over the CDF rows serves 8 queries
    alg_bytes = passes * n_db * 800 * 4
    peak, _ = hbm_peak()
    line = {"metric": "retrieval_queries_per_sec_at_100k_db", "value": nq / (ms * 1e-3), "unit": "queries/s",
            "n_gpus": 1, "steps": args.steps, "warmup": max(args.warmup, 3), "ms_per_step": ms,
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"Wasserstein top-{k} of {nq} queries over a {n_db} x 800 descriptor database",
                       "ms_per_query": ms / nq, "reference_target_ms_per_query": 27.0},
            "roofline": {"bound": "hbm", "achieved": alg_bytes / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": alg_bytes / (ms * 1e-3) / 1e9 / peak, "traffic": None,
                         "note": "whole call (all kernels + host launch gaps); algorithmic bytes = one pass over the "
                                 "CDF rows per group of <= 8 queries"},
            "gpu_launches": args.steps * (passes + 1)}
    if not args.no_cpu:
        from oracle import retrieval_oracle as ro
        dbc, qc = db.cpu(), q.cpu()
        n = min(nq, 4)
        t0 = time.perf_counter()
        for i in range(n):
            ro.query_topk(qc[i], dbc, k)
        cpu_ms = 1e3 * (time.perf_counter() - t0) / n
        line["cpu_baseline"] = {"value": 1e3 / cpu_ms, "unit": "queries/s", "cores": torch.get_num_threads(),
                                "kind": "port", "sample": f"{n} queries, oracle/retrieval_oracle.py (torch CPU)"}
    emit(line)


# ----------------------------------------------------------------------------- keyframe gate (secondary)
def run_keyframe(args):
    """Secondary workload (SURVEY.md 8(f) rank 3): voxel-IoU of (last keyframe, scan) pairs, the
    expensive criterion of the reference's keyframe gate (pose_utils.py:323-389), 5000 + 5000 points
    per pair as after its subsample. Kernel time with device-resident pairs, the public batched call
    from host arrays, and the reference's own compute_overlap on one core."""
    import ctypes as C

    import numpy as np
    import torch

    from neural_spectral_codec_b200 import _lib, keyframe as kf, synth
    dev = torch.device("cuda")
    lib = _lib.load()
    n_pairs = args.pairs
    shape = synth.SensorShape("kf", 32, -24.8, 2.0, 400)
    rng = np.random.default_rng(0)
    clouds = [synth.make_scan(shape, 300 + i).numpy() for i in range(16)]
    pairs = []
    for i in range(n_pairs):
        a, b = clouds[i % 16], clouds[(i + 1 + i // 16) % 16]
        pa = a[rng.choice(len(a), 5000, replace=False)]
        pb = b[rng.choice(len(b), 5000, replace=False)]
        T = np.eye(4)
        ang = 0.01 * (i % 7)
        T[:2, :2] = [[np.cos(ang), -np.sin(ang)], [np.sin(ang), np.cos(ang)]]
        T[0, 3] = 0.05 * (i % 5)
        pairs.append((pa, pb, T))
    iou = kf.compute_overlap_batch(pairs)                       # warm-up + result
    t0 = time.perf_counter()
    for _ in range(3):
        kf.compute_overlap_batch(pairs)
    api_s = (time.perf_counter() - t0) / 3
    # kernel alone, inputs resident
    pts = torch.from_numpy(np.concatenate([np.concatenate([p[0], p[1]]) for p in pairs])).to(dev)
    offs = torch.arange(0, 2 * n_pairs + 1, dtype=torch.int64, device=dev) * 5000
    Ts = torch.from_numpy(np.stack([p[2] for p in pairs])).to(dev)
    cnt = torch.empty((n_pairs, 3), dtype=torch.int32, device=dev)
    out = torch.empty((n_pairs,), dtype=torch.float64, device=dev)
    total = 10000 * n_pairs
    ws = torch.empty(int(lib.nsc_voxel_overlap_workspace_bytes(total, 10000, n_pairs)) // 4 + 1, dtype=torch.int32, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def launch():
        st = lib.nsc_voxel_overlap_batch(pts.data_ptr(), 4, 0, offs.data_ptr(), total, 10000, Ts.data_ptr(), n_pairs, 0.2,
                                         cnt.data_ptr(), out.data_ptr(), ws.data_ptr(), ws.numel() * 4, stream)
        assert st == 0
    for _ in range(3):
        launch()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(args.steps):
        launch()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"overlap": out, "voxel_counts": cnt})
    assert np.array_equal(out.cpu().numpy(), iou)
    peak, _ = hbm_peak()
    line = {"metric": "keyframe_overlap_pairs_per_sec", "value": n_pairs / (ms * 1e-3), "unit": "pairs/s", "n_gpus": 1,
            "steps": args.steps, "warmup": 3, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64 transform / f32 voxels / int32 sets", "data": "synthetic",
            "config": {"workload": f"voxel IoU of {n_pairs} cloud pairs of 5000 + 5000 xyzi points, 0.2 m voxels"},
            "roofline": {"bound": "latency (shared-memory hash set: one atomicCAS chain per point)",
                         "achieved": 16.0 * total / (ms * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": 16.0 * total / (ms * 1e-3) / 1e9 / peak, "traffic": None},
            "e2e": {"value": n_pairs / api_s, "unit": "pairs/s", "api": "keyframe.compute_overlap_batch(host arrays)",
                    "h2d_bytes_per_step": 16 * total, "d2h_bytes_per_step": 8 * n_pairs},
            "gpu_launches": args.steps}
    if not args.no_cpu:
        src = reference_src()
        kind = "reference" if src else "port"
        if src:
            sys.path.insert(0, src)
            from data.pose_utils import compute_overlap as ref_overlap
        else:
            from oracle.keyframe_oracle import compute_overlap as ref_overlap
        n = min(n_pairs, 24)
        t0 = time.perf_counter()
        got = [ref_overlap(p[0], p[1], p[2], voxel_size=0.2) for p in pairs[:n]]
        cpu_s = (time.perf_counter() - t0) / n
        line["cpu_baseline"] = {"value": 1.0 / cpu_s, "unit": "pairs/s", "cores": 1, "kind": kind,
                                "sample": f"{n} pairs, compute_overlap (pose_utils.py:323-389), one process"}
        line["checks"] = {"equal_to_cpu": bool(np.array_equal(np.array(got), iou[:n]))}
    emit(line)


# ----------------------------------------------------------------------------- wire format (secondary)
def run_quantize(args):
    """Secondary workload (SURVEY.md 8(f) rank 4): the uint16 wire format of a 100 k x 800 database
    (encoding/quantization.py:131-192, generalised from 50 to 800 bins): quantise + dequantise."""
    import numpy as np
    import torch

    from neural_spectral_codec_b200.quantization import HistogramQuantizer
    dev = torch.device("cuda")
    n = args.db
    g = torch.Generator(device=dev).manual_seed(3)
    h = torch.rand((n, 800), generator=g, device=dev) ** 4
    h /= h.sum(1, keepdim=True)
    qz = HistogramQuantizer(n_bins=800, device=dev)
    for _ in range(3):                       # warm-up of both directions (and of the allocator's blocks)
        q = qz.quantize(h)
        d = qz.dequantize(q)
    torch.cuda.synchronize()
    e0, e1, e2, e3 = (torch.cuda.Event(enable_timing=True) for _ in range(4))
    e0.record()
    for _ in range(args.steps):
        q = qz.quantize(h)
    e1.record()
    torch.cuda.synchronize()
    e2.record()
    for _ in range(args.steps):
        d = qz.dequantize(q)
    e3.record()
    torch.cuda.synchronize()
    ms_q, ms_d = e0.elapsed_time(e1) / args.steps, e2.elapsed_time(e3) / args.steps
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"quantized": q, "dequantized": d})
    peak, _ = hbm_peak()
    bytes_q = n * 800 * (4 + 2)
    line = {"metric": "descriptors_quantised_per_sec", "value": n / (ms_q * 1e-3), "unit": "descriptors/s", "n_gpus": 1,
            "steps": args.steps, "warmup": 3, "ms_per_step": ms_q, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32 -> u16", "data": "synthetic",
            "config": {"workload": f"uint16 quantisation of {n} x 800 descriptors (sum of a row = 65535 exactly)",
                       "dequantise_ms": ms_d},
            "roofline": {"bound": "hbm", "achieved": bytes_q / (ms_q * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": bytes_q / (ms_q * 1e-3) / 1e9 / peak, "traffic": None,
                         "dequantise_frac": bytes_q / (ms_d * 1e-3) / 1e9 / peak},
            "gpu_launches": 2 * args.steps,
            "checks": {"row_sums_65535": bool((q.to(torch.int32).sum(1) == 65535).all().item()),
                       "max_roundtrip_error": float((d - h).abs().max().item())}}
    if not args.no_cpu:
        from oracle import quantization_oracle as qo
        hc = h[:2000].cpu().numpy()
        t0 = time.perf_counter()
        want = np.stack([qo.quantize(r) for r in hc])
        cpu_s = (time.perf_counter() - t0) / len(hc)
        line["cpu_baseline"] = {"value": 1.0 / cpu_s, "unit": "descriptors/s", "cores": 1, "kind": "port",
                                "sample": f"{len(hc)} rows, oracle/quantization_oracle.py (the reference's quantiser "
                                          "is hard-wired to 50 bins)"}
        line["checks"]["equal_to_cpu"] = bool(np.array_equal(want, q[:2000].cpu().numpy()))
    emit(line)


DUMP_BYTES = 64_000_000 - (64 << 10)     # 64 MB in all, less room for the .npy headers


def dump_outputs(dump_dir, arrays):
    """``arrays``: name -> torch tensor or numpy array, all with the same number of rows. Writes
    ``dump_dir/<name>.npy``; floating arrays keep their type, integer ones become float32 (up to
    16 bits) or float64, both exact. Above DUMP_BYTES in all, every array keeps the same seeded
    sample of rows, in order, and ``rows.npy`` lists them."""
    import numpy as np
    import torch
    arrays = {name: a if torch.is_tensor(a) else torch.from_numpy(np.asarray(a)) for name, a in arrays.items()}
    out_type = {name: torch.float64 if a.element_size() > (4 if a.is_floating_point() else 2) else torch.float32
                for name, a in arrays.items()}
    n = len(next(iter(arrays.values())))
    row_bytes = sum(a.numel() * out_type[name].itemsize for name, a in arrays.items()) / max(n, 1)
    rows = None
    if n * row_bytes > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n, int(DUMP_BYTES // (row_bytes + 8)), replace=False))
    os.makedirs(dump_dir, exist_ok=True)
    for name, a in arrays.items():
        a = a.detach().to(out_type[name])           # where the array lives; only the kept rows reach the host
        if rows is not None:
            a = a[torch.from_numpy(rows).to(a.device)]
        np.save(os.path.join(dump_dir, name + ".npy"), a.cpu().numpy())
    if rows is not None:
        np.save(os.path.join(dump_dir, "rows.npy"), rows.astype(np.float64))


def emit(line: dict) -> None:
    """The one JSON line goes to the REAL stdout; everything else a library prints to fd 1
    (e.g. NCCL's version banner) was redirected to stderr in main()."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scans", type=int, default=N_SCANS, help="scans per GPU")
    ap.add_argument("--e2e-scans", type=int, default=1024, help="scans per end-to-end step")
    ap.add_argument("--c5-scans", type=int, default=100000, help="N > 1: total scans of the sharded config")
    ap.add_argument("--gather", default="fused", choices=["nccl", "fused"])
    ap.add_argument("--gather-lag", type=int, default=0, choices=[0, 1],
                    help="fused gather: 1 = pipelined (wait for the previous step's peers only), 0 = every step complete on return")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline legs")
    ap.add_argument("--no-extras", action="store_true",
                    help="headline line only: skip the other configs, the per-scan call pattern and the H2D ceiling")
    ap.add_argument("--no-checks", action="store_true",
                    help="measurement-only library builds (tools/ab.py experiments) whose output is not a descriptor")
    ap.add_argument("--shape", default="hdl64", choices=sorted(SHAPE_DESC),
                    help="sensor shape of the synthetic scans (BASELINE.json configs 2-4; default = the metric's config)")
    ap.add_argument("--shuffle", action="store_true", help="random point order inside each scan")
    ap.add_argument("--workload", default="encode", choices=["encode", "retrieval", "keyframe", "quantize"],
                    help="encode = the BASELINE.json metric (default); retrieval / keyframe = secondary lines "
                         "for the stage-1 retrieval and the keyframe-gate voxel IoU")
    ap.add_argument("--pairs", type=int, default=512, help="keyframe: cloud pairs per launch")
    ap.add_argument("--db", type=int, default=100000, help="retrieval: database rows")
    ap.add_argument("--queries", type=int, default=8, help="retrieval: queries per call")
    ap.add_argument("--topk", type=int, default=10, help="retrieval: K")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the timed path returned in its last step to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs needs the GPU path (--impl b200)")
    if args.impl == "reference":
        run_reference_arm(args)
        return
    args.warmup = max(args.warmup, 3)
    if args.workload == "retrieval":
        run_retrieval(args)
    elif args.workload == "keyframe":
        run_keyframe(args)
    elif args.workload == "quantize":
        run_quantize(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
