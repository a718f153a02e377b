#!/usr/bin/env python
"""End-to-end example on synthetic scans: encode a sequence from host memory, put the descriptors
into the retrieval database with their positions, query with the spatial filter, build the same
database from the encoder's uint16 wire rows and compare its neighbours, and pack one keyframe
record. Mirrors what the reference's online loop does per scan
(src/pipeline.py:230-273: encode_points -> add_keyframe -> get_loop_closures), batched.

    python examples/encode_and_retrieve.py [--scans 200]
"""
import argparse
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from neural_spectral_codec_b200 import SpectralEncoder, synth  # noqa: E402
from neural_spectral_codec_b200.quantization import (CompressedDescriptor, HistogramQuantizer,  # noqa: E402
                                                     compute_point_cloud_hash)
from neural_spectral_codec_b200.retrieval import WassersteinRetriever  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--scans", type=int, default=200)
    a = ap.parse_args()
    # a "trajectory" that revisits its start: scan i and scan i + n/2 see the same scene
    half = a.scans // 2
    scans = [synth.make_scan(synth.HDL64, i % half).numpy() for i in range(a.scans)]
    positions = np.stack([[10.0 * (i % half), 200.0 * (i // half), 0.0] for i in range(a.scans)])

    enc = SpectralEncoder(n_elevation=16, n_azimuth=360, n_bins=50, alpha=2.0, learnable_alpha=True,
                          target_elevation_bins=16).to("cuda")
    enc.encode_scans(scans[:4])                                   # warm-up: allocates the staging buffers
    t0 = time.perf_counter()
    desc = enc.encode_scans(scans)                                # (B, 800) numpy, host in / host out
    dt = time.perf_counter() - t0
    print(f"encoded {a.scans} scans ({sum(len(s) for s in scans) / 1e6:.1f} M points) in {dt * 1e3:.1f} ms "
          f"= {a.scans / dt:.0f} scans/s from pageable host arrays")

    retr = WassersteinRetriever(device="cuda")
    retr.add_to_database(desc, positions=positions)
    q = slice(half, half + 5)                                     # second pass over the same places
    idx, dist, cnt = retr.query_batch(desc[q], top_k=3, query_positions=positions[q],
                                      spatial_filter_distance=50.0)
    for j in range(5):
        print(f"query scan {half + j}: nearest database scans {idx[j].tolist()} "
              f"(expected first: {j}), distances {np.round(dist[j].cpu().numpy(), 5).tolist()}")

    # the same database kept in the uint16 wire format: rows straight from the encoder's epilogue,
    # a quarter of the float32 database's memory
    rows16 = enc.encode_scans(scans, dtype=np.uint16)
    retr16 = WassersteinRetriever(device="cuda", database_dtype=torch.uint16)
    retr16.add_to_database(rows16, positions=positions)
    idx16, dist16, _ = retr16.query_batch(desc[q], top_k=3, query_positions=positions[q],
                                          spatial_filter_distance=50.0)
    print(f"uint16 database ({retr16.database_cdfs.element_size() * retr16.database_cdfs.numel() // 1024} KB of CDF "
          f"rows): same neighbours as float32: {torch.equal(idx16, idx)}, max |distance difference| = "
          f"{float((dist16 - dist)[torch.isfinite(dist)].abs().max()):.2g}")

    qz = HistogramQuantizer(n_bins=enc.output_dim)
    rec = CompressedDescriptor(histogram=qz.quantize(desc[0]), pose=np.array([0, 0, 0, 1, 0, 0, 0], np.float32),
                               timestamp=0.0, keyframe_id=0, point_cloud_hash=compute_point_cloud_hash(scans[0]))
    print(f"keyframe record: {len(rec.to_bytes())} bytes (uint16 histogram sum = {int(rec.histogram.sum())})")


if __name__ == "__main__":
    main()
