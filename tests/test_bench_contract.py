"""bench.py prints exactly one JSON line with the contract's keys (reference arm runs on CPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def test_reference_arm_prints_one_json_line():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    lines = [l for l in r.stdout.splitlines() if l.strip()]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "scans_per_sec_encoded_to_800d" and d["unit"] == "scans/s"
    assert d["value"] > 0 and d["higher_is_better"] is True and d["vs_baseline"] is None
    assert d["cpu_baseline"]["kind"] in ("reference", "port") and d["cpu_baseline"]["cores"] >= 1
    assert d["steps"] == 1 and d["warmup"] == 0                     # honours --steps / --warmup
    assert d["e2e"] == {"value": d["value"], "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert "workload" in d["config"] and "model" not in d["config"]


def test_other_ranks_of_the_reference_arm_do_nothing():
    env = dict(os.environ, RANK="1", WORLD_SIZE="2", LOCAL_RANK="1")
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--gpus", "2"],
                       capture_output=True, text=True, timeout=120, env=env)
    assert r.returncode == 0 and r.stdout.strip() == ""


def test_both_arms_describe_the_same_config():
    """The driver compares the `config` object of the GPU arm and of the reference arm."""
    import argparse
    sys.path.insert(0, ROOT)
    import bench
    for gpus in (1, 8):
        a = argparse.Namespace(scans=bench.N_SCANS, shape="hdl64", shuffle=False, gather="fused", gather_lag=0, gpus=gpus)
        assert bench.make_config(a, gpus) == bench.make_config(a, gpus)
        assert "model" not in bench.make_config(a, gpus) and "workload" in bench.make_config(a, gpus)
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                        "--warmup", "0", "--gpus", "8"], capture_output=True, text=True, timeout=600,
                       env=dict(os.environ, RANK="0", WORLD_SIZE="8"))
    d = json.loads(r.stdout.strip().splitlines()[-1])
    a = argparse.Namespace(scans=bench.N_SCANS, shape="hdl64", shuffle=False, gather="fused", gather_lag=0, gpus=8)
    assert d["config"] == bench.make_config(a, 8) and d["n_gpus"] == 8


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "0"],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode == 2 and "--steps" in r.stderr and r.stdout == ""


def test_dump_outputs_converts_exactly_and_samples_rows_above_64_mb(tmp_path):
    sys.path.insert(0, ROOT)
    import bench
    bench.dump_outputs(str(tmp_path / "small"), {"q": np.arange(12, dtype=np.uint16).reshape(6, 2),
                                                  "i": np.arange(6, dtype=np.int64) + 2 ** 40,
                                                  "f": np.linspace(0, 1, 6)})
    q, i, f = (np.load(tmp_path / "small" / f"{k}.npy") for k in ("q", "i", "f"))
    assert q.dtype == np.float32 and q.tolist() == np.arange(12).reshape(6, 2).tolist()
    assert i.dtype == np.float64 and i.tolist() == [2 ** 40 + k for k in range(6)]
    assert f.dtype == np.float64 and not os.path.exists(tmp_path / "small" / "rows.npy")

    n = 22000                                        # 22000 x 800 float32 = 70 MB
    big = {"d": np.repeat(np.arange(n, dtype=np.float32)[:, None], 800, 1), "label": np.arange(n, dtype=np.int32)}
    bench.dump_outputs(str(tmp_path / "big"), big)
    bench.dump_outputs(str(tmp_path / "again"), big)
    rows = np.load(tmp_path / "big" / "rows.npy")
    np.testing.assert_array_equal(np.load(tmp_path / "again" / "rows.npy"), rows)     # the same sample every time
    d, label = np.load(tmp_path / "big" / "d.npy"), np.load(tmp_path / "big" / "label.npy")
    assert sum(os.path.getsize(tmp_path / "big" / f) for f in os.listdir(tmp_path / "big")) <= 64_000_000
    assert len(rows) > n // 2 and np.all(np.diff(rows) > 0)
    np.testing.assert_array_equal(d, big["d"][rows.astype(np.int64)])
    np.testing.assert_array_equal(label, rows)


@pytest.mark.gpu
def test_dumped_descriptors_are_the_timed_output_for_the_seeded_scans(tmp_path):
    from neural_spectral_codec_b200 import SpectralEncoder, synth
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "2", "--warmup", "0",
                        "--scans", "40", "--no-cpu", "--no-extras", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    d = json.loads(r.stdout.strip().splitlines()[-1])
    assert d["steps"] == 2 and d["gpu_launches"] == 2 and d["checks"]["ok"]
    assert os.listdir(tmp_path) == ["descriptors.npy"]
    got = np.load(tmp_path / "descriptors.npy")
    # plumbing only (the dump is the last timed step for the seeded scans): parity with the oracle is checks.ok
    enc = SpectralEncoder(n_elevation=16, n_azimuth=360, n_bins=50, alpha=2.0, learnable_alpha=True,
                          target_elevation_bins=16).to("cuda")
    pts, offs = synth.make_batch(synth.HDL64, 0, 40, device="cuda")
    want = enc.encode_points_batch(pts, offs).cpu().numpy()
    assert got.dtype == np.float32 and got.shape == (40, 800)
    np.testing.assert_array_equal(got, want)
