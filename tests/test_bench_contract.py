"""CPU: the reference arm of bench.py (the oracle on the host cores) prints one JSON line with the keys
the driver reads; the default arm refuses to run without a GPU instead of falling back to the CPU."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from conftest import ROOT


def test_reference_arm_json_line():
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--fragments", "64"], capture_output=True, text=True, timeout=300)
    assert out.returncode == 0, out.stderr[-500:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    assert line["impl"] == "reference" and line["unit"] == "GB/s" and line["higher_is_better"] is True
    assert line["value"] > 0 and line["n_gpus"] == 1 and line["dtype"] == "u8"
    assert line["cpu_baseline"]["kind"] == "port" and line["cpu_baseline"]["cores"] >= 1
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["e2e"]["d2h_bytes_per_step"] == 0
    assert line["e2e"]["value"] == line["value"]


def test_default_arm_needs_a_gpu():
    import torch
    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "0",
                          "--fragments", "16"], capture_output=True, text=True, timeout=300)
    assert out.returncode != 0          # no CPU fallback: the product path fails loudly


def test_dump_outputs_samples_within_the_budget(tmp_path, monkeypatch):
    """outputs longer than their share are sampled at the same seeded positions every time; values stay exact"""
    import torch
    sys.path.insert(0, ROOT)
    import bench
    monkeypatch.setattr(bench, "DUMP_BYTES", 16000)                     # 1000 elements per output
    stream = torch.from_numpy(np.random.default_rng(1).integers(0, 256, 50000, dtype=np.uint8))
    index = torch.arange(101, dtype=torch.int64) * 3 + (1 << 40)
    for d in ("a", "b"):
        bench.dump_outputs(str(tmp_path / d), {"compressed": stream, "compressed_index": index}, 2026)
    a = np.load(tmp_path / "a" / "compressed.npy")
    assert a.dtype == np.float32 and a.size == 1000
    assert np.array_equal(a, np.load(tmp_path / "b" / "compressed.npy"))
    pos = np.sort(np.random.default_rng(2026).integers(0, stream.numel(), 1000))
    assert np.array_equal(a, stream.numpy()[pos].astype(np.float32))
    i = np.load(tmp_path / "a" / "compressed_index.npy")                 # short: written whole, float64 is exact
    assert i.dtype == np.float64 and np.array_equal(i.astype(np.int64), index.numpy())
    assert sum(f.stat().st_size for f in (tmp_path / "a").iterdir()) <= 16000 + 2 * 128


def test_dump_outputs_is_refused_outside_config_2():
    for extra in (["--impl", "reference"], ["--config", "3"]):
        out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", "unused"] + extra,
                             capture_output=True, text=True, timeout=300)
        assert out.returncode == 2 and "--dump-outputs" in out.stderr


@pytest.mark.gpu
def test_dumped_outputs_are_the_oracles_stream_and_the_input(tmp_path):
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pyoracle
    from snappy_jl_b200 import synth
    steps, nfrag, seed = 3, 32, 2026
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", str(steps), "--warmup", "1",
                          "--fragments", str(nfrag), "--no-extra", "--no-cpu-baseline", "--no-e2e",
                          "--dump-outputs", str(tmp_path)], capture_output=True, text=True, timeout=600)
    assert out.returncode == 0, out.stderr[-2000:]
    assert json.loads(out.stdout.strip().splitlines()[-1])["steps"] == steps
    raw = synth.mix(nfrag, seed=seed)                  # bench.py's config 2 input
    sys.path.insert(0, ROOT)
    import bench
    assert 3 * 8 * raw.size <= bench.DUMP_BYTES        # each of the three outputs is small enough to be dumped whole
    want = pyoracle.compress_np(raw)
    assert np.array_equal(np.load(tmp_path / "compressed.npy"), want.astype(np.float32))
    assert np.array_equal(np.load(tmp_path / "uncompressed.npy"), raw.astype(np.float32))
    _, sizes = pyoracle.compress_fragments(raw, raw.size, 0, nfrag)
    idx = np.load(tmp_path / "compressed_index.npy").astype(np.int64)
    assert idx[0] == len(pyoracle.encode32(raw.size)) and np.array_equal(np.diff(idx), sizes.astype(np.int64))
