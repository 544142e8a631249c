"""GPU: range reads (snappy_b200_uncompress_range*_device) against a full uncompress_device, alternating them in the
same run, on a 1 GiB synth.mix stream (256 MiB repeated 4 times; larger than the 126 MB L2) with its side index.

Cases (offsets drawn from --seed, a new one for every call):
  range_4k / range_1m / range_64m   one read of 4 KiB / 1 MiB / 64 MiB with the index (path 0)
  range_1m_noindex                  one read of 1 MiB without the index (the parse over the whole stream, path 1)
  batch_1024 / batch_16384          uncompress_ranges_device with 1024 / 16384 random reads of 4 KiB, all indexed
  c_batch_1024 / c_batch_16384      the same batches, timing only the C call (its argument arrays and outputs are
                                    built before the clock starts): the difference to batch_* is the Python wrapper
Every call synchronises, so a host clock around it is the call's time; `kernel_ms` is the library's event time of its
decode launch (last_kernel_ms(1)) and `range_launches` its launch count.

    python tools/bench_range.py [--reps 20] [--warmup 3] [--out FILE] [--small]
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from snappy_jl_b200 import _abi, device, synth  # noqa: E402

FRAGMENT = 65536


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed(fn):
    """a case that times itself returns its own milliseconds"""
    t0 = time.perf_counter()
    own = fn()
    t = (time.perf_counter() - t0) * 1e3
    return (own if own is not None else t), device.last_kernel_ms(1)


def stats(ms):
    a = np.array(ms)
    return {"median_ms": round(float(np.median(a)), 4), "min_ms": round(float(a.min()), 4),
            "p90_ms": round(float(np.percentile(a, 90)), 4), "n": int(a.size)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--out", default=None)
    ap.add_argument("--small", action="store_true", help="tiny sizes (a rehearsal of the script, not a measurement)")
    a = ap.parse_args()
    info = {"card": card(), "torch": torch.__version__}
    print(json.dumps(info), flush=True)
    frags = 64 if a.small else 4096
    part = torch.from_numpy(synth.mix(frags, seed=a.seed)).cuda()
    raw = part.repeat(4)
    n = raw.numel()
    stream, index = device.compress_device(raw, want_index=True)
    stream = stream.clone()
    full_out = torch.empty(n, dtype=torch.uint8, device="cuda")
    rng = np.random.default_rng(a.seed)

    def single(length, with_index):
        out = torch.empty(length, dtype=torch.uint8, device="cuda")

        def run():
            off = int(rng.integers(0, n - length + 1))
            device.uncompress_range_device(stream, off, length, index=index if with_index else None, out=out)
        return run

    def batch(count, length=4096):
        def run():
            offs = [int(o) for o in rng.integers(0, n - length + 1, count)]
            outs, st = device.uncompress_ranges_device([stream] * count, offs, [length] * count, [index] * count)
            assert set(st) == {0}
        return run

    def c_batch(count, length=4096):
        outs = torch.empty(count * length, dtype=torch.uint8, device="cuda")
        ptrs = lambda v: (ctypes.c_void_p * count)(*v)
        sp, ip, op = ptrs([stream.data_ptr()] * count), ptrs([index.data_ptr()] * count), \
            ptrs([outs.data_ptr() + k * length for k in range(count)])
        in_lens, lens = (ctypes.c_size_t * count)(*[stream.numel()] * count), (ctypes.c_size_t * count)(*[length] * count)
        statuses = (ctypes.c_int * count)()
        cs = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

        def run():
            offs = (ctypes.c_uint64 * count)(*[int(o) for o in rng.integers(0, n - length + 1, count)])
            t0 = time.perf_counter()
            rc = _abi.lib().snappy_b200_uncompress_ranges_device(sp, in_lens, ip, offs, lens, op, count, statuses, cs)
            t = (time.perf_counter() - t0) * 1e3
            assert rc == 0 and set(statuses) == {0}
            return t
        return run

    def full():
        device.uncompress_device(stream, out=full_out, index=index)

    cases = [("range_4k", single(4096, True)), ("range_1m", single(1 << 20, True)),
             ("range_64m", single(min(64 << 20, n // 2), True)), ("range_1m_noindex", single(1 << 20, False)),
             ("batch_1024", batch(1024)), ("batch_16384", batch(16384)), ("c_batch_1024", c_batch(1024)),
             ("c_batch_16384", c_batch(16384))]
    # correctness of what is timed: seeded reads against the input
    for length in (4096, 1 << 20):
        off = int(rng.integers(0, n - length + 1))
        for idx in (index, None):
            got = device.uncompress_range_device(stream, off, length, index=idx)
            assert torch.equal(got, raw[off: off + length])
    offs = [int(o) for o in rng.integers(0, n - 4096 + 1, 1024)]
    outs, st = device.uncompress_ranges_device([stream] * 1024, offs, [4096] * 1024, [index] * 1024)
    assert set(st) == {0} and all(torch.equal(o, raw[f: f + 4096]) for o, f in zip(outs, offs))
    results = []
    for name, fn in cases:
        for _ in range(a.warmup):
            fn()
            full()
        tr, kr, tf, kf, launches = [], [], [], [], set()
        for k in range(a.reps):
            for which in ((0, 1) if k % 2 == 0 else (1, 0)):
                if which == 0:
                    t, km = timed(fn)
                    tr.append(t)
                    kr.append(km)
                    launches.add(device.last_launch_count(1))
                else:
                    t, km = timed(full)
                    tf.append(t)
                    kf.append(km)
        rec = {"case": name, "range": stats(tr), "range_kernel_ms": stats(kr), "full": stats(tf),
               "full_kernel_ms": stats(kf), "range_launches": sorted(launches),
               "full_over_range": round(float(np.median(tf) / np.median(tr)), 3)}
        print(json.dumps(rec), flush=True)
        results.append(rec)
    doc = dict(info, stream_bytes=int(stream.numel()), uncompressed_bytes=n, fragments=n // FRAGMENT, reps=a.reps,
               warmup=a.warmup, seed=a.seed, results=results)
    if a.out:
        with open(a.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
