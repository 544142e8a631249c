"""GPU: validation (snappy_b200_validate_*) against uncompress, in the same run, alternating the two.

Cases (seeded inputs):
  stream1g_index     1 GiB mix stream with its side index: validate_device vs uncompress_device
  stream1g_noindex   the same stream without the index (the parse decides)
  stream1g_corrupt   the same stream with one byte flipped near the end, without the index
  pages              2^20 pages of 4 KiB: validate_batched_device vs uncompress_batched_device
  host_pinned        the 1 GiB stream from pinned host memory: validate_compressed_buffer vs uncompress
  host_pageable      the same from pageable host memory
Every call synchronises, so a host clock around it is the call's time.  Inputs are larger than the 126 MB L2.
The 1 GiB input is 256 MiB of synth.mix repeated 4 times and the pages are 64 MiB of it repeated 64 times (the codec
works on independent 64 KiB fragments / pages, so the repetition changes no work; it keeps the set-up short).

    python tools/bench_validate.py [--reps 25] [--warmup 3] [--out FILE]
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

import snappy_jl_b200 as Snappy  # noqa: E402
from snappy_jl_b200 import _abi, device, synth  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


def timed(fn):
    t0 = time.perf_counter()
    r = fn()
    return (time.perf_counter() - t0) * 1e3, r


def stats(ms):
    a = np.array(ms)
    return {"median_ms": round(float(np.median(a)), 3), "min_ms": round(float(a.min()), 3),
            "p90_ms": round(float(np.percentile(a, 90)), 3), "max_ms": round(float(a.max()), 3), "n": int(a.size)}


def ab(name, validate, uncompress, reps, warmup, nbytes):
    """alternate the two calls: warm-up, then `reps` pairs; returns the result record"""
    for _ in range(warmup):
        validate()
        uncompress()
    tv, tu, rv, ru = [], [], None, None
    for k in range(reps):
        for which in ((0, 1) if k % 2 == 0 else (1, 0)):
            if which == 0:
                t, rv = timed(validate)
                tv.append(t)
            else:
                t, ru = timed(uncompress)
                tu.append(t)
    v, u = stats(tv), stats(tu)
    rec = {"case": name, "bytes": int(nbytes), "validate": v, "uncompress": u,
           "speedup_median": round(u["median_ms"] / v["median_ms"], 2), "validate_result": rv, "uncompress_result": ru}
    print(json.dumps(rec), flush=True)
    return rec


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=25)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--out", default=None)
    ap.add_argument("--small", action="store_true", help="tiny sizes (a rehearsal of the script, not a measurement)")
    args = ap.parse_args()
    assert torch.cuda.is_available(), "bench_validate needs a GPU"
    torch.cuda.set_device(0)
    info = {"card": card(), "torch": torch.__version__, "reps": args.reps, "warmup": args.warmup, "seed": args.seed}
    print(json.dumps(info), flush=True)
    lib = _abi.lib()
    results = []
    path = lambda: lib.snappy_b200_get_option(b"last_decode_path")

    # ---- the 1 GiB stream
    base_frags, reps1g = (64, 2) if args.small else (4096, 4)
    raw = torch.from_numpy(np.tile(synth.mix(base_frags, seed=args.seed), reps1g)).cuda()
    stream, index = device.compress_device(raw, want_index=True)
    stream = stream.clone()
    out = torch.empty_like(raw)
    n = raw.numel()

    def dv(s, idx):
        def f():
            st, claimed = device.validate_device(s, index=idx)
            return [st, claimed, path()]
        return f

    def du(s, idx):
        def f():
            try:
                device.uncompress_device(s, out=out, index=idx)
                return [0, path()]
            except Snappy.SnappyError as e:
                return [e.status, path()]
        return f

    results.append(ab("stream1g_index", dv(stream, index), du(stream, index), args.reps, args.warmup, n))
    results.append(ab("stream1g_noindex", dv(stream, None), du(stream, None), args.reps, args.warmup, n))
    assert torch.equal(out, raw), "uncompress of the 1 GiB stream differs from its input"
    for k in range(64):  # the first byte near the end whose flip makes uncompress fail (a literal byte would not)
        bad = stream.clone()
        bad[bad.numel() - 1000 - 37 * k] ^= 0x5A
        if du(bad, None)()[0] != 0:
            break
    results.append(ab("stream1g_corrupt", dv(bad, None), du(bad, None), args.reps, args.warmup, n))
    del bad

    # ---- host calls on the same stream
    h_stream = stream.cpu().numpy()
    pinned_in = torch.empty(h_stream.size, dtype=torch.uint8, pin_memory=True)
    pinned_in.numpy()[:] = h_stream
    pinned_out = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    pageable_out = np.empty(n, dtype=np.uint8)
    pageable_out[:] = 0

    def hv(a):
        return lambda: Snappy.validate(a)

    def hu(a, o):
        def f():
            ol = ctypes.c_size_t(o.size)
            return lib.snappy_b200_uncompress(ctypes.c_void_p(a.ctypes.data), a.size, ctypes.c_void_p(o.ctypes.data),
                                              ctypes.byref(ol))
        return f

    results.append(ab("host_pinned", hv(pinned_in.numpy()), hu(pinned_in.numpy(), pinned_out.numpy()), args.reps,
                      args.warmup, n))
    results.append(ab("host_pageable", hv(h_stream), hu(h_stream, pageable_out), args.reps, args.warmup, n))
    assert np.array_equal(pageable_out, raw.cpu().numpy())
    del pinned_in, pinned_out, pageable_out, h_stream, stream, index, out, raw
    torch.cuda.empty_cache()

    # ---- 2^20 pages of 4 KiB
    count = (1 << 12) if args.small else (1 << 20)
    page = 4096
    block = synth.pages(min(count, 1 << 14), page, seed=args.seed).reshape(-1)
    flat = torch.from_numpy(np.tile(block, count * page // block.size)).cuda()
    offs = torch.arange(count, dtype=torch.int64, device="cuda") * page
    sizes = torch.full((count,), page, dtype=torch.int32, device="cuda")
    cdata, coffs, csizes = device.compress_batched_device(flat, offs, sizes)
    back = torch.empty_like(flat)

    def pv():
        st, claimed = device.validate_batched_device(cdata, coffs, csizes)
        return [int(st.abs().sum().item()), int(claimed.to(torch.int64).sum().item())]

    def pu():
        got, st = device.uncompress_batched_device(cdata, coffs, csizes, back, offs, sizes)
        return [int(st.abs().sum().item()), int(got.to(torch.int64).sum().item())]

    results.append(ab("pages_4k", pv, pu, args.reps, args.warmup, flat.numel()))
    assert torch.equal(back, flat), "batched uncompress differs from its input"
    doc = {"info": info, "results": results}
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
