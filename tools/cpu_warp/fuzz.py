"""Fuzz campaign for the kernel sources on the CPU warp (TEST INFRASTRUCTURE; minutes of CPU, not part of pytest).

    python tools/cpu_warp/fuzz.py [seed] [count] [legs]

Generates `count` inputs (small alphabets, periodic data with mutations, runs, dictionary words, concatenations,
boundary sizes), then runs: the window compress kernel (shared / global tables, rules 0/1/2, three ring sizes), the
step-wise chain kernel, the indexed decoder, the page kernels, and the index-free parse on the Snappy.jl and Google
snappy streams of every input.  Then the corruption corpus's mutations (tests/test_decode_corruption.py: random and
boundary faults, truncations, header lies, two faults, accepted quirks) of the multi-fragment streams (Snappy.jl's and
Google snappy's in turn) go through the index-free decode chain (run_decode_parsed.cpp: parse, tiles, bounded serial
walk; parse chunks of 512 B, 1 KiB and 4 KiB, and without clean cuts) and the page decoder, against the oracle's status
and bytes.  `legs`: comma-separated subset of "compress,decode,pages,parse,corrupt" (default: all).  Any mismatch
against the oracle / the sequential walk is printed; exit status 1.
Last run of every leg but "corrupt" (seed 12345, 201 inputs, ~15 min on 8 cores): no mismatch anywhere.
Last run of "corrupt" (seed 12345, 201 inputs: 5028 mutated streams, ~5 min on 8 cores): no mismatch anywhere."""
import concurrent.futures
import os
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "oracle"))


def inputs(seed, count):
    rng = np.random.default_rng(seed)

    def alpha(n):
        return rng.integers(0, int(rng.choice([1, 2, 3, 4, 16, 256])), n, dtype=np.uint8).tobytes()

    def period(n):
        p = int(rng.integers(1, 5000))
        a = np.tile(rng.integers(0, 256, p, dtype=np.uint8), n // p + 1)[:n].copy()
        m = int(rng.integers(0, max(1, n // 200)))
        if m and n:
            a[rng.integers(0, n, m)] = rng.integers(0, 256, m, dtype=np.uint8)
        return a.tobytes()

    def runs(n):
        out = bytearray()
        while len(out) < n:
            out += bytes([int(rng.integers(0, 256))]) * int(rng.integers(1, 400))
            if rng.random() < 0.3:
                out += rng.integers(0, 256, int(rng.integers(1, 100)), dtype=np.uint8).tobytes()
        return bytes(out[:n])

    def words(n):
        ws = [rng.integers(0, 256, int(rng.integers(1, 17)), dtype=np.uint8).tobytes() for _ in range(int(rng.integers(2, 200)))]
        out = bytearray()
        while len(out) < n:
            out += ws[int(rng.integers(0, len(ws)))]
        return bytes(out[:n])

    gens = [alpha, period, runs, words]
    sizes = [0, 1, 14, 15, 16, 17, 31, 32, 33, 63, 64, 65, 511, 512, 513, 1023, 1024, 1025, 2047, 2048, 2049, 4095, 4096,
             4097, 65535, 65536, 65537, 65536 + 15, 65536 + 16, 131072, 131073]
    for i, n in enumerate(sizes):
        yield gens[i % 4](n)
    for _ in range(max(0, count - len(sizes))):
        parts, tot = [], int(rng.integers(1, 200000))
        while tot > 0:
            n = min(tot, int(rng.integers(1, 70000)))
            parts.append(gens[int(rng.integers(0, 4))](n))
            tot -= n
        yield b"".join(parts)


def main():
    import pyarrow as pa
    import pyoracle
    seed = int(sys.argv[1]) if len(sys.argv) > 1 else 12345
    count = int(sys.argv[2]) if len(sys.argv) > 2 else 201
    legs = set(sys.argv[3].split(",")) if len(sys.argv) > 3 else {"compress", "decode", "pages", "parse", "corrupt"}
    d = tempfile.mkdtemp(prefix="cpu_warp_fuzz_")
    obj = os.path.join(d, "oracle.o")
    subprocess.check_call(["gcc", "-O2", "-c", "-o", obj, os.path.join(ROOT, "oracle", "snappy_oracle.c")])
    exe = {}
    for name, src in (("window", "run_window_kernel"), ("decode", "run_decode_kernel"), ("pages", "run_pages_kernel"),
                      ("parse", "run_parse_kernel"), ("decode_parsed", "run_decode_parsed")):
        exe[name] = os.path.join(d, name)
        subprocess.check_call(["g++", "-O1", "-std=c++17", "-DSB200_CPU_EMU", "-DSB200_EXPERIMENTS", "-I" + os.path.join(ROOT, "tools", "cpu_warp"), "-o",
                               exe[name], os.path.join(ROOT, "tools", "cpu_warp", "%s.cpp" % src), obj])
    raw, streams = [], []
    codec = pa.Codec("snappy")
    for i, b in enumerate(inputs(seed, count)):
        p = os.path.join(d, "f%03d.bin" % i)
        open(p, "wb").write(b)
        raw.append(p)
        for tag, comp in (("jl", pyoracle.compress(b)), ("g", codec.compress(b, asbytes=True) if b else pyoracle.compress(b))):
            q = os.path.join(d, "f%03d.%s.sn" % (i, tag))
            open(q, "wb").write(comp)
            streams.append(q)
    bad = 0

    def go(what, cmd, env=None, files=None):
        """`files` (appended to cmd) are split over the CPU's cores"""
        nonlocal bad
        groups = [files[k::os.cpu_count() or 1] for k in range(os.cpu_count() or 1)] if files else [[]]
        with concurrent.futures.ThreadPoolExecutor(len(groups)) as ex:
            runs = list(ex.map(lambda g: subprocess.run(cmd + g, env=dict(os.environ, **(env or {})), capture_output=True,
                                                        text=True), [g for g in groups if g or not files]))
        lines = [l for p in runs for l in p.stdout.splitlines()]
        wrong = [l for l in lines if "0 mismatches" not in l and "no body" not in l and "header rejected" not in l]
        failed = any(p.returncode != 0 for p in runs) or bool(wrong)
        print("%-44s %s (%d lines)" % (what, "MISMATCH" if failed else "ok", len(lines)), flush=True)
        for l in wrong[:5] + [l for p in runs for l in p.stderr.splitlines()][:5]:
            print("   ", l)
        bad += failed

    if "compress" in legs:
        for table, rules, ring in (("smem", 0, 1024), ("smem", 0, 2048), ("smem", 2, 4096), ("global", 0, 1024),
                                   ("global", 1, 2048), ("global", 2, 1024)):
            go("window %s rules %d ring %d" % (table, rules, ring), [exe["window"]] + raw,
               {"TABLE": table, "RULES": str(rules), "RING": str(ring)})
        go("window + slowcont", [exe["window"]] + raw, {"SLOWCONT": "1"})
        go("chain kernel", [exe["window"]] + raw, {"KERNEL": "chain"})
    if "decode" in legs:
        go("indexed decoder", [exe["decode"], "indexed"] + raw)
        go("exact decoder on the streams", [exe["decode"], "exact"] + streams)
    if "pages" in legs:
        for rules in (0, 2):
            go("pages rules %d" % rules, [exe["pages"]] + raw[3:40], {"RULES": str(rules)})
    if "parse" in legs:
        go("index-free parse", [exe["parse"]] + streams)
    if "corrupt" in legs:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from test_decode_corruption import mutations
        rng = np.random.default_rng(seed)
        mutated = []
        for i, s in enumerate(streams):
            data = open(s, "rb").read()
            if i % 2 != (i // 2) % 2 or pyoracle.uncompressed_length(data) <= 65536:
                continue  # multi-fragment streams only, Snappy.jl's and Google snappy's in turn
            for k, (name, m) in enumerate(mutations(pyoracle, rng, os.path.basename(s), data, range(4))):
                q = os.path.join(d, "m%05d_%s" % (len(mutated), name.replace("/", "__")))
                open(q, "wb").write(m)
                mutated.append(q)
        go("corrupt streams, parsed decode", [exe["decode_parsed"], "parsed"], files=mutated)
        for env in ({"PSHIFT": "9"}, {"PSHIFT": "12"}, {"CLEAN_CUTS": "0"}):
            go("corrupt streams, parsed decode %s" % env, [exe["decode_parsed"], "parsed"], env, files=mutated[::3])
        go("corrupt streams, pages", [exe["decode_parsed"], "pages"], files=mutated)
    print("inputs in", d)
    return 1 if bad else 0


if __name__ == "__main__":
    sys.exit(main())
