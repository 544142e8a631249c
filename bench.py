#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric on BASELINE.json's configs.

Default (`--config 2`): a step = compress the 1 GiB synthetic mixed-compressibility buffer (16384 x 64 KiB fragments,
BASELINE config 2) into one Snappy stream, then uncompress it.
  value : uncompressed GB / (t_compress + t_uncompress), inputs resident in HBM, CUDA-event timed, max over ranks;
          compress_gbps / uncompress_gbps are the two directions separately.
  e2e   : the same through the reference-facing host-buffer C ABI (snappy_b200_compress / snappy_b200_uncompress)
          from pinned host memory, H2D + D2H inside the timed region; e2e_pageable: from ordinary (pageable) arrays,
          which is what the reference API hands over (src/Snappy.jl:25,48 allocate fresh Vector{UInt8}).
  roofline : the dominant kernel's (N + C) algorithmic bytes / its CUDA-event duration vs measured HBM, its measured
          DRAM traffic and its share of the SMs' issue slots (profiles/traffic.json holds the ncu captures).
  cpu_baseline : the oracle (C restatement of Snappy.jl) on this box's host cores.
The other configs run in the same process and are nested under "configs" (one JSON line in total, the headline keys
stay those of config 2); `--config 3|4|5` prints the full line of that config instead:
  3  arbitrary-stream uncompress: the 1 GiB stream the ORACLE produced (no side index), index-free parse + decode
  4  2^20 independent 4 KiB pages, one stream per page, batched API
  5  8 GiB source-code-like corpus as 8 streams x 1 GiB (one stream cannot exceed 2^32 - 1 bytes,
     src/Snappy.jl:21), the SAME 8 streams sharded over 1/2/4/8 GPUs: strong scaling
`--steps K` is the number of timed steps of every leg: the headline config, the nested ones and both e2e legs.
`--dump-outputs DIR` (config 2) writes what the last timed step returned to its caller as DIR/<name>.npy, so that two
builds run with the same arguments (hence the same inputs) can be compared output for output.
`--impl reference` times the oracle alone (the reference is Julia and cannot run in this image).
N > 1 (torchrun), config 2: weak scaling -- N streams of 1 GiB, every stream sharded over the N ranks along
whole-fragment boundaries; sizes by ncclAllGather on the compute stream, fragments stored straight into the owner's
buffer over NVLink (snappy_b200_comm_*, the library's own exchange; torch.distributed carries the NCCL id only).
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True  # the tree may be read-only: a benchmark run leaves nothing in it

import numpy as np  # noqa: E402

GIB = 1 << 30
FRAGMENT = 65536
METRIC = "compress+uncompress GB/s (1 GiB synth mixed buffer; uncompressed bytes / (t_compress + t_uncompress))"
METRICS = {
    2: METRIC,
    3: "arbitrary-stream uncompress GB/s (1 GiB oracle-produced stream, no side index; uncompressed bytes / t)",
    4: "batched pages compress+uncompress GB/s (2^20 x 4 KiB pages, one stream per page; bytes / (t_c + t_u))",
    5: "sharded corpus compress+uncompress GB/s (8 x 1 GiB source-like streams over N GPUs; bytes / (t_c + t_u))",
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5])
    ap.add_argument("--fragments", type=int, default=16384, help="fragments per GPU / per stream (16384 = 1 GiB)")
    ap.add_argument("--pages", type=int, default=1 << 20, help="config 4: number of 4 KiB pages")
    ap.add_argument("--streams", type=int, default=8, help="config 5: number of streams")
    ap.add_argument("--seed", type=int, default=2026)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="config 2 only: skip the nested legs of configs 3, 4, 5")
    ap.add_argument("--extra-steps", type=int, default=None, help="timed steps of each nested config leg "
                                                                  "(default: --steps)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="config 2: write the last timed step's outputs to DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.extra_steps is None:
        args.extra_steps = args.steps
    if args.dump_outputs and (args.config != 2 or args.impl != "b200"):
        ap.error("--dump-outputs writes the outputs of config 2 of the b200 arm")
    return args


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


def gpu_local_cpus(dev_index):
    """CPUs on the NUMA node the GPU's PCIe root hangs off (sysfs), or None."""
    try:
        import torch
        pr = torch.cuda.get_device_properties(dev_index)
        bdf = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        txt = open("/sys/bus/pci/devices/%s/local_cpulist" % bdf).read().strip()
        cpus = set()
        for part in txt.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        return cpus or None
    except Exception:
        return None


class gpu_local_node:
    """Host buffers of the e2e legs are allocated while this thread is confined to the GPU-local CPUs, so that first
    touch puts them on the GPU's NUMA node (a remote node costs ~30 % of PCIe throughput: 69 vs 52 ms per step,
    bimodal from run to run).  The affinity is restored on exit: the CPU baseline uses every core."""

    def __init__(self, dev_index):
        self.dev, self.old, self.local = dev_index, None, False

    def __enter__(self):
        try:
            cpus = gpu_local_cpus(self.dev)
            old = os.sched_getaffinity(0)
            if cpus and (cpus & old) and (cpus & old) != old:
                os.sched_setaffinity(0, cpus & old)
                self.old = old
            self.local = bool(cpus and (cpus & old))
        except Exception:
            self.old = None
        return self

    def __exit__(self, *exc):
        if self.old is not None:
            try:
                os.sched_setaffinity(0, self.old)
            except Exception:
                pass
        return False


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.FIELDS, "--format=csv,noheader,nounits",
                 "-lms", "100"], stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.proc is None:
            return out
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        try:
            for line in open(self.path):
                p = [x.strip() for x in line.split(",")]
                if len(p) < 9:
                    continue
                try:
                    sm.append(float(p[1]))
                    mx.append(float(p[2]))
                except ValueError:
                    continue
                for nm, v in zip(names, p[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(nm)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            out["sm_mhz"] = float(np.median(sm))
            out["sm_max_mhz"] = float(max(mx))
        out["reasons"] = sorted(reasons)
        return out


# ------------------------------------------------------------------------------------------
# synthetic inputs.  Generating them is the slowest part of a run (numpy, ~26 s per GiB of mix, ~43 s per GiB of
# source-like text on one core), so the pieces are made by worker processes side by side into shared memory.
# ------------------------------------------------------------------------------------------
def make_input(nfrag, seed):
    from snappy_jl_b200 import synth
    return synth.mix(nfrag, seed=seed)


PIECE_FRAGS = 2048  # 128 MiB: shard boundaries at 1, 2, 4 and 8 ranks fall on piece boundaries of a 1 GiB stream


def piece_seed(kind, seed, stream, piece):
    return seed + {"mix": 0, "source": 500000, "pages": 700000}[kind] + 1000 * stream + piece


def Generator(workers):
    from snappy_jl_b200 import synth
    return synth.ParallelGenerator(workers)


# ------------------------------------------------------------------------------------------
# CPU legs (oracle): cpu_baseline of the b200 arm, and the whole --impl reference arm
# ------------------------------------------------------------------------------------------
def _oracle():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pyoracle
    pyoracle.build()
    return pyoracle


def oracle_roundtrip_threads(raw, threads):
    """T host threads over T independent buffers (the Threads.@threads analogue of SURVEY 8(d)):
    each compresses and uncompresses its own slice as an independent stream.  Returns seconds
    (compress, uncompress).  ctypes releases the GIL, so the threads run in parallel."""
    pyoracle = _oracle()
    nfrag = (raw.size + FRAGMENT - 1) // FRAGMENT
    per = (nfrag + threads - 1) // threads
    slices = [raw[i * per * FRAGMENT: min((i + 1) * per * FRAGMENT, raw.size)] for i in range(threads)]
    slices = [s for s in slices if s.size]
    comp = [None] * len(slices)
    back = [None] * len(slices)

    def run(fn):
        ts = [threading.Thread(target=fn, args=(i,)) for i in range(len(slices))]
        t0 = time.perf_counter()
        for t in ts:
            t.start()
        for t in ts:
            t.join()
        return time.perf_counter() - t0

    def c(i):
        comp[i] = pyoracle.compress_np(slices[i])

    def u(i):
        back[i] = pyoracle.uncompress_np(comp[i])

    tc = run(c)
    tu = run(u)
    assert all(np.array_equal(b, s) for b, s in zip(back, slices)), "oracle round trip failed"
    return tc, tu, sum(int(x.size) for x in comp)


def oracle_stream_parallel(raw, threads):
    """The oracle's stream of `raw` (ONE stream, src/Snappy.jl:20-36), its fragments compressed by T threads:
    fragments are independent (table reset per fragment, :30), so runs of fragments concatenate to exactly the
    bytes sjo_compress produces (tests/test_oracle.py::test_fragment_api_consistent)."""
    pyoracle = _oracle()
    nfrag = (raw.size + FRAGMENT - 1) // FRAGMENT
    per = (nfrag + threads - 1) // threads
    parts = [None] * threads

    def work(i):
        f0 = i * per
        nf = min(per, nfrag - f0)
        if nf > 0:
            parts[i] = pyoracle.compress_fragments(raw, raw.size, f0, nf)[0]

    ts = [threading.Thread(target=work, args=(i,)) for i in range(threads)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    hdr = np.frombuffer(pyoracle.encode32(raw.size), dtype=np.uint8)
    return np.concatenate([hdr] + [p for p in parts if p is not None])


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    cores = os.cpu_count() or 1
    # bounded sample: 256 MiB of the same workload per step (the full size x (W+K) steps would take minutes)
    nfrag = min(args.fragments, 4096)
    if args.config == 5:
        from snappy_jl_b200 import synth
        raw = synth.source_like(nfrag * FRAGMENT, seed=piece_seed("source", args.seed, 0, 0))
        what = "source-like corpus"
    elif args.config == 4:
        from snappy_jl_b200 import synth
        raw = synth.mix(nfrag, seed=piece_seed("pages", args.seed, 0, 0))
        what = "page mix"
    else:
        raw = make_input(nfrag, args.seed)
        what = "mix"
    threads = cores
    if args.config == 4:
        # pages: every 4 KiB page is its own stream; T threads each walk their share of the pages
        pyoracle = _oracle()
        pages = raw.reshape(-1, 4096)

        def roundtrip():
            comp = [None] * len(pages)

            def c(t):
                for i in range(t, len(pages), threads):
                    comp[i] = pyoracle.compress_np(pages[i])

            def u(t):
                for i in range(t, len(pages), threads):
                    pyoracle.uncompress_np(comp[i])

            out = []
            for fn in (c, u):
                ts = [threading.Thread(target=fn, args=(t,)) for t in range(threads)]
                t0 = time.perf_counter()
                for t in ts:
                    t.start()
                for t in ts:
                    t.join()
                out.append(time.perf_counter() - t0)
            return out[0], out[1], 0
    else:
        def roundtrip():
            return oracle_roundtrip_threads(raw, threads)
    for _ in range(args.warmup):
        roundtrip()
    tc = tu = 0.0
    for _ in range(args.steps):
        a, b, _ = roundtrip()
        tc += a
        tu += b
    n = raw.size * args.steps
    if args.config == 3:  # uncompress only
        value, ms = n / tu / 1e9, tu / args.steps * 1e3
    else:
        value, ms = n / (tc + tu) / 1e9, (tc + tu) / args.steps * 1e3
    sample = "%d MiB of the %s (seed %d) per step, %d independent buffers on %d threads" % (
        raw.size >> 20, what, args.seed, threads, threads)
    line = {
        "impl": "reference", "metric": METRICS[args.config], "value": value, "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms,
        "higher_is_better": True, "scaling": "strong" if args.config == 5 else "weak", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic",
        "compress_gbps": n / tc / 1e9, "uncompress_gbps": n / tu / 1e9,
        "config": {"workload": workload_name(args.config, args) + "; reference arm runs a bounded sample",
                   "sample": sample},
        "cpu_baseline": {"value": value, "unit": "GB/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "reference is pure Julia (no Julia in this image): this is oracle/snappy_oracle.c, the C "
                "restatement of Snappy.jl, on host cores",
    }
    print(json.dumps(line), flush=True)
    return 0


def workload_name(config, args):
    if config == 2:
        return ("1 GiB synthetic mixed-compressibility buffer (%d x 64 KiB fragments) per GPU, compress then "
                "uncompress" % args.fragments)
    if config == 3:
        return ("arbitrary-stream uncompress: the %d-fragment mix compressed by the ORACLE into one stream, handed "
                "over with no side index (index-free parse + decode)" % args.fragments)
    if config == 4:
        return "%d independent 4 KiB pages (cut from the mix generator), one stream per page, batched API" % args.pages
    return ("%d streams x %d fragments of source-code-like text (%.1f GiB), the same streams at every N, each sharded "
            "over the N GPUs along whole-fragment boundaries" % (args.streams, args.fragments,
                                                                args.streams * args.fragments * FRAGMENT / GIB))


# ------------------------------------------------------------------------------------------
# oracle spot checks of what was timed ("bit-exact" is asserted, not assumed)
# ------------------------------------------------------------------------------------------
def check_fragments_vs_oracle(raw_of, total_len, stream_np_of, index_np, count, seed):
    """`count` sampled fragments of a stream: the GPU's bytes for the fragment (cut with the side index) must equal
    the oracle's compress of the same 64 KiB with the table sized from the stream's TOTAL length.
    raw_of(lo, hi) / stream_np_of(lo, hi) return numpy slices."""
    pyoracle = _oracle()
    nfrag = (total_len + FRAGMENT - 1) // FRAGMENT
    rng = np.random.default_rng(seed)
    picks = sorted(set([0, nfrag - 1] + [int(x) for x in rng.integers(0, nfrag, max(count - 2, 0))]))
    for f in picks:
        lo, hi = f * FRAGMENT, min((f + 1) * FRAGMENT, total_len)
        want = pyoracle.compress_one_fragment(np.ascontiguousarray(raw_of(lo, hi)), total_len)
        got = stream_np_of(int(index_np[f]), int(index_np[f + 1]))
        if got.size != want.size or not np.array_equal(got, want):
            raise AssertionError("fragment %d differs from the oracle (%d vs %d bytes)" % (f, got.size, want.size))
    return len(picks)


# ------------------------------------------------------------------------------------------
def run_b200(args):
    import torch
    import torch.distributed as dist
    import snappy_jl_b200 as Snappy
    from snappy_jl_b200 import device, multi

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1
    cores = os.cpu_count() or 1
    ctx = {"torch": torch, "dist": dist, "Snappy": Snappy, "device": device, "multi": multi, "world": world,
           "rank": rank, "local": local, "dev": dev, "cores": cores, "args": args}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    ctx["barrier"] = barrier

    # ---- the library's communicator (all configs at N > 1, config 5 at every N) ---------------------------
    comm, comm_note = None, None
    try:
        comm = multi.LibComm()
        # a first tiny collective maps the arenas (cudaIpc) now, where a failure is still harmless
        one = torch.zeros(FRAGMENT, dtype=torch.uint8, device=dev)
        comm.compress([one], [world * FRAGMENT])
    except Exception as e:  # e.g. cudaIpc not permitted on this box: the torch.distributed assembly still works
        comm_note = "snappy_b200_comm unavailable (%s): torch.distributed all-to-all assembly" % str(e)[:160]
    if world > 1:
        flag = torch.tensor([1 if comm is not None else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0 and comm is not None:
            comm.close()
            comm = None
            comm_note = comm_note or "snappy_b200_comm unavailable on another rank"
    ctx["comm"], ctx["comm_note"] = comm, comm_note

    # ---- inputs: every config's pieces are generated side by side ------------------------------------------
    want = [args.config] if (args.config != 2 or args.no_extra) else [2, 3, 4, 5]
    if world > 1:
        want = [c for c in want if c in (2, 5)] if args.config == 2 else want
    gen = Generator(max(1, cores // world))
    plan = {}
    t_gen = time.perf_counter()
    if 2 in want or 3 in want:
        if world == 1:
            plan["mix"] = gen.add("mixwhole", args.seed, args.fragments)
        elif 2 in want:
            per = args.fragments // world
            plan["mix_shards"] = [gen.add("mixwhole", args.seed + 1000 * s + rank, per) for s in range(world)]
    if 4 in want:
        per_frag = FRAGMENT // 4096
        need = (args.pages + per_frag - 1) // per_frag
        # N > 1: the pages are split over the ranks (independent streams: no exchange at all)
        mine = need // world + (1 if rank < need % world else 0)
        first = rank * (need // world) + min(rank, need % world)
        plan["pages"] = []
        f = first
        while f < first + mine:
            k = min(PIECE_FRAGS, first + mine - f)
            plan["pages"].append(gen.add("pages", piece_seed("pages", args.seed, 0, f), k))
            f += k
    if 5 in want:
        S = args.streams
        pieces = (args.fragments + PIECE_FRAGS - 1) // PIECE_FRAGS
        plan["source"] = {}
        for s in range(S):
            lo, hi = multi.shard_bounds(args.fragments * FRAGMENT, world)[rank]
            f = lo // FRAGMENT
            while f < hi // FRAGMENT:
                p = f // PIECE_FRAGS
                k = min((p + 1) * PIECE_FRAGS, hi // FRAGMENT) - f
                # a run that starts inside a piece regenerates the piece and cuts it (never at 1, 2, 4, 8 ranks)
                assert f % PIECE_FRAGS == 0 or pieces == 1, "shard boundary inside a generator piece"
                plan["source"].setdefault(s, []).append(gen.add("source", piece_seed("source", args.seed, s, p), k))
                f += k
    gen.run()
    ctx["gen"], ctx["plan"] = gen, plan
    ctx["gen_seconds"] = time.perf_counter() - t_gen

    results = {}
    try:
        for cfg in want:
            results[cfg] = {2: config2, 3: config3, 4: config4, 5: config5}[cfg](ctx, nested=(cfg != args.config))
    finally:
        gen.close()
    if rank == 0:
        line = results[args.config]
        extra = {("c%d" % c): results[c] for c in want if c != args.config}
        if extra:
            line["configs"] = extra
        line["input_generation_s"] = ctx["gen_seconds"]
        if comm_note:
            line["comm_note"] = comm_note
        print(json.dumps(line), flush=True)
    if comm is not None:
        comm.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def timed_loop(ctx, steps, warmup, do_c, do_u, after_c=None):
    """W untimed + K timed steps; CUDA events on the current stream, barrier + synchronize around every step, max
    over ranks.  Returns (t_c ms, t_u ms, last results) summed over the K steps."""
    torch, dist, world, dev = ctx["torch"], ctx["dist"], ctx["world"], ctx["dev"]
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    rc = ru = None
    for _ in range(warmup):
        rc = do_c() if do_c else None
        ru = do_u(rc) if do_u else None
    tc = tu = 0.0
    for _ in range(steps):
        ctx["barrier"]()
        ev[0].record()
        rc = do_c() if do_c else rc
        ev[1].record()
        if after_c:
            after_c()
        ru = do_u(rc) if do_u else None
        ev[2].record()
        ctx["barrier"]()
        a, b = ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])
        if world > 1:
            t = torch.tensor([a, b], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            a, b = float(t[0]), float(t[1])
        tc += a
        tu += b
    return tc, tu, rc, ru


DUMP_BYTES = 60 * 10 ** 6  # array data of one --dump-outputs run; with the .npy headers it stays under 64 MB


def dump_outputs(where, arrays, seed):
    """Writes every tensor of `arrays` (name -> 1-D tensor) as where/<name>.npy: float32 when its integers fit one
    exactly (up to 16 bits), float64 otherwise.  Each gets an equal share of DUMP_BYTES; a longer one is replaced by
    its elements at sorted positions drawn with `seed`, so the same positions of equally long outputs are compared."""
    import torch
    os.makedirs(where, exist_ok=True)
    keep = DUMP_BYTES // (8 * len(arrays))
    for name, t in arrays.items():
        if t.numel() > keep:
            pos = np.sort(np.random.default_rng(seed).integers(0, t.numel(), keep))
            t = t[torch.from_numpy(pos).to(t.device)]
        a = t.cpu().numpy()
        np.save(os.path.join(where, name + ".npy"), a.astype(np.float32 if a.dtype.itemsize <= 2 else np.float64))


def traffic_entry(kernel):
    try:
        with open(os.path.join(ROOT, "profiles", "traffic.json")) as f:
            return json.load(f).get(kernel)
    except Exception:
        return None


def roofline_of(kernel, k_ms, alg_bytes, sm_mhz=None, sms=148, note=None, scale_capture=True):
    peak, peak_src = measured_peak()
    achieved = (alg_bytes / (k_ms / 1e3) / 1e9) if k_ms > 0 else 0.0
    r = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak if peak else None,
         "traffic": None, "kernel": kernel, "kernel_ms": k_ms, "algorithmic_bytes": alg_bytes, "peak_source": peak_src}
    ent = traffic_entry(kernel) if scale_capture else None  # the captures are of the 1 GiB mix: other workloads get none
    if isinstance(ent, (int, float)):
        r["traffic"] = ent
    if isinstance(ent, dict):
        # DRAM bytes per launch of this kernel on the 1 GiB mix, from the committed ncu capture (profiles/)
        r["traffic"] = ent.get("dram_bytes_per_launch", ent.get("per_launch_estimate"))
        r["traffic_source"] = ent.get("source", ent.get("note"))
        inst = ent.get("warp_instructions_per_launch")
        if inst and k_ms > 0:
            mhz = sm_mhz or 1965.0
            slots = k_ms / 1e3 * mhz * 1e6 * sms * 4  # one warp instruction per SM sub-partition and cycle
            r["issue"] = {"inst": inst, "slots": slots, "frac": inst / slots,
                          "note": "inst = smsp__inst_executed.sum of the capture; slots = kernel time x SM clock x "
                                  "%d SMs x 4 schedulers" % sms}
    if note:
        r["note"] = note
    return r


# ------------------------------------------------------------------------------------------ config 2
def config2(ctx, nested=False):
    torch, dist, Snappy, device, multi = ctx["torch"], ctx["dist"], ctx["Snappy"], ctx["device"], ctx["multi"]
    world, rank, local, dev, args, comm = ctx["world"], ctx["rank"], ctx["local"], ctx["dev"], ctx["args"], ctx["comm"]
    gen, plan = ctx["gen"], ctx["plan"]
    nfrag = args.fragments
    n = nfrag * FRAGMENT
    launches = 0
    if world == 1:
        raw = gen.view(*plan["mix"])
        with gpu_local_node(local):
            host_in = torch.from_numpy(raw.copy()).pin_memory()
        d_in = host_in.to(dev, non_blocking=True)
        torch.cuda.synchronize()
        cap = Snappy.maxlength_compressed(n)
        d_out = torch.empty(cap, dtype=torch.uint8, device=dev)
        d_back = torch.empty(n, dtype=torch.uint8, device=dev)

        def do_c():
            return device.compress_device(d_in, out=d_out, want_index=True)

        def do_u(rc):
            return device.uncompress_device(rc[0], out=d_back, index=rc[1], claimed=n)
    else:
        # stream s = concat over ranks r of mix(nfrag/world, seed(s, r)); this rank holds run r = rank of every s
        per = nfrag // world
        shards = [torch.from_numpy(gen.view(*p).copy()).to(dev) for p in plan["mix_shards"]]
        totals = [per * world * FRAGMENT] * world
        n = totals[0]
        codec = multi.CudaCodec()
        if comm is not None:
            outs = [torch.empty(per * FRAGMENT, dtype=torch.uint8, device=dev) for _ in range(world)]

            def do_c():
                return comm.compress(shards, totals)

            def do_u(rc):
                return comm.uncompress(rc[0], rc[1], totals, outs=outs)
        else:
            def do_c():
                return multi.compress_streams(shards, totals, codec)

            def do_u(rc):
                return multi.uncompress_streams(rc[0], rc[1], totals[rank], codec)

    kc = ku = 0.0
    sampler = ClockSampler(local)
    kstat = {"c": 0.0, "u": 0.0, "l": 0}

    def after_c():
        kstat["c"] += device.last_kernel_ms(0)
        kstat["l"] += device.last_launch_count(0)

    # warm-up, then the timed steps
    for _ in range(args.warmup):
        do_u(do_c())
    if rank == 0 and not nested and not os.environ.get("SNAPPY_BENCH_NO_SAMPLER"):
        sampler.start()
    steps = args.steps if not nested else args.extra_steps

    def do_u_counted(r):
        out = do_u(r)
        kstat["u"] += device.last_kernel_ms(1)
        kstat["l"] += device.last_launch_count(1)
        return out

    try:
        tc, tu, rc, back = timed_loop(ctx, steps, 0, do_c, do_u_counted, after_c=after_c)
    finally:
        clocks = sampler.stop() if (rank == 0 and not nested) else None
    kc, ku = kstat["c"] / steps, kstat["u"] / steps
    launches = kstat["l"] * (world if world > 1 else 1)

    # ---- correctness of what was timed: round trip of everything + sampled fragments against the oracle ----
    checked = 0
    if world == 1:
        stream, index = rc
        assert torch.equal(back, d_in), "round trip mismatch in the timed configuration"
        csize = int(stream.numel())
        idx = index.cpu().numpy()
        s_np = stream.cpu().numpy()
        checked = check_fragments_vs_oracle(lambda lo, hi: raw[lo:hi], n, lambda a, b: s_np[a:b], idx, 64, args.seed)
        del s_np
        my_c_bytes = csize
        my_n = n
    else:
        if comm is not None:
            streams, indexes, lens = rc
            for s in range(world):
                assert torch.equal(back[s], shards[s]), "round trip mismatch (stream %d)" % s
            csize = int(lens[rank])
            stream, index = streams[rank], indexes[rank]
        else:
            stream, index = rc
            for s in range(world):
                assert torch.equal(back[s], shards[s]), "round trip mismatch (stream %d)" % s
            csize = int(stream.numel())
        # the owner checks the fragments of its assembled stream that came from ITS OWN run against the oracle
        # (it holds those input bytes), and through the side index every rank's segment boundaries
        idx = index.cpu().numpy()
        s_np = stream.cpu().numpy()
        lo_b, hi_b = multi.shard_bounds(n, world)[rank]
        mine = shards[rank].cpu().numpy()
        pyoracle = _oracle()
        rng = np.random.default_rng(args.seed + rank)
        f0 = lo_b // FRAGMENT
        nf = (hi_b - lo_b + FRAGMENT - 1) // FRAGMENT
        for f in sorted(set([0, nf - 1] + [int(x) for x in rng.integers(0, nf, 62)])):
            want_b = pyoracle.compress_one_fragment(np.ascontiguousarray(mine[f * FRAGMENT: (f + 1) * FRAGMENT]), n)
            got = s_np[int(idx[f0 + f]): int(idx[f0 + f + 1])]
            assert got.size == want_b.size and np.array_equal(got, want_b), \
                "rank %d: fragment %d of its stream differs from the oracle" % (rank, f0 + f)
            checked += 1
        assert int(idx[-1]) == csize and int(idx[0]) == len(multi.encode_header(n))
        my_n = sum(int(x.numel()) for x in shards)
        # bytes this rank's compress kernel produced: its run of every stream
        ratio = csize / n
        my_c_bytes = int(my_n * ratio)
    if args.dump_outputs and rank == 0 and not nested:
        # what compress_device / uncompress_device (or the communicator) handed back in the last timed step
        outs = {"compressed": stream[:csize], "compressed_index": index}
        outs.update({"uncompressed": back} if world == 1 else {"uncompressed_%d" % s: back[s] for s in range(world)})
        dump_outputs(args.dump_outputs, outs, args.seed)

    total_bytes = n * (world if world > 1 else 1)  # uncompressed bytes all ranks processed per step
    t_step_ms = (tc + tu) / steps
    value = total_bytes * steps / ((tc + tu) / 1e3) / 1e9
    comp_gbps = total_bytes * steps / (tc / 1e3) / 1e9
    unc_gbps = total_bytes * steps / (tu / 1e3) / 1e9

    # ---- roofline of the dominant kernel (per launch on THIS rank; N + C algorithmic bytes) --------------------
    alg = my_n + my_c_bytes
    dominant = "compress" if kc >= ku else "uncompress"
    k_ms = kc if dominant == "compress" else ku
    roofline = roofline_of("k_compress_window_mixed" if dominant == "compress" else "k_decode_fragments", k_ms, alg,
                           sm_mhz=(clocks or {}).get("sm_mhz"))
    roofline["other"] = {"compress_kernel_ms": kc, "uncompress_kernel_ms": ku,
                         "uncompress_achieved": (alg / (ku / 1e3) / 1e9) if ku > 0 else None}

    # ---- e2e through the host-buffer C ABI.  N > 1: every rank on its own buffer at the same time (the
    # Threads.@threads-over-independent-buffers use of the reference API), aggregate over the ranks --------------
    e2e = None
    if not args.no_e2e and not nested:
        import ctypes
        lib = Snappy._abi.lib()
        if world == 1:
            src_np = raw
        else:
            src_np = np.concatenate([gen.view(*p) for p in plan["mix_shards"]])
            with gpu_local_node(local):
                host_in = torch.from_numpy(src_np.copy()).pin_memory()
        en = int(host_in.numel())
        ecap = Snappy.maxlength_compressed(en)
        with gpu_local_node(local) as numa:
            h_out = torch.empty(ecap, dtype=torch.uint8).pin_memory()
            h_back = torch.empty(en, dtype=torch.uint8).pin_memory()

        def e2e_step(pin, pout, pback):
            ol = ctypes.c_size_t(ecap)
            r1 = lib.snappy_b200_compress(pin, en, pout, ctypes.byref(ol))
            assert r1 == 0, r1
            bl = ctypes.c_size_t(en)
            r2 = lib.snappy_b200_uncompress(pout, ol.value, pback, ctypes.byref(bl))
            assert r2 == 0 and bl.value == en, r2
            return ol.value

        def e2e_run(pin, pout, pback, reps):
            e2e_step(pin, pout, pback)
            ctx["barrier"]()
            t0 = time.perf_counter()
            for _ in range(reps):
                c_len = e2e_step(pin, pout, pback)
            torch.cuda.synchronize()
            dt = (time.perf_counter() - t0) / reps
            if world > 1:
                t = torch.tensor([dt], dtype=torch.float64, device=dev)
                dist.all_reduce(t, op=dist.ReduceOp.MAX)
                dt = float(t[0])
            return dt, c_len

        reps = args.steps
        dt, c_len = e2e_run(host_in.data_ptr(), h_out.data_ptr(), h_back.data_ptr(), reps)
        assert torch.equal(h_back, host_in)
        e2e = {"value": en * world / dt / 1e9, "unit": "GB/s", "h2d_bytes_per_step": (en + c_len) * world,
               "d2h_bytes_per_step": (c_len + en) * world, "ms_per_step": dt * 1e3, "reps": reps,
               "api": "snappy_b200_compress + snappy_b200_uncompress on pinned host buffers" +
                      ("" if world == 1 else ", every rank on its own %d MiB buffer at the same time" % (en >> 20)),
               "pinned_on_gpu_numa_node": numa.local}
        launches_e2e = device.last_launch_count(0) + device.last_launch_count(1)
        e2e["gpu_launches_per_step"] = launches_e2e
        # the same from PAGEABLE memory: what a plain Vector{UInt8} is
        with gpu_local_node(local):
            p_in = np.array(host_in.numpy(), copy=True)
            p_out = np.empty(ecap, dtype=np.uint8)
            p_back = np.empty(en, dtype=np.uint8)
            p_out[::4096] = 0
            p_back[::4096] = 0
        dtp, _ = e2e_run(p_in.ctypes.data, p_out.ctypes.data, p_back.ctypes.data, reps)
        assert np.array_equal(p_back, p_in)
        e2e["pageable"] = {"value": en * world / dtp / 1e9, "unit": "GB/s", "ms_per_step": dtp * 1e3,
                           "of_pinned": dt / dtp,
                           "api": "the same calls on ordinary (pageable) numpy arrays: what the reference API "
                                  "hands over (src/Snappy.jl:25,48)"}
        del p_in, p_out, p_back

    # ---- cpu_baseline: the oracle on host cores, rank 0 at N = 1 only -------------------------
    cpu = None
    if world == 1 and rank == 0 and not args.no_cpu_baseline and not nested:
        cores = ctx["cores"]
        sample_frag = min(nfrag, 4096)
        sample = raw[: sample_frag * FRAGMENT]
        a1, b1, _ = oracle_roundtrip_threads(sample, 1)
        aT, bT, _ = oracle_roundtrip_threads(sample, cores)
        cpu = {"value": sample.size / (aT + bT) / 1e9, "unit": "GB/s", "cores": cores, "kind": "port",
               "sample": "first %d MiB of the same buffer, %d independent buffers on %d threads" % (
                   sample.size >> 20, cores, cores),
               "single_thread": {"value": sample.size / (a1 + b1) / 1e9,
                                 "compress_gbps": sample.size / a1 / 1e9,
                                 "uncompress_gbps": sample.size / b1 / 1e9},
               "compress_gbps": sample.size / aT / 1e9, "uncompress_gbps": sample.size / bT / 1e9}

    if rank != 0:
        return None
    sharding = "none" if world == 1 else (
        "%d streams x %d ranks, whole-fragment runs; ncclAllGather of the byte counts on the compute stream, fragments "
        "and side-index entries stored straight into the owner's buffer over NVLink (snappy_b200_comm)" % (world, world)
        if comm is not None else
        "%d streams x %d ranks, whole-fragment runs, torch.distributed size all-gather + all-to-all assembly" % (world, world))
    return {
        "metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": steps,
        "warmup": args.warmup, "ms_per_step": t_step_ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic",
        "compress_gbps": comp_gbps, "uncompress_gbps": unc_gbps,
        "compressed_ratio": csize / n,
        "config": {"workload": workload_name(2, args) + "; round trip asserted, %d sampled fragments per rank "
                               "byte-identical to the oracle (Snappy.jl restatement)" % checked,
                   "bytes_per_gpu": n, "seed": args.seed,
                   "l2": "inputs (1 GiB) larger than L2 (126 MB); no explicit flush",
                   "sharding": sharding},
        "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": launches, "clocks": clocks,
    }


# ------------------------------------------------------------------------------------------ config 3
def config3(ctx, nested=False):
    """the ORACLE's 1 GiB stream, no side index (replicas at N > 1: the parse does not shard, SURVEY.md 8(e))"""
    torch, device, args, dev, rank, world = ctx["torch"], ctx["device"], ctx["args"], ctx["dev"], ctx["rank"], ctx["world"]
    raw = ctx["gen"].view(*ctx["plan"]["mix"])
    n = raw.size
    t0 = time.perf_counter()
    stream_np = oracle_stream_parallel(raw, ctx["cores"])
    t_oracle = time.perf_counter() - t0
    d_stream = torch.from_numpy(stream_np).to(dev)
    d_raw = torch.from_numpy(raw.copy()).to(dev)
    d_back = torch.empty(n, dtype=torch.uint8, device=dev)
    steps = args.steps if not nested else args.extra_steps
    k = {"u": 0.0, "l": 0}

    def do_u(_):
        r = device.uncompress_device(d_stream, out=d_back, index=None, claimed=n)
        k["u"] += device.last_kernel_ms(1)
        k["l"] += device.last_launch_count(1)
        return r

    for _ in range(args.warmup):
        do_u(None)
    k["u"], k["l"] = 0.0, 0
    _, tu, _, back = timed_loop(ctx, steps, 0, None, do_u)
    assert torch.equal(back, d_raw), "config 3: decoded bytes differ from the input"
    value = n * world * steps / (tu / 1e3) / 1e9
    ku = k["u"] / steps
    if rank != 0:
        return None
    return {
        "metric": METRICS[3], "value": value, "unit": "GB/s", "n_gpus": world, "steps": steps, "warmup": args.warmup,
        "ms_per_step": tu / steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8",
        "data": "synthetic", "uncompress_gbps": value, "compressed_ratio": stream_np.size / n,
        "compressed_gbps": stream_np.size * world * steps / (tu / 1e3) / 1e9,
        "config": {"workload": workload_name(3, args) + "; output compared with the input byte for byte",
                   "stream_from": "oracle/snappy_oracle.c (sjo_compress_fragments on %d threads, %.1f s)" % (
                       ctx["cores"], t_oracle),
                   "parse_plus_other_ms": tu / steps - ku, "l2": "stream (0.48 GB) and output (1 GiB) larger than L2"},
        "roofline": roofline_of("k_decode_fragments", ku, n + stream_np.size,
                                note="decode kernel only; the index-free parse is the rest of the step"),
        "gpu_launches": k["l"],
    }


# ------------------------------------------------------------------------------------------ config 4
def config4(ctx, nested=False):
    """2^20 independent 4 KiB pages through the batched API (pages split over the ranks at N > 1: no exchange)"""
    torch, dist, device, args, dev, rank, world = (ctx["torch"], ctx["dist"], ctx["device"], ctx["args"], ctx["dev"],
                                                   ctx["rank"], ctx["world"])
    gen = ctx["gen"]
    parts = [gen.view(*p) for p in ctx["plan"]["pages"]]
    per_frag = FRAGMENT // 4096
    have = sum(p.size for p in parts) // 4096
    npages = min(have, args.pages // world + (1 if rank < args.pages % world else 0)) if world > 1 else min(have, args.pages)
    d_in = torch.empty(npages * 4096, dtype=torch.uint8, device=dev)
    off = 0
    for p in parts:
        k = min(p.size, npages * 4096 - off)
        if k <= 0:
            break
        d_in[off: off + k] = torch.from_numpy(p[:k].copy()).to(dev)
        off += k
    in_off = torch.arange(npages, dtype=torch.int64, device=dev) * 4096
    in_sz = torch.full((npages,), 4096, dtype=torch.int32, device=dev)
    cap = 32 + 4096 + 4096 // 6
    cap = (cap + 15) // 16 * 16
    out_off = torch.arange(npages, dtype=torch.int64, device=dev) * cap
    d_out = torch.empty(npages * cap, dtype=torch.uint8, device=dev)
    d_back = torch.empty(npages * 4096, dtype=torch.uint8, device=dev)
    steps = args.steps if not nested else args.extra_steps
    k = {"c": 0.0, "u": 0.0, "l": 0}

    def do_c():
        r = device.compress_batched_device(d_in, in_off, in_sz, out=d_out, out_offsets=out_off)
        k["c"] += device.last_kernel_ms(0)
        k["l"] += device.last_launch_count(0)
        return r

    def do_u(rc):
        r = device.uncompress_batched_device(rc[0], rc[1], rc[2], d_back, in_off, in_sz)
        k["u"] += device.last_kernel_ms(1)
        k["l"] += device.last_launch_count(1)
        return r

    for _ in range(args.warmup):
        do_u(do_c())
    k["c"] = k["u"] = 0.0
    k["l"] = 0
    tc, tu, rc, ru = timed_loop(ctx, steps, 0, do_c, do_u)
    out, _, out_sz = rc
    sizes, statuses = ru
    assert int(statuses.abs().sum().item()) == 0 and torch.equal(d_back, d_in), "config 4: page round trip"
    # >= 1000 sampled pages: the page's stream must be the oracle's compress of the page (own varint, table sized
    # from the page length, src/Snappy.jl:26-27)
    pyoracle = _oracle()
    rng = np.random.default_rng(args.seed + 4 + rank)
    picks = sorted(set([0, npages - 1] + [int(x) for x in rng.integers(0, npages, 1022)]))
    sel = torch.tensor(picks, dtype=torch.int64, device=dev)
    szs = out_sz[sel].cpu().numpy()
    rows = out.view(npages, cap)[sel].cpu().numpy()
    src = d_in.view(npages, 4096)[sel].cpu().numpy()
    for i in range(len(picks)):
        want = pyoracle.compress_np(src[i])
        assert int(szs[i]) == want.size and np.array_equal(rows[i, : want.size], want), "config 4: page %d" % picks[i]
    total = npages * 4096
    csize = int(out_sz.sum().item())
    if world > 1:
        t = torch.tensor([total, csize], dtype=torch.int64, device=dev)
        dist.all_reduce(t)
        total, csize = int(t[0]), int(t[1])
    value = total * steps / ((tc + tu) / 1e3) / 1e9
    kc, ku = k["c"] / steps, k["u"] / steps
    if rank != 0:
        return None
    mine = npages * 4096
    return {
        "metric": METRICS[4], "value": value, "unit": "GB/s", "n_gpus": world, "steps": steps, "warmup": args.warmup,
        "ms_per_step": (tc + tu) / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic", "compress_gbps": total * steps / (tc / 1e3) / 1e9,
        "uncompress_gbps": total * steps / (tu / 1e3) / 1e9, "compressed_ratio": csize / total,
        "config": {"workload": workload_name(4, args) + "; round trip of every page asserted, %d sampled pages "
                               "byte-identical to the oracle" % len(picks),
                   "pages_this_rank": npages, "l2": "input (4 GiB at N = 1) larger than L2"},
        "roofline": roofline_of("k_compress_pages_window", kc, mine + int(out_sz.sum().item())),
        "other_kernel": {"k_decode_pages_ms": ku},
        "gpu_launches": k["l"] * world,
    }


# ------------------------------------------------------------------------------------------ config 5
def config5(ctx, nested=False):
    """8 streams x 1 GiB of source-like text, the same streams at every N; every stream sharded over the N ranks"""
    torch, dist, device, multi, args = ctx["torch"], ctx["dist"], ctx["device"], ctx["multi"], ctx["args"]
    dev, rank, world, comm, gen = ctx["dev"], ctx["rank"], ctx["world"], ctx["comm"], ctx["gen"]
    S = args.streams
    total_len = args.fragments * FRAGMENT
    totals = [total_len] * S
    if comm is None:
        raise RuntimeError("config 5 needs the library communicator: " + str(ctx["comm_note"]))
    shards, shards_np = [], []
    for s in range(S):
        views = [gen.view(*p) for p in ctx["plan"]["source"].get(s, [])]
        a = np.concatenate(views) if len(views) > 1 else (views[0] if views else np.zeros(0, dtype=np.uint8))
        shards_np.append(a)
        shards.append(torch.from_numpy(np.ascontiguousarray(a).copy()).to(dev) if a.size else None)
    lo_b, hi_b = multi.shard_bounds(total_len, world)[rank]
    outs = [torch.empty(hi_b - lo_b, dtype=torch.uint8, device=dev) for _ in range(S)]
    steps = args.steps if not nested else args.extra_steps
    k = {"c": 0.0, "u": 0.0, "l": 0}

    def do_c():
        r = comm.compress(shards, totals)
        k["c"] += device.last_kernel_ms(0)
        k["l"] += device.last_launch_count(0)
        return r

    def do_u(rc):
        r = comm.uncompress(rc[0], rc[1], totals, outs=outs)
        k["u"] += device.last_kernel_ms(1)
        k["l"] += device.last_launch_count(1)
        return r

    for _ in range(args.warmup):
        do_u(do_c())
    k["c"] = k["u"] = 0.0
    k["l"] = 0
    tc, tu, rc, back = timed_loop(ctx, steps, 0, do_c, do_u)
    streams, indexes, lens = rc
    for s in range(S):
        if shards[s] is not None:
            assert torch.equal(back[s], shards[s]), "config 5: round trip of stream %d on rank %d" % (s, rank)
    # sampled fragments of this rank's runs against the oracle, located through the owners' side indexes: the
    # owner publishes its index (small), every rank cuts the bytes of ITS fragments out of the owner's stream
    pyoracle = _oracle()
    checked = 0
    f0 = lo_b // FRAGMENT
    nf = (hi_b - lo_b + FRAGMENT - 1) // FRAGMENT
    rng = np.random.default_rng(args.seed + 5 + rank)
    for s in range(S):
        owner = s % world
        nfr = args.fragments
        if world > 1:
            idx_t = indexes[s].clone() if comm.owns(s) else torch.empty(nfr + 1, dtype=torch.int64, device=dev)
            dist.broadcast(idx_t, src=owner)
            idx = idx_t.cpu().numpy()
        else:
            idx = indexes[s].cpu().numpy()
        picks = sorted(set([0, nf - 1] + [int(x) for x in rng.integers(0, nf, 6)])) if nf else []
        # the bytes of my sampled fragments: pulled from the owner
        for f in picks:
            a, b = int(idx[f0 + f]), int(idx[f0 + f + 1])
            if world > 1:
                buf = torch.empty(b - a, dtype=torch.uint8, device=dev)
                if comm.owns(s):
                    buf.copy_(streams[s][a:b])
            else:
                buf = streams[s][a:b]
            got = buf.cpu().numpy() if (world == 1 or comm.owns(s)) else None
            if got is not None:
                want = pyoracle.compress_one_fragment(
                    np.ascontiguousarray(shards_np[s][f * FRAGMENT: (f + 1) * FRAGMENT]), total_len)
                assert got.size == want.size and np.array_equal(got, want), \
                    "config 5: stream %d fragment %d differs from the oracle" % (s, f0 + f)
                checked += 1
        assert int(idx[-1]) == lens[s]
    total = S * total_len
    csize = sum(lens)
    value = total * steps / ((tc + tu) / 1e3) / 1e9
    kc, ku = k["c"] / steps, k["u"] / steps
    if world > 1:
        t = torch.tensor([checked], dtype=torch.int64, device=dev)
        dist.all_reduce(t)
        checked = int(t[0])
    if rank != 0:
        return None
    my_n = sum(a.size for a in shards_np)
    return {
        "metric": METRICS[5], "value": value, "unit": "GB/s", "n_gpus": world, "steps": steps, "warmup": args.warmup,
        "ms_per_step": (tc + tu) / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "u8", "data": "synthetic", "compress_gbps": total * steps / (tc / 1e3) / 1e9,
        "uncompress_gbps": total * steps / (tu / 1e3) / 1e9, "compressed_ratio": csize / total,
        "config": {"workload": workload_name(5, args) + "; round trip asserted, %d sampled fragments byte-identical "
                               "to the oracle" % checked,
                   "sharding": "stream s owned by rank s mod N; ncclAllGather of byte counts + NVLink peer stores "
                               "(snappy_b200_comm)" if world > 1 else "one GPU: all streams in one kernel pass",
                   "l2": "inputs larger than L2"},
        "roofline": roofline_of("k_compress_window_mixed", kc, my_n + int(csize * my_n / total),
                                note="per launch on this rank: its runs of all streams", scale_capture=False),
        "other_kernel": {"k_decode_fragments_ms": ku},
        "gpu_launches": k["l"] * world,
    }


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    return run_b200(args)


if __name__ == "__main__":
    sys.exit(main())
