"""Validation (snappy_b200_validate_*): the status uncompress would return with unlimited room, without an output.

Contract (include/snappy_b200.h): for any bytes, validation returns exactly what snappy_b200_uncompress returns when
the output capacity is unlimited -- 0 or the reference's status 2..6, never BUFFER_TOO_SMALL -- and a side index,
right or wrong, cannot change it.  The chain mirrors uncompress_device_locked: path 0 (every fragment of the side index
is clean), 1 (the relaxed parse decides: its first failing element, or a complete error-free parse whose lengths add
up), 2 (the parse lost the chain: status-only walk from the last tile start it reached), 3 (status-only walk over the
whole stream).

CPU: the status-only kernels run on the CPU warp with a NULL output pointer (tools/cpu_warp/run_decode_parsed.cpp,
modes `validate` and `validate-pages`) over test_decode_corruption's corpus, without an index, with the oracle's index
and with a stale one.  GPU (-m gpu): the device, host and batched calls against the oracle and against uncompress."""
import collections
import os

import numpy as np
import pytest

from conftest import ROOT
from test_decode_corruption import (CPU_SEED, FRAGMENT, GPU_SEED, ZERO_LITERAL, Elements, _claimed, _stale_index,
                                    base_streams, build_driver, corrupt_corpus, run_driver, subset, write_cases)


def oracle_index(oracle, s):
    """the side index of a stream the oracle accepts whose elements start on every 64 KiB boundary, else None"""
    try:
        el = Elements(s, oracle)
    except (AssertionError, IndexError, ValueError, oracle.OracleError):
        return None
    if any(int(el.op[e]) != (k + 1) * FRAGMENT for k, e in enumerate(el.boundaries())):
        return None
    return [el.hdr] + [int(el.ip[e]) for e in el.boundaries()] + [len(s)]


def line_fields(line):
    """(status, parsed status, oracle status, path or None, step3) of a `validate` line"""
    head = line.split(": status ", 1)[1]
    st, rest = head.split(" parsed ", 1)
    dec, rest = rest.split(" (oracle ", 1)
    want, rest = rest.split(") path ", 1)
    path = rest.split(":", 1)[0].split()[0]
    return int(st), int(dec), int(want), (None if path == "-" else int(path)), " step3:" in line


def run_validate(exe, files, env=None):
    """the driver's `validate` lines in file order"""
    by_file = {l.split(": status ", 1)[0]: l for l in run_driver(exe, "validate", files, env)}
    assert len(by_file) == len(files)
    return [by_file[f] for f in files]


def write_index(path, idx):
    np.asarray(idx, dtype="<u8").tofile(path)


# ---------------------------------------------------------------------------------------------- CPU tests
@pytest.fixture(scope="module")
def validate_corpus(oracle, tmp_path_factory):
    """the CPU corpus with two side indexes per stream: the oracle's (valid streams) and the stale one of its base"""
    d = str(tmp_path_factory.mktemp("validate_corpus"))
    cases = corrupt_corpus(oracle, CPU_SEED, 80, max_frags=12)
    files = write_cases(d, cases)
    bases = dict(base_streams(oracle, 12))
    for (name, s), f in zip(cases, files):
        claimed = _claimed(oracle, s)
        if claimed is None:
            continue
        write_index(f + ".sidx", _stale_index(oracle, bases[name.split("/")[1]], claimed))
        idx = oracle_index(oracle, s)
        if idx is not None:
            write_index(f + ".oidx", idx)
    exe = build_driver(str(tmp_path_factory.mktemp("validate_driver")))
    return cases, files, exe


@pytest.mark.parametrize("suffix", [None, ".oidx", ".sidx"], ids=["no_index", "oracle_index", "stale_index"])
def test_validate_kernels_match_oracle_and_decode_on_the_corpus(oracle, validate_corpus, suffix):
    """every corpus stream through the status-only chain with a NULL output: the oracle's status, and the same status
    as the decoding chain (`parsed`); with the oracle's index the valid streams take path 0"""
    cases, files, exe = validate_corpus
    lines = run_validate(exe, files, {"IDX_SUFFIX": suffix} if suffix else None)
    bad = [l for l in lines if "0 mismatches" not in l]
    assert not bad, "\n".join(bad[:20])
    paths = collections.Counter()
    for (name, s), line in zip(cases, lines):
        st, dec, want, path, step3 = line_fields(line)
        assert st == dec == want == oracle.status_of_uncompress(s), line
        paths[path] += 1
    print("paths", dict(paths))
    if suffix == ".oidx":
        assert paths[0] >= 20, paths
    else:
        assert paths[0] == 0 or suffix == ".sidx", paths
    assert paths[1] >= 5 and paths[2] >= 5, paths


def test_complete_error_free_parse_means_the_reference_accepts(oracle, validate_corpus):
    """the claim path 1 rests on: whenever the parse followed the chain to the end, met no failing element and the
    lengths add up, the oracle accepts the stream -- on every corpus stream that gets there"""
    cases, files, exe = validate_corpus
    lines = run_validate(exe, files)
    claimed_ok = [(name, line) for (name, s), line in zip(cases, lines) if line_fields(line)[4]]
    assert len(claimed_ok) >= 30, len(claimed_ok)
    wrong = [line for (name, line) in claimed_ok if line_fields(line)[2] != 0]
    assert not wrong, "\n".join(wrong[:20])


@pytest.mark.parametrize("pshift", ["9", "12"])
def test_validate_kernels_parse_chunk_variants(validate_corpus, pshift):
    cases, files, exe = validate_corpus
    pick = subset(cases)
    lines = run_validate(exe, [files[i] for i in pick], {"PSHIFT": pshift})
    bad = [l for l in lines if "0 mismatches" not in l]
    assert not bad, "\n".join(bad[:20])


def test_validate_pages_kernel_matches_oracle(validate_corpus):
    """every corpus stream as one page of k_validate_pages (no output), plus empty pages: status and claimed length"""
    cases, files, exe = validate_corpus
    lines = run_driver(exe, "validate-pages", files)
    bad = [l for l in lines if "0 mismatches" not in l]
    assert not bad, "\n".join(bad[:20])
    assert len(lines) >= len(files)
    assert sum("(empty page)" in l and "status 6 (oracle 6)" in l for l in lines) >= 2


# ---------------------------------------------------------------------------------------------- GPU tests
def _path(snappy):
    return snappy._abi.lib().snappy_b200_get_option(b"last_decode_path")


def _dev(torch, s):
    return torch.from_numpy(np.frombuffer(bytes(s), dtype=np.uint8).copy()).cuda() if len(s) else \
        torch.empty(0, dtype=torch.uint8, device="cuda")


@pytest.fixture(scope="module")
def gpu_cases(oracle):
    cases = corrupt_corpus(oracle, GPU_SEED, 160, max_frags=40)
    return cases, [oracle.status_of_uncompress(s) for _, s in cases]


@pytest.mark.gpu
def test_device_and_host_validate_match_oracle_on_the_corpus(snappy, oracle, gpu_cases):
    """every GPU corpus stream: device validate without an index, with the oracle's index and with a stale index, and
    host validate -- the oracle's status and the header's claimed length"""
    import torch
    from snappy_jl_b200 import device
    cases, want = gpu_cases
    bases = dict(base_streams(oracle, 40))
    wrong, paths = [], collections.Counter()
    for (name, s), want_st in zip(cases, want):
        claimed = _claimed(oracle, s)
        d = _dev(torch, s)
        indexes = [("no index", None)]
        if claimed is not None:
            indexes.append(("stale index", _stale_index(oracle, bases[name.split("/")[1]], claimed)))
            idx = oracle_index(oracle, s)
            if idx is not None:
                indexes.append(("oracle index", idx))
        for what, idx in indexes:
            t = None if idx is None else torch.tensor(idx, dtype=torch.int64, device="cuda")
            st, got_claimed = device.validate_device(d, index=t)
            paths[(what, _path(snappy))] += 1
            if st != want_st or got_claimed != claimed:
                wrong.append("%s: %s: status %d (oracle %d), claimed %r (%r)" % (name, what, st, want_st, got_claimed, claimed))
        st = snappy.validate(s)
        if st != want_st:
            wrong.append("%s: host: status %d (oracle %d)" % (name, st, want_st))
    print("paths", dict(paths))
    assert not wrong, "\n".join(wrong[:20])
    assert paths[("oracle index", 0)] >= 20, paths
    for p in (1, 2, 3):
        assert paths[("no index", p)] >= 1, paths


@pytest.mark.gpu
@pytest.mark.parametrize("option,value", [("parse_chunk_log2", 9), ("parse_chunk_log2", 13), ("clean_cuts", 0)])
def test_device_validate_option_variants(snappy, oracle, gpu_cases, option, value):
    import torch
    from snappy_jl_b200 import device
    cases, want = gpu_cases
    defaults = {"parse_chunk_log2": 10, "clean_cuts": 1}
    wrong = []
    try:
        device.set_option(option, value)
        for (name, s), want_st in zip(cases, want):
            st, _ = device.validate_device(_dev(torch, s))
            if st != want_st:
                wrong.append("%s: status %d (oracle %d)" % (name, st, want_st))
    finally:
        for k, v in defaults.items():
            device.set_option(k, v)
    assert not wrong, "\n".join(wrong[:20])


@pytest.mark.gpu
def test_batched_validate_with_corrupt_neighbours(snappy, oracle, gpu_cases):
    """corpus streams of up to 4 MiB as pages between valid pages: per page the oracle's status, the status
    uncompress_batched_device reports with room for the claimed length, and the claimed length"""
    import torch
    from snappy_jl_b200 import device, synth
    cases, want = gpu_cases
    pages = []  # (stream, status)
    for k, ((name, s), st) in enumerate(zip(cases, want)):
        if len(s) > 4 << 20:
            continue
        pages.append((s, st))
        raw = synth.mix(1, seed=k, tail=int(k * 37 % 5000))[: 1000 + 997 * k % 70000]
        pages.append((oracle.compress(raw.tobytes()), 0))
    pages.append((b"", 6))
    in_off, flat, out_off, caps, o = [], bytearray(), [], [], 0
    for s, _ in pages:
        in_off.append(len(flat))
        flat += s + bytes(-len(s) % 16)
        cap = _claimed(oracle, s) or 0
        caps.append(cap)
        out_off.append(o)
        o += (cap + 15) // 16 * 16
    data = torch.from_numpy(np.frombuffer(bytes(flat) + bytes(16), dtype=np.uint8).copy()).cuda()
    t = lambda v, dt: torch.tensor(v, dtype=dt, device="cuda")
    offs, sizes = t(in_off, torch.int64), t([len(p[0]) for p in pages], torch.int32)
    statuses, claimed = device.validate_batched_device(data, offs, sizes)
    out = torch.empty(max(o, 1), dtype=torch.uint8, device="cuda")
    _, dec = device.uncompress_batched_device(data, offs, sizes, out, t(out_off, torch.int64), t(caps, torch.int32))
    statuses, claimed, dec = statuses.cpu().numpy(), claimed.cpu().numpy(), dec.cpu().numpy()
    wrong = []
    for k, (s, st) in enumerate(pages):
        if statuses[k] != st or dec[k] != st or claimed[k] != caps[k]:
            wrong.append("page %d: status %d, uncompress %d (oracle %d), claimed %d (%d)"
                         % (k, statuses[k], dec[k], st, claimed[k], caps[k]))
    assert not wrong, "\n".join(wrong[:20])


@pytest.mark.gpu
def test_validate_data_files_and_parquet_pages(snappy, oracle):
    """tests/data/*.snappy through host and device validate, and every page of pyarrow-written Parquet files through
    validate_pages: 0 on the pyarrow pages, -1 on uncompressed ones, the oracle's status on a corrupted page"""
    import torch
    from snappy_jl_b200 import device
    data = os.path.join(ROOT, "tests", "data")
    names = sorted(f for f in os.listdir(data) if f.endswith(".snappy"))
    assert {"baddata1.snappy", "baddata2.snappy", "baddata3.snappy", "alice29.snappy"} <= set(names)
    for f in names:
        s = open(os.path.join(data, f), "rb").read()
        want = oracle.status_of_uncompress(s)
        assert snappy.validate(s) == want, f
        assert device.validate_device(_dev(torch, s))[0] == want, f
    pa = pytest.importorskip("pyarrow")
    pq = pytest.importorskip("pyarrow.parquet")
    import io
    from snappy_jl_b200 import parquet_pages as pp
    rows = 60_000
    t = pa.table({"id": np.arange(rows, dtype=np.int64), "text": ["row %d" % (i % 977) for i in range(rows)],
                  "raw": np.arange(rows, dtype=np.int32)})
    buf = io.BytesIO()
    pq.write_table(t, buf, compression={"id": "snappy", "text": "snappy", "raw": "none"}, data_page_size=4096)
    f = buf.getvalue()
    pages, st = pp.validate_pages(f)
    snappy_pages = [i for i, p in enumerate(pages) if p["codec"] == "SNAPPY" and p["compressed"] > 0]
    assert len(snappy_pages) > 20 and any(p["codec"] == "UNCOMPRESSED" for p in pages)
    for i, p in enumerate(pages):
        assert st[i] == (0 if i in snappy_pages else -1), (i, p, st[i])
    # corrupt one byte near the end of a few page streams: the oracle's status on those pages, 0 on the rest
    g = bytearray(f)
    hit = snappy_pages[3::max(1, len(snappy_pages) // 5)]
    for i in hit:
        p = pages[i]
        g[p["stream"] + p["compressed"] - 2] ^= 0x5A
    _, st2 = pp.validate_pages(bytes(g), pages)
    for i in snappy_pages:
        p = pages[i]
        body = bytes(g[p["stream"]: p["stream"] + p["compressed"]])
        want = oracle.status_of_uncompress(body)
        if want == 0 and _claimed(oracle, body) != p["uncompressed"]:
            want = 2
        assert st2[i] == want, (i, st2[i], want)


@pytest.mark.gpu
def test_huge_claim_needs_no_large_allocation(snappy):
    """a 20-byte stream whose header claims 0xFFFFFFFF bytes: judged (the lengths do not add up: status 2; a copy that
    reaches before the output: status 3) without an allocation anywhere near the claimed length"""
    import torch
    from snappy_jl_b200 import device
    hdr = bytes([0xFF, 0xFF, 0xFF, 0xFF, 0x0F])
    lit = hdr + bytes([13 << 2]) + bytes(range(14))                    # 5 + 1 + 14 = 20 bytes
    cpy = hdr + bytes([3 << 2]) + b"abcd" + bytes([(9 << 2) | 2, 100, 0]) + bytes(7)  # copy of offset 100 after 4 bytes
    assert len(lit) == 20 and len(cpy) == 20
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    for s, want in ((lit, 2), (cpy, 3)):
        assert snappy.validate(s) == want
        assert device.validate_device(_dev(torch, s)) == (want, 0xFFFFFFFF)
    free1, _ = torch.cuda.mem_get_info()
    assert free0 - free1 < 64 << 20, (free0, free1)


@pytest.mark.gpu
def test_host_validate_large_streams_pinned_and_pageable(snappy, oracle):
    """streams of more than 64 MiB with a fault in the first, a middle and the last part, a truncation, a header that
    claims one fragment too many and a valid stream with a trailing byte: host validate from pageable (numpy) and pinned
    (torch pin_memory) buffers"""
    import torch
    from snappy_jl_b200 import synth
    tile = synth.mix(256, seed=31)
    parts0, _ = oracle.compress_fragments(tile, tile.size, 0, 256)
    reps = (72 << 20) // parts0.size + 1
    total = tile.size * reps
    parts, sizes = oracle.compress_fragments(tile, total, 0, 256)
    hdr = np.frombuffer(oracle.encode32(total), dtype=np.uint8)
    good = np.concatenate([hdr] + [parts] * reps)
    assert good.size > 64 << 20
    streams = [("good", good)]
    for where in (0.03, 0.5, 0.97):
        st, k = 0, 0
        while st == 0:
            bad = good.copy()
            pos = int(good.size * where) + 7919 * k
            bad[pos: pos + 24] ^= 0xA7
            st = oracle.status_of_uncompress(bad)
            k += 1
            assert k < 40
        streams.append(("garbled@%.2f" % where, bad))
    streams.append(("truncated", good[: good.size - 12345]))
    streams.append(("claimed+65536", np.concatenate([np.frombuffer(oracle.encode32(total + FRAGMENT), dtype=np.uint8),
                                                      good[hdr.size:]])))
    streams.append(("trailing_byte", np.concatenate([good, np.array([9], dtype=np.uint8)])))
    cut = hdr.size + parts.size * (reps // 2) + int(sizes[:100].sum())
    streams.append(("zero_literal", np.concatenate([good[:cut], np.frombuffer(ZERO_LITERAL, dtype=np.uint8), good[cut:]])))
    wrong = []
    for name, s in streams:
        want = oracle.status_of_uncompress(s)
        pinned = torch.empty(s.size, dtype=torch.uint8, pin_memory=True)
        pinned.numpy()[:] = s
        for what, buf in (("pageable", s), ("pinned", pinned.numpy())):
            st = snappy.validate(buf)
            if st != want:
                wrong.append("%s: %s: status %d (oracle %d)" % (name, what, st, want))
    assert not wrong, "\n".join(wrong)
