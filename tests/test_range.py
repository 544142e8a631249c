"""Range decoding (snappy_b200_uncompress_range_device / _ranges_device): bytes [offset, offset + length) of a stream's
output, decoding only the tiles that overlap them.

Contract (include/snappy_b200.h):
- header first (BAD_VARINT), then the range (offset + length > claimed: BAD_ARGUMENT), then the stream;
- without an index the call is exact: the status of uncompress with unlimited room, and on OK that output's slice;
- with an index the touched fragments offset // 64 KiB .. (offset + length - 1) // 64 KiB are trusted to start where
  the index says.  If each is clean as k_decode_fragments defines it, the call returns OK and their bytes; otherwise it
  returns what the no-index call returns.

CPU: tools/cpu_warp/run_decode_parsed.cpp, mode `range`, runs the chain kernel for kernel over test_decode_corruption's
corpus with every range kind, without an index, with the oracle's index and with a stale one; the expected result comes
from the oracle and from `fragment_clean` below, a model of the per-fragment rule.  GPU (-m gpu): the device calls
against slices of uncompress_device's output, on the corpus, the data files, foreign streams and a 1 GiB stream."""
import collections
import os
import zlib

import numpy as np
import pytest

from conftest import ROOT
from test_decode_corruption import (CPU_SEED, FRAGMENT, GPU_SEED, _claimed, _stale_index, base_streams, build_driver,
                                    corrupt_corpus, run_driver, write_cases)
from test_validate import oracle_index, write_index

BAD_VARINT, BAD_ARGUMENT = 6, 10


# ---------------------------------------------------------------------------------------------- the model
def fragment_clean(s, idx, f, hdr, claimed):
    """k_decode_fragments' verdict on fragment f under the side index idx: it starts at idx[f] (fragment 0 behind the
    header), ends exactly at idx[f + 1] (the last one at the end of the stream), its elements parse inside it, none has
    length 0 or reaches before the fragment, and they produce exactly its 64 KiB (or the tail).  Unlike the reference's
    loop (src/internal.jl:416), a lone trailing byte is not skipped: the fragment must end on an element boundary."""
    nfrag = (claimed + FRAGMENT - 1) // FRAGMENT
    ip, ie, n = idx[f], idx[f + 1], len(s)
    on = min(FRAGMENT, claimed - f * FRAGMENT)
    if not (ip <= ie <= n and (f != 0 or ip == hdr) and (f != nfrag - 1 or ie == n)):
        return False
    p, op = ip, 0
    while p < ie:
        c = s[p]
        kind = c & 3
        extra = (c >> 2) - 59 if kind == 0 and (c >> 2) >= 60 else (0 if kind == 0 else (4 if kind == 3 else kind))
        if p + 1 + extra > ie:
            return False
        v = int.from_bytes(s[p + 1: p + 1 + extra], "little")
        if kind == 0:
            length, off = ((v if extra else c >> 2) + 1) & 0xFFFFFFFF, 0
            if length > ie - p - 1 - extra:
                return False
        elif kind == 1:
            length, off = 4 + ((c >> 2) & 7), ((c >> 5) << 8) | v
        else:
            length, off = (c >> 2) + 1, v
        if length == 0 or length > on or (kind and (off == 0 or off > op)):
            return False
        op += length
        if op > on:
            return False
        p += 1 + extra + (0 if kind else length)
    return op == on


def touched(offset, length):
    return range(offset // FRAGMENT, (offset + length - 1) // FRAGMENT + 1) if length else range(0)


def touched_bytes(oracle, s, idx, claimed, offset, length):
    """the oracle's decode of the touched fragments, each on its own, sliced to the range"""
    fs = touched(offset, length)
    parts = []
    for f in fs:
        on = min(FRAGMENT, claimed - f * FRAGMENT)
        parts.append(oracle.uncompress(oracle.encode32(on) + bytes(s[idx[f]: idx[f + 1]])))
    b = b"".join(parts)
    a = offset - fs[0] * FRAGMENT
    return b[a: a + length]


def expect(oracle, s, claimed, idx, offset, length, full):
    """(status, bytes or None, True when the index decides) of a range read; full = (status, output) of uncompress"""
    if claimed is None:
        return BAD_VARINT, None, False
    if offset + length > claimed:
        return BAD_ARGUMENT, None, False
    hdr = oracle.parse32(s, 0)[1]
    if idx is not None and all(fragment_clean(s, idx, f, hdr, claimed) for f in touched(offset, length)):
        return 0, (touched_bytes(oracle, s, idx, claimed, offset, length) if length else b""), True
    st, out = full
    return st, (bytes(out[offset: offset + length]) if st == 0 else None), False


def ranges_for(claimed, every_boundary=True):
    """empty, whole, one byte at each end, fragment-aligned, +-1 around every boundary (else the first and the last),
    inside one fragment, across 3+, and one past the end"""
    if claimed is None:
        return [(0, 0), (0, 1)]
    c = claimed
    r = [(0, 0), (c, 0), (0, c), (c, 1)]
    if c:
        r += [(0, 1), (c - 1, 1), (c // 3, min(1000, c - c // 3))]
    if c >= 2 * FRAGMENT:
        r.append((FRAGMENT, FRAGMENT))
    bounds = list(range(FRAGMENT, c - 1, FRAGMENT))
    r += [(b - 1, 2) for b in (bounds if every_boundary else bounds[:1] + bounds[-1:][: len(bounds) - 1])]
    if c > 3 * FRAGMENT:
        r.append((FRAGMENT // 2 + 7, 2 * FRAGMENT + 100))
    return r


def full_result(oracle, s):
    try:
        return 0, oracle.uncompress_np(s)
    except oracle.OracleError as e:
        return e.code, None


# ---------------------------------------------------------------------------------------------- CPU tests
@pytest.fixture(scope="module")
def range_corpus(oracle, tmp_path_factory):
    """the CPU corpus, each stream with its ranges and two side indexes: the oracle's (valid streams) and the stale one
    of its base"""
    d = str(tmp_path_factory.mktemp("range_corpus"))
    cases = corrupt_corpus(oracle, CPU_SEED, 80, max_frags=12)
    files = write_cases(d, cases)
    bases = dict(base_streams(oracle, 12))
    info = []
    for k, ((name, s), f) in enumerate(zip(cases, files)):
        claimed = _claimed(oracle, s)
        rs = ranges_for(claimed, every_boundary=k % 8 == 0)  # each range runs the whole chain on the CPU warp
        with open(f + ".ranges", "w") as fp:
            fp.write("".join("%d %d\n" % r for r in rs))
        idx = {None: None}
        if claimed is not None:
            idx[".sidx"] = _stale_index(oracle, bases[name.split("/")[1]], claimed)
            write_index(f + ".sidx", idx[".sidx"])
            o = oracle_index(oracle, s)
            if o is not None:
                idx[".oidx"] = o
                write_index(f + ".oidx", o)
        info.append((claimed, rs, idx, full_result(oracle, s)))
    exe = build_driver(str(tmp_path_factory.mktemp("range_driver")))
    return cases, files, info, exe


def parse_line(line):
    """(file, offset, length, status, path or None, crc, guard ok) of a `range` line"""
    f, rest = line.split(": range ", 1)
    rng, rest = rest.split(" status ", 1)
    off, length = (int(x) for x in rng.split("+"))
    t = rest.split()
    return f, off, length, int(t[0]), (None if t[2] == "-" else int(t[2])), int(t[4], 16), t[6] == "ok"


def run_range(exe, files, env):
    got = collections.defaultdict(list)
    for line in run_driver(exe, "range", files, env):
        r = parse_line(line)
        got[r[0]].append(r[1:])
    return got


def check_corpus(oracle, range_corpus, suffix, env=None, pick=None):
    cases, files, info, exe = range_corpus
    pick = range(len(cases)) if pick is None else pick
    got = run_range(exe, [files[i] for i in pick], dict(env or {}, **({"IDX_SUFFIX": suffix} if suffix else {})))
    wrong, paths, decided = [], collections.Counter(), 0
    for i in pick:
        (name, s), f, (claimed, rs, idx, full) = cases[i], files[i], info[i]
        lines = got[f]
        assert len(lines) == len(rs), (f, len(lines), len(rs))
        use = idx.get(suffix) if suffix else None
        for (off, length), (goff, glen, st, path, crc, guard) in zip(rs, lines):
            assert (goff, glen) == (off, length)
            want_st, want_b, by_index = expect(oracle, s, claimed, use, off, length, full)
            decided += by_index
            paths[path] += 1
            ok = st == want_st and guard and (st != 0 or crc == zlib.crc32(want_b))
            if by_index:  # e.g. every range of a valid stream under the oracle's index, unless a quirk (a lone
                ok = ok and path == 0  # trailing byte, a zero-length literal) leaves a touched fragment unclean
            if not ok:
                wrong.append("%s %d+%d: status %d path %s guard %s (want %d)" % (name, off, length, st, path, guard, want_st))
    return wrong, paths, decided


@pytest.mark.parametrize("suffix", [None, ".oidx", ".sidx"], ids=["no_index", "oracle_index", "stale_index"])
def test_range_chain_on_the_corpus(oracle, range_corpus, suffix):
    """every corpus stream and range through the range chain on the CPU warp: no index -> the oracle's status and
    slice; an index -> the touched fragments' bytes when they are all clean under it, else the no-index result; no
    sentinel around the output or the scratch slot changes"""
    # the index-free chain parses the whole stream for every range: every second stream keeps the CPU time in bounds
    pick = None if suffix == ".oidx" else range(0, len(range_corpus[0]), 2)
    wrong, paths, decided = check_corpus(oracle, range_corpus, suffix, pick=pick)
    print("paths", dict(paths), "decided by the index", decided)
    assert not wrong, "\n".join(wrong[:20])
    if suffix is None:
        assert paths[0] == 0 and paths[1] >= 100 and paths[2] + paths[3] >= 10, paths
    else:
        assert paths[0] >= 100 and decided >= 100, (paths, decided)
    if suffix == ".sidx":  # the stale index reaches both sides of the rule
        assert paths[1] >= 50 and paths[2] + paths[3] >= 10, paths


@pytest.mark.parametrize("pshift", ["9", "12"])
def test_range_chain_parse_chunk_variants(oracle, range_corpus, pshift):
    cases = range_corpus[0]
    pick = [i for i in range(len(cases)) if i % 16 == 1]
    for suffix in (None, ".sidx"):
        wrong, _, _ = check_corpus(oracle, range_corpus, suffix, {"PSHIFT": pshift}, pick)
        assert not wrong, "\n".join(wrong[:20])


def test_trailing_byte_is_checked_against_the_kernel_rule(oracle, range_corpus):
    """a valid stream with a lone trailing byte: the reference skips the byte (src/internal.jl:416), so the oracle
    accepts the last fragment on its own, but its index entry ends behind an element boundary, so the kernel's rule
    rejects it -- ranges in that fragment take the no-index chain and still read the reference's bytes"""
    cases, files, info, exe = range_corpus
    hits = [i for i, (name, _) in enumerate(cases) if "trailing" in name and ".oidx" in info[i][2]]
    assert hits, "the corpus has no valid stream with a trailing byte"
    for i in hits:
        s, (claimed, rs, idx, full) = cases[i][1], info[i]
        o = idx[".oidx"]
        last = (claimed + FRAGMENT - 1) // FRAGMENT - 1
        hdr = oracle.parse32(s, 0)[1]
        on = claimed - last * FRAGMENT
        assert len(oracle.uncompress(oracle.encode32(on) + bytes(s[o[last]: o[last + 1]]))) == on
        assert not fragment_clean(s, o, last, hdr, claimed)
        lines = run_range(exe, [files[i]], {"IDX_SUFFIX": ".oidx"})[files[i]]
        for (off, length), (_, _, st, path, crc, guard) in zip(rs, lines):
            if length and last in touched(off, length) and off + length <= claimed:
                assert st == 0 and path != 0 and guard and crc == zlib.crc32(bytes(full[1][off: off + length]))


# ---------------------------------------------------------------------------------------------- GPU tests
GUARD = 4096


def _dev(torch, s):
    return torch.from_numpy(np.frombuffer(bytes(s), dtype=np.uint8).copy()).cuda() if len(s) else \
        torch.empty(0, dtype=torch.uint8, device="cuda")


def _path(snappy):
    return snappy._abi.lib().snappy_b200_get_option(b"last_decode_path")


def read_range(snappy, device, torch, d, off, length, index=None):
    """(status, bytes or None, guards intact) of uncompress_range_device into a view between guard regions"""
    buf = torch.full((length + 2 * GUARD,), 0xEE, dtype=torch.uint8, device="cuda")
    try:
        got = device.uncompress_range_device(d, off, length, index=index, out=buf[GUARD: GUARD + length])
        st, b = 0, got.cpu().numpy().tobytes()
    except snappy.SnappyError as e:
        st, b = e.status, None
    g = torch.cat([buf[:GUARD], buf[GUARD + length:]]).cpu().numpy()
    return st, b, bool(np.all(g == 0xEE))


def device_full(snappy, device, d):
    try:
        return 0, device.uncompress_device(d).cpu().numpy()
    except snappy.SnappyError as e:
        return e.status, None


def gpu_ranges(claimed, rng, k=3):
    """a handful of the CPU kinds plus k random ranges"""
    r = ranges_for(claimed)
    keep = r[:7] + r[7::max(1, len(r) // 4)]
    if claimed:
        for _ in range(k):
            a = int(rng.integers(0, claimed))
            keep.append((a, int(rng.integers(0, min(claimed - a, 3 * FRAGMENT) + 1))))
    return keep


@pytest.mark.gpu
def test_device_range_matches_uncompress_on_the_corpus(snappy, oracle):
    """the GPU corpus: every range kind without an index, with the oracle's index and with a stale index, against
    uncompress_device's status and slice and the fragment rule; guard regions untouched"""
    import torch
    from snappy_jl_b200 import device
    cases = corrupt_corpus(oracle, GPU_SEED, 160, max_frags=40)
    bases = dict(base_streams(oracle, 40))
    rng = np.random.default_rng(5)
    wrong, paths = [], collections.Counter()
    for name, s in cases:
        claimed = _claimed(oracle, s)
        d = _dev(torch, s)
        full = device_full(snappy, device, d)
        kinds = [("none", None)]
        if claimed is not None:
            kinds.append(("stale", _stale_index(oracle, bases[name.split("/")[1]], claimed)))
            o = oracle_index(oracle, s)
            if o is not None:
                kinds.append(("oracle", o))
        for off, length in gpu_ranges(claimed, rng):
            for what, idx in kinds:
                t = None if idx is None else torch.tensor(idx, dtype=torch.int64, device="cuda")
                st, b, guard = read_range(snappy, device, torch, d, off, length, t)
                want_st, want_b, by_index = expect(oracle, s, claimed, idx, off, length, full)
                p = _path(snappy)
                paths[(what, p)] += 1
                if st != want_st or not guard or (st == 0 and b != want_b) or (by_index and p != 0):
                    wrong.append("%s %s %d+%d: status %d path %d guard %s (want %d)" % (name, what, off, length, st, p,
                                                                                       guard, want_st))
    print("paths", dict(paths))
    assert not wrong, "\n".join(wrong[:20])
    assert paths[("oracle", 0)] >= 100 and paths[("none", 1)] >= 100, paths
    assert paths[("none", 2)] + paths[("none", 3)] >= 10, paths


def _check_stream(snappy, device, torch, s, index, ranges):
    """ranges of one valid stream, with and without its index, against the slice of uncompress_device's output"""
    d = _dev(torch, s)
    full = device.uncompress_device(d)
    bad = []
    for off, length in ranges:
        want_st = BAD_ARGUMENT if off + length > full.numel() else 0
        want = full[off: off + length].cpu().numpy().tobytes() if want_st == 0 else None
        for idx in (None, index) if index is not None else (None,):
            st, b, guard = read_range(snappy, device, torch, d, off, length, idx)
            if st != want_st or b != want or not guard:
                bad.append("%d+%d index %s: status %d guard %s" % (off, length, idx is not None, st, guard))
    return bad


@pytest.mark.gpu
def test_device_range_on_data_files_pyarrow_and_foreign_streams(snappy, oracle):
    """tests/data (the .snappy files as they are, the others compressed on the device with their index), pyarrow's
    streams, block-structured streams and the long-range-copy streams of test_gpu_foreign (merged tiles, one tile for
    the whole stream), and a corrupt one that only the whole-stream chain judges"""
    import torch
    from snappy_jl_b200 import device, synth
    from test_gpu_foreign import _blocky_stream, _copy4, _lit
    rng = np.random.default_rng(11)
    data = os.path.join(ROOT, "tests", "data")
    wrong = []
    for f in sorted(os.listdir(data)):
        raw = open(os.path.join(data, f), "rb").read()
        if f.endswith(".snappy"):
            claimed = _claimed(oracle, raw)
            full = full_result(oracle, raw)
            d = _dev(torch, raw)
            for off, length in gpu_ranges(claimed, rng):
                st, b, guard = read_range(snappy, device, torch, d, off, length)
                want_st, want_b, _ = expect(oracle, raw, claimed, None, off, length, full)
                if st != want_st or b != want_b or not guard:
                    wrong.append("%s %d+%d: status %d (want %d)" % (f, off, length, st, want_st))
            continue
        src = _dev(torch, raw)
        stream, index = device.compress_device(src, want_index=True)
        wrong += [f + " " + w for w in _check_stream(snappy, device, torch, stream.cpu().numpy().tobytes(), index,
                                                     gpu_ranges(len(raw), rng))]
    raw = synth.mix(20, seed=3, tail=555)
    pa = pytest.importorskip("pyarrow")
    s = pa.Codec("snappy").compress(raw.tobytes(), asbytes=True)
    o = oracle_index(oracle, s)
    wrong += ["pyarrow " + w for w in _check_stream(snappy, device, torch, s, None if o is None else
                                                    torch.tensor(o, dtype=torch.int64, device="cuda"),
                                                    gpu_ranges(raw.size, rng, 10))]
    raw = synth.mix(48, seed=17, tail=4321)
    for block in (7777, 50000, 32768):
        s = _blocky_stream(oracle, raw, block)
        wrong += ["blocky %d " % block + w for w in _check_stream(snappy, device, torch, s, None,
                                                                  gpu_ranges(raw.size, rng, 10))]
        assert _path(snappy) == 1
    # long-range copies: tiles merged around them, and a chain that leaves one tile for the whole stream
    g = np.random.default_rng(99)
    for layout in ("merged", "one_tile"):
        parts, out = [], bytearray()

        def lit(n):
            b = g.integers(0, 256, n, dtype=np.uint8).tobytes()
            parts.append(_lit(b))
            out.extend(b)

        def cp(length, offset):
            parts.append(_copy4(length, offset))
            for _ in range(length):
                out.append(out[-offset])
        if layout == "merged":
            for i in range(24):
                lit(50000 + 977 * i)
                if i in (5, 6, 17):
                    cp(64, 300000 + i)
                if i == 11:
                    cp(40, 70000)
                    cp(64, 131072)
        else:
            lit(70000)
            for i in range(40):
                lit(30000)
                cp(64, 65000)
        s = oracle.encode32(len(out)) + b"".join(parts)
        wrong += [layout + " " + w for w in _check_stream(snappy, device, torch, s, None,
                                                          gpu_ranges(len(out), rng, 10))]
        assert _path(snappy) == 1
    # a corrupt stream that no parse can judge alone: validation gives the status of every range
    bad = oracle.encode32(70064) + _lit(bytes(70000)) + _copy4(64, 70001)
    want = oracle.status_of_uncompress(bad)
    for off, length in ((0, 10), (69990, 20), (0, 70064)):
        st, _, guard = read_range(snappy, device, torch, _dev(torch, bad), off, length)
        if st != want or not guard:
            wrong.append("bad %d+%d: status %d (want %d)" % (off, length, st, want))
    assert not wrong, "\n".join(wrong[:20])


@pytest.mark.gpu
def test_device_range_on_a_1_gib_stream(snappy, oracle):
    """a 1 GiB synth.mix stream: 200 seeded random ranges with and without its index against the full decode; the
    indexed reads take path 0 and one launch"""
    import torch
    from snappy_jl_b200 import device, synth
    raw = torch.from_numpy(synth.mix(16384, seed=2)).cuda()
    stream, index = device.compress_device(raw, want_index=True)
    n = raw.numel()
    rng = np.random.default_rng(200)
    wrong = []
    for k in range(200):
        length = int(rng.choice([1, 4096, 65536, 1 << 20, 64 << 20]) if k % 2 else rng.integers(0, 300000))
        off = int(rng.integers(0, n - length + 1))
        want = raw[off: off + length]
        for idx in (index, None):
            buf = torch.full((length + 2 * GUARD,), 0xEE, dtype=torch.uint8, device="cuda")
            got = device.uncompress_range_device(stream, off, length, index=idx, out=buf[GUARD: GUARD + length])
            guard = bool((buf[:GUARD] == 0xEE).all() and (buf[GUARD + length:] == 0xEE).all())
            if not torch.equal(got, want) or not guard:
                wrong.append("%d+%d index %s" % (off, length, idx is not None))
            if idx is not None and length and (_path(snappy) != 0 or device.last_launch_count(1) != 1):
                wrong.append("%d+%d: path %d launches %d" % (off, length, _path(snappy), device.last_launch_count(1)))
    assert not wrong, "\n".join(wrong[:20])


@pytest.mark.gpu
def test_range_huge_claim_bad_ranges_and_bad_header(snappy):
    """a 20-byte stream that claims 4 GiB: its status (INVALID_INPUT) with and without a garbage index, and no
    allocation near the claimed length; offset + length > claimed -> BAD_ARGUMENT; a bad header -> BAD_VARINT first"""
    import torch
    from snappy_jl_b200 import device
    hdr = bytes([0xFF, 0xFF, 0xFF, 0xFF, 0x0F])
    lit = hdr + bytes([13 << 2]) + bytes(range(14))
    d = _dev(torch, lit)
    garbage = torch.tensor(list(range(0, 65537 * 3, 3)), dtype=torch.int64, device="cuda")
    torch.cuda.synchronize()
    free0, _ = torch.cuda.mem_get_info()
    for idx in (None, garbage):
        for off, length in ((0, 14), (0, 100), (1 << 31, 4096), (0xFFFFFFFF - 10, 10)):
            st, _, guard = read_range(snappy, device, torch, d, off, length, idx)
            assert st == 2 and guard, (off, length, idx is not None, st)
        assert read_range(snappy, device, torch, d, 0xFFFFFFFF, 1, idx)[0] == BAD_ARGUMENT
    free1, _ = torch.cuda.mem_get_info()
    assert free0 - free1 < 256 << 20, (free0, free1)
    good = _dev(torch, bytes([10, 9 << 2]) + b"abcdefghij")
    assert read_range(snappy, device, torch, good, 3, 7)[:2] == (0, b"defghij")
    assert read_range(snappy, device, torch, good, 3, 8)[0] == BAD_ARGUMENT
    assert read_range(snappy, device, torch, good, 11, 0)[0] == BAD_ARGUMENT
    assert read_range(snappy, device, torch, _dev(torch, bytes([0x80, 0x80])), 1 << 40, 5)[0] == BAD_VARINT
    assert read_range(snappy, device, torch, _dev(torch, b""), 0, 0)[0] == BAD_VARINT


@pytest.mark.gpu
def test_batched_ranges_match_the_single_call(snappy, oracle):
    """4096 requests over valid and corrupt streams, without an index, with the right and a wrong index, several on
    one stream: each request's status and bytes equal the single call's; the indexed clean requests take one launch"""
    import torch
    from snappy_jl_b200 import device, synth
    raw = [synth.mix(k, seed=40 + k, tail=123 * k) for k in (3, 17, 40)]
    streams, indexes = [], []
    for r in raw:
        s, i = device.compress_device(torch.from_numpy(r).cuda(), want_index=True)
        streams.append(s.clone())
        indexes.append(i)
    bad = streams[1].clone()
    bad[bad.numel() // 2: bad.numel() // 2 + 30] ^= 0x5A
    streams.append(bad)
    indexes.append(indexes[1])
    wrong_idx = indexes[2][: indexes[1].numel()].clone()
    rng = np.random.default_rng(4096)
    reqs = []
    for k in range(4096):
        j = int(rng.integers(0, len(streams)))
        claimed = [r.size for r in raw][min(j, 2)] if j < 3 else raw[1].size
        length = int(rng.choice([0, 1, 100, 4096, 70000, 200000]))
        length = min(length, claimed)
        off = int(rng.integers(0, claimed - length + 1)) if k % 97 else claimed + 1
        kind = k % 3
        idx = None if kind == 0 else (indexes[j] if kind == 1 else (wrong_idx if j == 1 else indexes[j]))
        reqs.append((j, off, length, idx))
    outs, statuses = device.uncompress_ranges_device([streams[r[0]] for r in reqs], [r[1] for r in reqs],
                                                     [r[2] for r in reqs], [r[3] for r in reqs])
    mism = []
    for k, (j, off, length, idx) in enumerate(reqs):
        st, b, _ = read_range(snappy, device, torch, streams[j], off, length, idx)
        if statuses[k] != st or (st == 0 and outs[k].cpu().numpy().tobytes() != b):
            mism.append("request %d (stream %d, %d+%d, index %s): status %d, single %d" % (k, j, off, length,
                                                                                         idx is not None, statuses[k], st))
    assert not mism, "\n".join(mism[:20])
    assert collections.Counter(statuses)[0] > 2000 and any(s not in (0, BAD_ARGUMENT) for s in statuses)
    clean = [r for r in reqs if r[3] is not None and r[0] != 3 and r[3] is indexes[r[0]] and r[1] + r[2] <= raw[min(r[0], 2)].size]
    outs, statuses = device.uncompress_ranges_device([streams[r[0]] for r in clean], [r[1] for r in clean],
                                                     [r[2] for r in clean], [r[3] for r in clean])
    assert set(statuses) == {0} and device.last_launch_count(1) == 1 and _path(snappy) == 0
    for (j, off, length, _), o in zip(clean, outs):
        assert o.cpu().numpy().tobytes() == raw[j][off: off + length].tobytes()


def _ranges_raw(torch, snappy, streams, lens_in, offsets, lengths, indexes):
    """snappy_b200_uncompress_ranges_device called directly: streams[i] may be None (a NULL pointer with lens_in[i]
    bytes); every output between guard regions.  Returns (statuses, bytes per request, guards intact)."""
    import ctypes
    count = len(streams)
    bufs = [torch.full((n + 2 * GUARD,), 0xEE, dtype=torch.uint8, device="cuda") for n in lengths]
    ptr = lambda t: t.data_ptr() if t is not None else 0
    statuses = (ctypes.c_int * count)()
    rc = snappy._abi.lib().snappy_b200_uncompress_ranges_device(
        (ctypes.c_void_p * count)(*[ptr(s) for s in streams]), (ctypes.c_size_t * count)(*lens_in),
        (ctypes.c_void_p * count)(*[ptr(i) for i in indexes]), (ctypes.c_uint64 * count)(*offsets),
        (ctypes.c_size_t * count)(*lengths), (ctypes.c_void_p * count)(*[b.data_ptr() + GUARD for b in bufs]), count,
        statuses, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    assert rc == 0, rc
    got = [b[GUARD: GUARD + n].cpu().numpy().tobytes() for b, n in zip(bufs, lengths)]
    guard = all(bool((b[:GUARD] == 0xEE).all() and (b[GUARD + n:] == 0xEE).all()) for b, n in zip(bufs, lengths))
    return list(statuses), got, guard


@pytest.mark.gpu
def test_small_batches_on_a_fresh_context_and_a_null_stream(snappy):
    """batches of 1, 3 and 5 indexed reads at unaligned offsets right after the contexts are released (the first
    launch sizes the scratch slots: one per launched warp, also when the warp count is odd), and a batch with a NULL
    stream pointer of non-zero length: BAD_ARGUMENT for that request, the others read as usual"""
    import torch
    from snappy_jl_b200 import device, synth
    raw = synth.mix(12, seed=77, tail=999)
    d = torch.from_numpy(raw).cuda()
    stream, index = device.compress_device(d, want_index=True)
    stream = stream.clone()
    n = raw.size
    for count in (1, 3, 5):
        snappy._abi.lib().snappy_b200_shutdown()
        offs = [FRAGMENT * (2 * k) + 1234 + 17 * k for k in range(count)]
        lengths = [4096 + 100 * k for k in range(count)]
        st, got, guard = _ranges_raw(torch, snappy, [stream] * count, [stream.numel()] * count, offs, lengths,
                                     [index] * count)
        assert st == [0] * count and guard, (count, st, guard)
        assert device.last_launch_count(1) == 1
        for b, o, length in zip(got, offs, lengths):
            assert b == raw[o: o + length].tobytes()
        assert device.uncompress_range_device(stream, n - 5, 5).cpu().numpy().tobytes() == raw[n - 5:].tobytes()
    st, got, guard = _ranges_raw(torch, snappy, [stream, None, stream], [stream.numel(), 100, stream.numel()],
                                 [70000, 0, 3], [5000, 10, 0], [index, None, None])
    assert st == [0, BAD_ARGUMENT, 0] and guard, st
    assert got[0] == raw[70000: 75000].tobytes()
    assert device.uncompress_range_device(stream, 0, 10, index=index).cpu().numpy().tobytes() == raw[:10].tobytes()


@pytest.mark.gpu
def test_wrapper_rejects_a_short_index_and_a_wrong_output(snappy):
    import torch
    from snappy_jl_b200 import device, synth
    raw = synth.mix(5, seed=78)
    stream, index = device.compress_device(torch.from_numpy(raw).cuda(), want_index=True)
    with pytest.raises(ValueError):
        device.uncompress_range_device(stream, 0, 10, index=index[:-1].clone())
    with pytest.raises(ValueError):
        device.uncompress_ranges_device([stream, stream], [0, 5], [10, 10], [index, index[:3].clone()])
    with pytest.raises(ValueError):
        device.uncompress_range_device(stream, 0, 10, out=torch.empty(10, dtype=torch.int32, device="cuda"))
    with pytest.raises(ValueError):
        device.uncompress_range_device(stream, 0, 10, out=torch.empty(10, dtype=torch.uint8))
    outs, st = device.uncompress_ranges_device([stream, stream], [0, 70000], [10, 3000], [index, None])
    assert st == [0, 0] and outs[1].cpu().numpy().tobytes() == raw[70000: 73000].tobytes()
