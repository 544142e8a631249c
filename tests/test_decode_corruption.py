"""Status parity on corrupt and quirky multi-fragment streams, on every decode path.

The decoder promises the reference's status for ANY input, and the reference's bytes when that status is OK
(include/snappy_b200.h).  For a stream longer than one 64 KiB fragment and without a side index, that status comes out
of a chain of parallel steps: the relaxed parse and its first-error rule (k_build_index), the PF_ANOMALY / PF_BROKEN ->
k_first_missing -> tvalid logic of decode_parsed_locked, the tile flags of k_decode_fragments and the bounded serial
walk over the rejected tiles (k_decode_serial_tiles).  k_decode_pages makes the same promise per Parquet page.

`corrupt_corpus` builds a few hundred streams from base streams of several fragments (random faults, faults aimed at
the 64 KiB boundaries, truncations, header lies, two faults in both orders, and valid streams with the quirks the
reference accepts); the oracle (oracle/snappy_oracle.c) gives every case its status and bytes.

CPU: the kernel sources run on the CPU warp (tools/cpu_warp/run_decode_parsed.cpp), launched as the host code
launches them.  GPU (-m gpu): the device API without an index, with a stale index, the host API, the option variants,
batched pages and the streamed host path.  `last_decode_path`: 1 parse + tiles, 2 parse + tiles + bounded serial walk,
3 whole-stream serial decoder."""
import collections
import concurrent.futures
import os
import subprocess

import numpy as np
import pytest

from conftest import ROOT, read_data

FRAGMENT = 65536
CATEGORIES = ("random", "targeted", "truncate", "header", "two_faults", "accepted")
ZERO_LITERAL = bytes([0xFC, 0xFF, 0xFF, 0xFF, 0xFF])  # 1 + 0xFFFFFFFF wraps to a literal of 0 bytes
CPU_SEED, GPU_SEED = 20261020, 4242


# ---------------------------------------------------------------------------------------------- the corpus
class Elements:
    """the element chain of a VALID stream: stream position, output position, length, copy offset (0: literal),
    header bytes (tag + extra) of every element"""

    def __init__(self, stream, oracle):
        s = np.frombuffer(stream, dtype=np.uint8)
        claimed, hdr = oracle.parse32(stream, 0)
        self.hdr, self.claimed = hdr, claimed
        ips, ops, lens, offs, heads = [], [], [], [], []
        ip, op, L = hdr, 0, s.size
        while ip + 1 < L:
            c = int(s[ip])
            kind = c & 3
            if kind == 0:
                n = c >> 2
                extra = n - 59 if n >= 60 else 0
                length = (int.from_bytes(s[ip + 1: ip + 1 + extra].tobytes(), "little") if extra else n) + 1
                off = 0
            elif kind == 1:
                extra, length, off = 1, 4 + ((c >> 2) & 7), ((c >> 5) << 8) | int(s[ip + 1])
            else:
                extra = 2 if kind == 2 else 4
                length, off = (c >> 2) + 1, int.from_bytes(s[ip + 1: ip + 1 + extra].tobytes(), "little")
            ips.append(ip)
            ops.append(op)
            lens.append(length)
            offs.append(off)
            heads.append(1 + extra)
            ip += 1 + extra + (length if off == 0 else 0)
            op += length
        assert op == claimed
        self.ip, self.op, self.len = np.array(ips), np.array(ops), np.array(lens)
        self.off, self.head = np.array(offs), np.array(heads)

    def covering(self, out_pos):
        """index of the element whose output covers out_pos"""
        return int(np.searchsorted(self.op, out_pos, side="right")) - 1

    def boundaries(self):
        return [self.covering(f * FRAGMENT) for f in range(1, (self.claimed + FRAGMENT - 1) // FRAGMENT)]


def _blocky_stream(oracle, raw, block):
    """every `block` bytes compressed on their own, concatenated behind one header: a valid stream whose elements
    straddle the 64 KiB boundaries wherever the block size does not divide 65536 (as in test_gpu_foreign.py)"""
    parts = [oracle.encode32(raw.size)]
    for o in range(0, raw.size, block):
        s = oracle.compress(raw[o: o + block].tobytes())
        _, k = oracle.parse32(s, 0)
        parts.append(s[k:])
    return b"".join(parts)


def base_streams(oracle, max_frags):
    """(name, stream) of valid streams of 2 .. max_frags fragments"""
    from snappy_jl_b200 import synth
    small = max(2, max_frags // 4)
    bases = [("mix_small", oracle.compress(synth.mix(2, seed=5, tail=777).tobytes())),
             ("mix_large", oracle.compress(synth.mix(max_frags - 1, seed=6, tail=4321).tobytes())),
             ("html_x_4", oracle.compress(read_data("html_x_4"))),
             ("urls", oracle.compress(read_data("urls.10K")[: max_frags * FRAGMENT - 1000])),
             # 64 KiB literals: the tile boundaries and the parse chunks fall inside literals
             ("random", oracle.compress(np.random.default_rng(7).integers(0, 256, small * FRAGMENT + 1234, dtype=np.uint8).tobytes())),
             # long overlapping copies
             ("zeros", oracle.compress(bytes(small * FRAGMENT + 100)))]
    raw = synth.mix(min(6, max_frags), seed=8, tail=999)
    try:
        import pyarrow as pa
        bases.append(("pyarrow_mix", pa.Codec("snappy").compress(raw.tobytes(), asbytes=True)))
    except ImportError:
        pass
    bases += [("blocky_7777", _blocky_stream(oracle, raw, 7777)), ("blocky_50000", _blocky_stream(oracle, raw, 50000))]
    return bases


def _with_header(oracle, stream, hdr, claimed):
    return oracle.encode32(claimed) + stream[hdr:]


def _insert(oracle, el, stream, at_elem, data, grow=0):
    """`data` spliced in front of element at_elem; the header grows by `grow` output bytes"""
    p = int(el.ip[at_elem])
    return _with_header(oracle, stream[:p] + data + stream[p:], el.hdr, el.claimed + grow)


def corrupt_corpus(oracle, seed, count, max_frags=40):
    """[(name, stream)] -- deterministic for a seed.  `count` random faults (spread over the base streams) plus the
    targeted, truncated, header-lie, two-fault and accepted cases of every base stream.  The name is
    "<category>/<base>/<what>"; `category(name)` gives the category back."""
    rng = np.random.default_rng(seed)
    bases = base_streams(oracle, max_frags)
    cases = []
    for bi, (bname, s) in enumerate(bases):
        cases += mutations(oracle, rng, bname, s, range(bi, count, len(bases)))
    return cases


def mutations(oracle, rng, bname, s, randoms):
    """the corpus cases made from one valid stream `s`; `randoms`: the labels of its random faults"""
    cases = []

    def put(cat, base, what, data):
        cases.append(("%s/%s/%s" % (cat, base, what), bytes(data)))

    el = Elements(s, oracle)
    a = np.frombuffer(s, dtype=np.uint8)
    L, hdr = a.size, el.hdr
    bnd = el.boundaries()
    picks = sorted({0, len(bnd) // 2, len(bnd) - 1}) if bnd else []
    lits = np.nonzero((el.off == 0) & (el.len > 200))[0]
    copies = np.nonzero(el.off > 0)[0]

    def flip(data, pos):
        data = bytearray(data)
        data[pos] ^= int(rng.integers(1, 256))
        return data

    def zero_offset(data, e):
        """copy element e with offset 0 (src/internal.jl:499)"""
        data, p = bytearray(data), int(el.ip[e])
        if data[p] & 3 == 1:
            data[p] &= 0x1F  # the offset's high bits live in the tag
        data[p + 1: p + int(el.head[e])] = bytes(int(el.head[e]) - 1)
        return bytes(data)

    # ---- random: 1-3 byte flips, XOR-garbled runs of 1-24 bytes (the header is left alone: see "header")
    for r in (randoms if L - hdr > 25 else ()):
        if r % 2 == 0:
            d = bytearray(s)
            for _ in range(int(rng.integers(1, 4))):
                d = flip(d, int(rng.integers(hdr, L)))
            put("random", bname, "flips%d" % r, d)
        else:
            d = a.copy()
            n = int(rng.integers(1, 25))
            p = int(rng.integers(hdr, L - n))
            d[p: p + n] ^= np.uint8(int(rng.integers(1, 256)))
            put("random", bname, "garble%d_%d" % (r, n), d)
    # ---- targeted: the element at a 64 KiB boundary and the bytes around it; tile 0, last tile, long literal
    for k in picks:
        e = bnd[k]
        for d in (-1, 0, 1):
            put("targeted", bname, "boundary%d%+d" % (k + 1, d), flip(s, int(el.ip[e]) + d))
    if L > hdr:
        put("targeted", bname, "tile0", flip(s, int(rng.integers(hdr, int(el.ip[bnd[0]]) if bnd else L))))
        put("targeted", bname, "last_tile", flip(s, int(rng.integers(int(el.ip[bnd[-1]]) if bnd else hdr, L))))
    if lits.size:
        e = int(lits[len(lits) // 2])
        inside = int(el.ip[e]) + int(el.head[e]) + int(el.len[e]) // 2
        put("targeted", bname, "literal_bytes", flip(s, inside))          # valid: other bytes
        put("targeted", bname, "literal_len", flip(s, int(el.ip[e]) + 1))  # its length field
    if copies.size:  # a copy offset of 0 in the last tile
        put("targeted", bname, "copy_offset0", zero_offset(s, int(copies[-1])))
    put("targeted", bname, "two_trailing_bytes", s + b"\x01\x02")  # a 4-byte copy with no room left: status 4
    # ---- truncation: at / one before / one after a boundary element, inside a long literal, inside the header
    for k in picks[:2]:
        p = int(el.ip[bnd[k]])
        for d in (-1, 0, 1):
            put("truncate", bname, "boundary%d%+d" % (k + 1, d), s[: p + d])
    if lits.size:
        e = int(lits[-1])
        put("truncate", bname, "in_literal", s[: int(el.ip[e]) + int(el.head[e]) + int(el.len[e]) // 2])
    put("truncate", bname, "in_header", s[: hdr - 1])
    put("truncate", bname, "header_only", s[:hdr])
    put("truncate", bname, "header_plus_1", s[: hdr + 1])
    # ---- header lies
    for d in (1, -1, 3, -3, FRAGMENT, -FRAGMENT):
        if 0 <= el.claimed + d < 1 << 32:
            put("header", bname, "claimed%+d" % d, _with_header(oracle, s, hdr, el.claimed + d))
    put("header", bname, "claimed0", _with_header(oracle, s, hdr, 0))
    # ---- two faults: one only the serial walk can judge, one the parse sees, in both orders
    late = copies[copies > (bnd[-1] if bnd else 0)] if copies.size else copies
    early = bnd[0] if bnd else 1
    if late.size and early < el.ip.size:
        zero_off = zero_offset(s, int(late[len(late) // 2]))
        put("two_faults", bname, "zero_literal_then_offset0", _insert(oracle, el, zero_off, early, ZERO_LITERAL))
        put("two_faults", bname, "long_literal_then_offset0",
            _insert(oracle, el, zero_off, early, bytes([62 << 2, 0xFF, 0xFF, 0x7F])))
    if copies.size:
        last = bnd[-1] if bnd else el.ip.size - 1
        put("two_faults", bname, "offset0_then_zero_literal", _insert(oracle, el, zero_offset(s, int(copies[0])), last, ZERO_LITERAL))
    # ---- streams the reference accepts
    put("accepted", bname, "trailing_byte", s + b"\x07")
    if bnd:
        put("accepted", bname, "zero_literal_at_tile_start", _insert(oracle, el, s, bnd[len(bnd) // 2], ZERO_LITERAL))
        mid = el.covering((len(bnd) // 2) * FRAGMENT + FRAGMENT // 2)
        put("accepted", bname, "zero_literal_mid_tile", _insert(oracle, el, s, mid, ZERO_LITERAL))
        # a copy whose offset is exactly its output position (reads from byte 0)
        e = el.covering(FRAGMENT + 1000)
        op = int(el.op[e])
        if op > 0:
            put("accepted", bname, "copy_offset_eq_pos", _insert(oracle, el, s, e, bytes([(40 - 1) << 2 | 3]) + op.to_bytes(4, "little"), 40))
        # a literal that straddles a boundary
        e = el.covering(len(bnd) * FRAGMENT - 80)
        put("accepted", bname, "straddling_literal",
            _insert(oracle, el, s, e, bytes([(61 << 2), 299 & 0xFF, 299 >> 8]) + rng.integers(0, 256, 300, dtype=np.uint8).tobytes(), 300))
    if copies.size:  # 2-byte-offset copies re-encoded with 4-byte offsets (same output)
        d, last = bytearray(), 0
        for e in copies[:: max(1, copies.size // 40)]:
            e = int(e)
            if int(el.head[e]) != 3:
                continue
            p = int(el.ip[e])
            d += s[last:p] + bytes([((int(el.len[e]) - 1) << 2) | 3]) + int(el.off[e]).to_bytes(4, "little")
            last = p + 3
        if last:
            put("accepted", bname, "copy4", bytes(d) + s[last:])
    return cases


def category(name):
    return name.split("/", 1)[0]


# ---------------------------------------------------------------------------------------------- the CPU warp driver
def build_driver(d):
    exe, obj = os.path.join(d, "run_decode_parsed"), os.path.join(d, "oracle.o")
    subprocess.check_call(["gcc", "-O2", "-c", "-o", obj, os.path.join(ROOT, "oracle", "snappy_oracle.c")])
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-DSB200_CPU_EMU", "-DSB200_EXPERIMENTS", "-I" + os.path.join(ROOT, "tools", "cpu_warp"),
                           "-o", exe, os.path.join(ROOT, "tools", "cpu_warp", "run_decode_parsed.cpp"), obj])
    return exe


def write_cases(d, cases):
    files = []
    for i, (name, data) in enumerate(cases):
        p = os.path.join(d, "c%04d_%s.snappy" % (i, name.replace("/", "__")))
        with open(p, "wb") as f:
            f.write(data)
        files.append(p)
    return files


def run_driver(exe, mode, files, env=None, jobs=None):
    """the driver over `files`, split over the CPU's cores; returns its lines in file order"""
    jobs = jobs or min(len(files), os.cpu_count() or 1)
    groups = [files[k::jobs] for k in range(jobs)]

    def one(group):
        p = subprocess.run([exe, mode] + group, env=dict(os.environ, **(env or {})), capture_output=True, text=True)
        return p

    with concurrent.futures.ThreadPoolExecutor(jobs) as ex:
        results = list(ex.map(one, groups))
    by_file, lines = {}, []
    for group, p in zip(groups, results):
        got = p.stdout.splitlines()
        assert p.returncode in (0, 1) and len(got) >= len(group), p.stdout[-2000:] + p.stderr[-2000:]
        if mode == "parsed":  # one line per file, in order
            by_file.update(zip(group, got))
        lines += got
    return [by_file[f] for f in files] if mode == "parsed" else lines


def driver_path(line):
    tok = line.split(" path ", 1)[1].split(":", 1)[0].split()[0]
    return None if tok == "-" else int(tok)


@pytest.fixture(scope="module")
def cpu_corpus(oracle, tmp_path_factory):
    d = str(tmp_path_factory.mktemp("corrupt_corpus"))
    cases = corrupt_corpus(oracle, CPU_SEED, 80, max_frags=12)
    return d, cases, write_cases(d, cases)


@pytest.fixture(scope="module")
def driver(tmp_path_factory):
    return build_driver(str(tmp_path_factory.mktemp("decode_parsed")))


def subset(cases, per_category=10):
    """a fixed subset that covers every category (and every base stream within it, as far as it goes)"""
    seen = collections.Counter()
    out = []
    for i, (name, _) in enumerate(cases):
        if seen[category(name)] < per_category and (i % 3 == 0 or category(name) in ("two_faults", "accepted")):
            seen[category(name)] += 1
            out.append(i)
    return out


# ---------------------------------------------------------------------------------------------- CPU tests
def test_corpus_is_deterministic_and_its_quirks_hold(oracle):
    """same seed, same corpus; the accepted quirks decode OK in the oracle, the two-fault cases fail, and the oracle's
    word on the two quirks of src/internal.jl:416 and :462 is what the corpus relies on"""
    a = corrupt_corpus(oracle, 1, 20, max_frags=3)
    b = corrupt_corpus(oracle, 1, 20, max_frags=3)
    assert a == b
    assert {category(n) for n, _ in a} == set(CATEGORIES)
    for name, s in a:
        st = oracle.status_of_uncompress(s)
        if category(name) == "accepted":
            assert st == 0, name
        if category(name) == "two_faults":
            assert st != 0, name
    s = oracle.compress(bytes(range(256)) * 600)
    assert oracle.status_of_uncompress(s + b"\x00") == 0
    assert oracle.status_of_uncompress(s + b"\x01\x02") == 4   # a copy of 4 bytes with no room left
    _, hdr = oracle.parse32(s, 0)
    assert oracle.uncompress(s[:hdr] + ZERO_LITERAL + s[hdr:]) == bytes(range(256)) * 600


def test_parsed_decode_matches_oracle_on_the_corpus(oracle, driver, cpu_corpus):
    """the whole CPU corpus through the index-free chain (clean cuts on, 1 KiB parse chunks): the oracle's status on
    every stream, its bytes on OK, nothing written behind `claimed`; and the corpus still reaches every path and every
    failure status, so it cannot silently decay into one that tests nothing"""
    d, cases, files = cpu_corpus
    lines = run_driver(driver, "parsed", files)
    bad = [l for l in lines if "0 mismatches" not in l]
    assert not bad, "\n".join(bad[:20])
    paths = collections.Counter(driver_path(l) for l in lines)
    statuses = collections.Counter(oracle.status_of_uncompress(s) for _, s in cases)
    cats = collections.Counter(category(n) for n, _ in cases)
    print("paths", dict(paths), "statuses", dict(statuses), "categories", dict(cats))
    for p in (1, 2, 3):
        assert paths[p] >= 5, (p, paths)
    for st in (0, 2, 3, 4, 5, 6):
        assert statuses[st] >= 5, (st, statuses)
    # the streams only the serial walk can judge really get there
    assert all(driver_path(l) == 2 for (n, _), l in zip(cases, lines) if "zero_literal_then" in n), "zero literal"
    assert 250 <= len(cases) <= 600


@pytest.mark.parametrize("env", [{"CLEAN_CUTS": "0"}, {"PSHIFT": "9"}, {"PSHIFT": "12"}],
                         ids=["clean_cuts0", "pshift9", "pshift12"])
def test_parsed_decode_variants_match_oracle(driver, cpu_corpus, env):
    """parse_chunk_log2 9 and 12 (parse chunks of 512 B / 4 KiB), and tiles on the 64 KiB boundaries instead of the
    clean cuts, on a fixed subset that covers every category"""
    d, cases, files = cpu_corpus
    pick = subset(cases)
    assert {category(cases[i][0]) for i in pick} == set(CATEGORIES)
    lines = run_driver(driver, "parsed", [files[i] for i in pick], env)
    bad = [l for l in lines if "0 mismatches" not in l]
    assert not bad, "\n".join(bad[:20])


def test_page_decoder_matches_oracle_on_the_corpus(driver, cpu_corpus):
    """every corpus stream as one page of k_decode_pages (status, out_size, bytes on OK, nothing written at or past
    out_cap), every fourth page with a slot one byte short, and empty pages"""
    d, cases, files = cpu_corpus
    lines = run_driver(driver, "pages", files)
    bad = [l for l in lines if "0 mismatches" not in l]
    assert not bad, "\n".join(bad[:20])
    assert len(lines) >= len(files)
    assert sum("status 7 (oracle 7)" in l for l in lines) >= 20
    assert sum("(empty page)" in l and "status 6 (oracle 6)" in l for l in lines) >= 2


# ---------------------------------------------------------------------------------------------- GPU tests
def _path(snappy):
    return snappy._abi.lib().snappy_b200_get_option(b"last_decode_path")


def _expect(oracle, s):
    """(status, bytes or None) of the oracle"""
    try:
        return 0, oracle.uncompress_np(s)
    except oracle.OracleError as e:
        return e.code, None


def _claimed(oracle, s):
    try:
        return oracle.parse32(s, 0)[0]
    except oracle.OracleError:
        return None


def _device_decode(snappy, device, torch, s, claimed, index=None):
    """(status, bytes, sentinels behind claimed intact) of device.uncompress_device"""
    d = torch.from_numpy(np.frombuffer(s, dtype=np.uint8).copy()).cuda() if s else torch.empty(0, dtype=torch.uint8, device="cuda")
    n = (claimed or 0) + 256
    out = torch.full((n,), 0xEE, dtype=torch.uint8, device="cuda")
    try:
        got = device.uncompress_device(d, out=out, index=index)
        st, data = 0, got.cpu().numpy()
    except snappy.SnappyError as e:
        st, data = e.status, None
    tail = out[(claimed or 0):].cpu().numpy()
    return st, data, bool(np.all(tail == 0xEE))


def _stale_index(oracle, base, claimed):
    """the side index of the unmutated base stream (element start at every 64 KiB output boundary), stretched or cut
    to the fragment count the mutated header claims"""
    el = Elements(base, oracle)
    idx = [el.hdr] + [int(el.ip[e]) for e in el.boundaries()]
    nfrag = (claimed + FRAGMENT - 1) // FRAGMENT
    idx = (idx + [len(base)] * (nfrag + 1))[: nfrag] + [len(base)]
    return idx


@pytest.fixture(scope="module")
def gpu_corpus(oracle):
    cases = corrupt_corpus(oracle, GPU_SEED, 160, max_frags=40)
    want = [_expect(oracle, s) for _, s in cases]
    return cases, want


@pytest.mark.gpu
def test_device_decode_matches_oracle_and_cpu_paths(snappy, oracle, tmp_path):
    """the CPU corpus's fixed subset (every category) through device.uncompress_device without an index: the oracle's
    status and bytes, no byte written behind `claimed`, and last_decode_path equal to the CPU driver's path for the
    same stream (drift between decode_parsed_locked and its mirror shows here)"""
    import torch
    from snappy_jl_b200 import device
    cases = corrupt_corpus(oracle, CPU_SEED, 80, max_frags=12)
    cases = [cases[i] for i in subset(cases, per_category=15)]
    exe = build_driver(str(tmp_path))
    lines = run_driver(exe, "parsed", write_cases(str(tmp_path), cases))
    wrong = []
    for (name, s), line in zip(cases, lines):
        want_st, want = _expect(oracle, s)
        claimed = _claimed(oracle, s)
        st, got, guard = _device_decode(snappy, device, torch, s, claimed)
        ok = st == want_st and guard and (st != 0 or np.array_equal(got, want))
        if claimed is not None and driver_path(line) is not None:
            ok = ok and _path(snappy) == driver_path(line)
        if not ok:
            wrong.append("%s: status %d (oracle %d) path %d, cpu: %s, guard %s" % (name, st, want_st, _path(snappy), line, guard))
    assert not wrong, "\n".join(wrong[:20])


@pytest.mark.gpu
def test_device_decode_matches_oracle_on_the_full_corpus(snappy, oracle, gpu_corpus):
    """the 2-40 fragment corpus through the device API without an index, with the stale side index of the unmutated
    base stream (it must fall back and change nothing), and through the host API"""
    import torch
    from snappy_jl_b200 import device
    cases, want = gpu_corpus
    bases = dict(base_streams(oracle, 40))
    wrong = []
    paths = collections.Counter()
    for (name, s), (want_st, want_b) in zip(cases, want):
        claimed = _claimed(oracle, s)
        st, got, guard = _device_decode(snappy, device, torch, s, claimed)
        paths[_path(snappy)] += 1
        if st != want_st or not guard or (st == 0 and not np.array_equal(got, want_b)):
            wrong.append("%s: no index: status %d (oracle %d) guard %s" % (name, st, want_st, guard))
        if claimed is not None:
            idx = torch.tensor(_stale_index(oracle, bases[name.split("/")[1]], claimed), dtype=torch.int64, device="cuda")
            st, got, guard = _device_decode(snappy, device, torch, s, claimed, index=idx)
            if st != want_st or not guard or (st == 0 and not np.array_equal(got, want_b)):
                wrong.append("%s: stale index: status %d (oracle %d) guard %s" % (name, st, want_st, guard))
        try:
            got, st = snappy.uncompress(s), 0
        except snappy.SnappyError as e:
            got, st = None, e.status
        if st != want_st or (st == 0 and got != want_b.tobytes()):
            wrong.append("%s: host API: status %d (oracle %d)" % (name, st, want_st))
    print("paths", dict(paths))
    assert not wrong, "\n".join(wrong[:20])
    assert paths[1] >= 5 and paths[2] >= 5 and paths[3] >= 5, paths


@pytest.mark.gpu
@pytest.mark.parametrize("option,value", [("parse_chunk_log2", 9), ("parse_chunk_log2", 13), ("clean_cuts", 0),
                                          ("decode_occupancy", 8), ("decode_occupancy", 10)])
def test_device_decode_option_variants_match_oracle(snappy, oracle, gpu_corpus, option, value):
    """the full corpus under the non-default parse chunk sizes, tiles on the 64 KiB boundaries, and the other
    instantiations of the indexed decoder (12, the default, runs in every other test)"""
    import torch
    from snappy_jl_b200 import device
    cases, want = gpu_corpus
    defaults = {"parse_chunk_log2": 10, "clean_cuts": 1, "decode_occupancy": 12}
    wrong = []
    try:
        device.set_option(option, value)
        for (name, s), (want_st, want_b) in zip(cases, want):
            st, got, guard = _device_decode(snappy, device, torch, s, _claimed(oracle, s))
            if st != want_st or not guard or (st == 0 and not np.array_equal(got, want_b)):
                wrong.append("%s: status %d (oracle %d) guard %s" % (name, st, want_st, guard))
    finally:
        for k, v in defaults.items():
            device.set_option(k, v)
    assert not wrong, "\n".join(wrong[:20])


@pytest.mark.gpu
def test_batched_pages_with_corrupt_neighbours(snappy, oracle, gpu_corpus):
    """corpus streams of up to 4 MiB as pages of one uncompress_batched_device call, between valid pages: the oracle's
    status per page (7 where the slot is one byte short), out_sizes, valid neighbours byte-exact, and the sentinel bytes
    between the page slots intact"""
    import torch
    from snappy_jl_b200 import device, synth
    cases, want = gpu_corpus
    pages = []  # (stream, cap, status, bytes)
    for k, ((name, s), (st, b)) in enumerate(zip(cases, want)):
        if len(s) > 4 << 20:
            continue
        claimed = _claimed(oracle, s)
        if claimed is None:
            pages.append((s, 0, st, None))
        elif k % 5 == 4 and claimed > 0:
            pages.append((s, claimed - 1, 7, None))
        else:
            pages.append((s, claimed, st, b))
        raw = synth.mix(1, seed=k, tail=int(k * 37 % 5000))[: 1000 + 997 * k % 70000]
        pages.append((oracle.compress(raw.tobytes()), raw.size, 0, raw))
    pages.append((b"", 0, 6, None))
    in_off, flat, out_off, o = [], bytearray(), [], 0
    for s, cap, _, _ in pages:
        in_off.append(len(flat))
        flat += s + bytes(-len(s) % 16)
        out_off.append(o)
        o += (cap + 256 + 15) // 16 * 16  # 256 sentinel bytes behind every slot
    data = torch.from_numpy(np.frombuffer(bytes(flat) + bytes(16), dtype=np.uint8).copy()).cuda()
    out = torch.full((o,), 0xEE, dtype=torch.uint8, device="cuda")
    t = lambda v, dt: torch.tensor(v, dtype=dt, device="cuda")
    sizes, statuses = device.uncompress_batched_device(
        data, t(in_off, torch.int64), t([len(p[0]) for p in pages], torch.int32), out, t(out_off, torch.int64),
        t([p[1] for p in pages], torch.int32))
    sizes, statuses, host = sizes.cpu().numpy(), statuses.cpu().numpy(), out.cpu().numpy()
    wrong = []
    for k, (s, cap, st, b) in enumerate(pages):
        slot_end = out_off[k + 1] if k + 1 < len(pages) else o
        if statuses[k] != st or sizes[k] != (cap if st == 0 else 0):
            wrong.append("page %d: status %d (oracle %d), size %d" % (k, statuses[k], st, sizes[k]))
        elif st == 0 and not np.array_equal(host[out_off[k]: out_off[k] + cap], b):
            wrong.append("page %d: bytes differ" % k)
        if not np.all(host[out_off[k] + cap: slot_end] == 0xEE):
            wrong.append("page %d: wrote past its out_cap" % k)
    assert not wrong, "\n".join(wrong[:20])


@pytest.mark.gpu
def test_streamed_host_uncompress_on_corrupt_and_quirky_streams(snappy, oracle):
    """streams of more than 64 MiB take the streamed host path (parsed in upload segments while the rest goes up):
    a fault in the first, a middle and the last upload segment, a truncation, a header that claims one fragment too
    many, and two valid streams the reference accepts: a lone trailing byte, a zero-length literal"""
    from snappy_jl_b200 import synth
    tile = synth.mix(256, seed=31)                        # 16 MiB
    parts0, _ = oracle.compress_fragments(tile, tile.size, 0, 256)
    reps = (72 << 20) // parts0.size + 1                  # > 64 MiB compressed
    total = tile.size * reps
    parts, sizes = oracle.compress_fragments(tile, total, 0, 256)
    hdr = np.frombuffer(oracle.encode32(total), dtype=np.uint8)
    good = np.concatenate([hdr] + [parts] * reps)
    raw = np.tile(tile, reps)
    assert good.size > 64 << 20
    streams = []
    for where in (0.03, 0.5, 0.97):
        st, k = 0, 0
        while st == 0:  # a garbled spot that only hits literal bytes leaves the stream valid: take the next one
            bad = good.copy()
            pos = int(good.size * where) + 7919 * k
            bad[pos: pos + 24] ^= 0xA7
            st = oracle.status_of_uncompress(bad)
            k += 1
            assert k < 40
        streams.append(("garbled@%.2f" % where, bad))
    streams.append(("truncated", good[: good.size - 12345]))
    streams.append(("claimed+65536", np.concatenate([np.frombuffer(oracle.encode32(total + FRAGMENT), dtype=np.uint8), good[hdr.size:]])))
    streams.append(("trailing_byte", np.concatenate([good, np.array([9], dtype=np.uint8)])))
    cut = hdr.size + parts.size * (reps // 2) + int(sizes[:100].sum())  # an element start (fragment boundary)
    streams.append(("zero_literal", np.concatenate([good[:cut], np.frombuffer(ZERO_LITERAL, dtype=np.uint8), good[cut:]])))
    wrong = []
    for name, s in streams:
        want_st = oracle.status_of_uncompress(s)
        if name in ("trailing_byte", "zero_literal"):
            assert want_st == 0
        try:
            got, st = snappy.uncompress_np(s), 0
        except snappy.SnappyError as e:
            got, st = None, e.status
        if st != want_st or (st == 0 and not np.array_equal(got, raw)):
            wrong.append("%s: status %d (oracle %d)" % (name, st, want_st))
    assert not wrong, "\n".join(wrong)
