"""CPU suite, part 1: pins the oracle (oracle/snappy_oracle.c) against everything the reference's
own tests hold for this path (test/runtests.jl), against the second transcription
(oracle/py_restatement.py) and against the committed golden vectors."""
import hashlib
import sys

import numpy as np
import pytest

from conftest import (ALL_FILES, ROUNDTRIP_FILES, corrupt_streams, dictionary_fuzz, edge_inputs,
                      read_data)

# test/runtests.jl:176-267 -- (a, b, limit, expected); find_match_length(c=a+b, 1, len(a)+1, len(a)+limit)
FML_KATS = [
    ("012345", "012345", 6, 6), ("01234567abc", "01234567abc", 11, 11),
    ("01234567abc", "01234567axc", 9, 9),
    ("01234567abc!", "01234567abc!", 11, 11), ("01234567abc!", "01234567abc?", 11, 11),
    ("01234567xxxxxxxx", "?1234567xxxxxxxx", 16, 0), ("01234567xxxxxxxx", "0?234567xxxxxxxx", 16, 1),
    ("01234567xxxxxxxx", "01237654xxxxxxxx", 16, 4), ("01234567xxxxxxxx", "0123456?xxxxxxxx", 16, 7),
    ("abcdefgh01234567xxxxxxxx", "abcdefgh?1234567xxxxxxxx", 24, 8),
    ("abcdefgh01234567xxxxxxxx", "abcdefgh0?234567xxxxxxxx", 24, 9),
    ("abcdefgh01234567xxxxxxxx", "abcdefgh01237654xxxxxxxx", 24, 12),
    ("abcdefgh01234567xxxxxxxx", "abcdefgh0123456?xxxxxxxx", 24, 15),
    ("01234567", "?1234567", 8, 0), ("01234567", "0?234567", 8, 1), ("01234567", "01?34567", 8, 2),
    ("01234567", "012?4567", 8, 3), ("01234567", "0123?567", 8, 4), ("01234567", "01234?67", 8, 5),
    ("01234567", "012345?7", 8, 6), ("01234567", "0123456?", 8, 7), ("01234567", "0123456?", 7, 7),
    ("01234567!", "0123456??", 7, 7),
    ("xxxxxxabcd", "xxxxxxabcd", 10, 10), ("xxxxxxabcd?", "xxxxxxabcd?", 10, 10),
    ("xxxxxxabcdef\0", "xxxxxxabcdef\0", 13, 13),
    ("xxxxxx0123abc!", "xxxxxx0123abc!", 12, 12), ("xxxxxx0123abc!", "xxxxxx0123abc?", 12, 12),
    ("xxxxxx0123abc", "xxxxxx0123axc", 13, 11),
    ("xxxxxx0123xxxxxxxx", "xxxxxx?123xxxxxxxx", 18, 6), ("xxxxxx0123xxxxxxxx", "xxxxxx0?23xxxxxxxx", 18, 7),
    ("xxxxxx0123xxxxxxxx", "xxxxxx0132xxxxxxxx", 18, 8), ("xxxxxx0123xxxxxxxx", "xxxxxx012?xxxxxxxx", 18, 9),
    ("xxxxxx0123", "xxxxxx?123", 10, 6), ("xxxxxx0123", "xxxxxx0?23", 10, 7),
    ("xxxxxx0123", "xxxxxx0132", 10, 8), ("xxxxxx0123", "xxxxxx012?", 10, 9),
    ("xxxxxxabcd0123xx", "xxxxxxabcd?123xx", 16, 10), ("xxxxxxabcd0123xx", "xxxxxxabcd0?23xx", 16, 11),
    ("xxxxxxabcd0123xx", "xxxxxxabcd0132xx", 16, 12), ("xxxxxxabcd0123xx", "xxxxxxabcd012?xx", 16, 13),
    ("xxxxxxabcd0123", "xxxxxxabcd?123", 14, 10), ("xxxxxxabcd0123", "xxxxxxabcd0?23", 14, 11),
    ("xxxxxxabcd0123", "xxxxxxabcd0132", 14, 12), ("xxxxxxabcd0123", "xxxxxxabcd012?", 14, 13),
]


def test_kat_count():
    assert len(FML_KATS) == 45  # test/runtests.jl: 45 passing KATs (+1 @test_broken, not a requirement)


@pytest.mark.parametrize("a,b,limit,want", FML_KATS)
def test_find_match_length_kats(oracle, a, b, limit, want):
    c = (a + b).encode("latin-1")
    # reference call: (c, 1, len(a)+1, len(a)+limit), 1-based inclusive limit
    assert oracle.find_match_length(c, 0, len(a), len(a) + limit) == want
    import py_restatement as P
    assert P.find_match_length(P.A1(bytearray(c)), 1, len(a) + 1, len(a) + limit) == want


def test_varint_roundtrip(oracle):
    for i in range(31):  # test/runtests.jl:157-163
        enc = oracle.encode32(1 << i)
        val, nxt = oracle.parse32(enc + b"\0" * (5 - len(enc)), 0)
        assert val == 1 << i and nxt == len(enc)
    assert oracle.encode32(2 ** 30) == bytes([0x80, 0x80, 0x80, 0x80, 0x04])
    assert oracle.encode32(0) == b"\0"
    assert oracle.encode32(0xFFFFFFFF) == bytes([0xFF, 0xFF, 0xFF, 0xFF, 0x0F])


@pytest.mark.parametrize("raw", [bytes([0xF0]), bytes([0x80, 0x80, 0x80, 0x80, 0x80, 0x0A]),
                                 bytes([0xFB, 0xFF, 0xFF, 0xFF, 0x7F]), b""])
def test_varint_rejects(oracle, raw):  # test/runtests.jl:101-111
    with pytest.raises(oracle.OracleError) as e:
        oracle.parse32(raw, 0)
    assert e.value.code == oracle.BAD_VARINT


def test_must_throw(oracle):  # test/runtests.jl:62-123
    import py_restatement as P
    for name, stream in corrupt_streams(oracle):
        with pytest.raises(oracle.OracleError):
            oracle.uncompress(stream)
        if len(stream) < 5000:
            with pytest.raises(P.SnappyError):
                P.uncompress(stream)
    for f in ("baddata1.snappy", "baddata2.snappy", "baddata3.snappy"):
        assert oracle.uncompressed_length(read_data(f)) < (1 << 20)  # runtests.jl:96


def test_baddata_error_positions(oracle):
    # SURVEY.md 8(c): corrupt copy offset at output positions 19791 / 82393 / 35399
    for f, pos in (("baddata1.snappy", 19791), ("baddata2.snappy", 82393), ("baddata3.snappy", 35399)):
        with pytest.raises(oracle.OracleError) as e:
            oracle.uncompress(read_data(f))
        assert e.value.code == oracle.CORRUPT_COPY_OFFSET and e.value.err_op == pos


@pytest.mark.parametrize("name", ALL_FILES)
def test_files_match_golden_and_roundtrip(oracle, golden, name):
    raw = read_data(name)
    c = oracle.compress(raw)
    g = golden["files"][name]
    assert len(raw) == g["raw_len"] and hashlib.sha256(raw).hexdigest() == g["raw_sha256"]
    assert len(c) == g["comp_len"] and hashlib.sha256(c).hexdigest() == g["comp_sha256"]
    assert oracle.uncompress(c) == raw and c != raw  # runtests.jl:29-31


def test_edges_match_golden(oracle, golden):
    for name, raw in edge_inputs().items():
        g = golden["edges"][name]
        c = oracle.compress(raw)
        assert len(c) == g["comp_len"] and hashlib.sha256(c).hexdigest() == g["comp_sha256"], name
        if "comp_hex" in g:
            assert c.hex() == g["comp_hex"], name
        assert oracle.uncompress(c) == raw


def test_known_bytes(oracle):
    # SURVEY.md Appendix C spot values
    assert oracle.compress(b"") == b"\x00"
    assert oracle.compress(b"a") == b"\x01\x00a"
    assert oracle.compress(b"abc") == b"\x03\x08abc"
    assert oracle.compress(bytes(range(60)))[:3] == b"\x3c\xf0\x3b"
    assert oracle.compress(b"a" * 70 + bytes(range(100, 130)))[:9] == bytes.fromhex("640061fe0100050174")
    assert oracle.compress(b"A" * 100000)[:8] == bytes.fromhex("a08d060041fe0100")


def test_decoder_quirks(oracle):
    # SURVEY.md B.3: a lone trailing byte is ignored
    assert oracle.uncompress(bytes([0x00, 0x00])) == b""
    assert oracle.uncompress(bytes([0x01, 0x00, 0x41, 0x77])) == b"A"


def test_c_oracle_equals_python_restatement_on_fuzz(oracle):
    import py_restatement as P
    n = 0
    for raw in dictionary_fuzz(7, 12, maxwords=1 << 11):
        assert oracle.compress(raw) == P.compress(raw)
        n += 1
    rng = np.random.default_rng(3)
    for size in (0, 1, 14, 15, 16, 17, 31, 32, 33, 63, 64, 65, 255, 256, 257, 4095, 4096, 70000):
        for alpha in (2, 4, 256):
            raw = rng.integers(0, alpha, size, dtype=np.uint8).tobytes()
            c = oracle.compress(raw)
            assert c == P.compress(raw), (size, alpha)
            assert P.uncompress(c) == raw and oracle.uncompress(c) == raw


def test_reference_fuzz_roundtrip(oracle):  # test/runtests.jl:35-60 (counts reduced, sizes kept)
    for raw in dictionary_fuzz(11, 10):
        c = oracle.compress(raw)
        assert oracle.uncompress(c) == raw and c != raw


def test_max_blowup(oracle):  # test/runtests.jl:148-154
    rng = np.random.default_rng(5)
    raw = rng.integers(0, 2 ** 32, 20000, dtype=np.uint32).view(np.uint8)
    raw = np.concatenate([raw, raw[::-1]]).tobytes()
    c = oracle.compress(raw)
    assert len(c) <= oracle.maxlength_compressed(len(raw))
    assert oracle.uncompress(c) == raw


def test_cross_decode_with_google_snappy(oracle):
    """format validity only (pyarrow bundles a newer Google snappy; bytes differ, both decode both)"""
    pa = pytest.importorskip("pyarrow")
    codec = pa.Codec("snappy")
    for name in ("html", "alice29.txt", "geo.protodata", "fireworks.jpeg"):
        raw = read_data(name)
        ours = oracle.compress(raw)
        assert codec.decompress(ours, decompressed_size=len(raw)).to_pybytes() == raw
        theirs = codec.compress(raw).to_pybytes()
        assert oracle.uncompress(theirs) == raw


def test_foreign_stream_alice29(oracle):
    """tests/data/alice29.snappy: a 32 KiB-block encoder's stream (SURVEY.md section 4)"""
    assert oracle.uncompress(read_data("alice29.snappy")) == read_data("alice29.txt")


def test_fragment_api_consistent(oracle):
    raw = read_data("urls.10K")
    whole = oracle.compress(raw)
    nfrag = (len(raw) + 65535) // 65536
    parts, sizes = oracle.compress_fragments(raw, len(raw), 0, nfrag)
    hdr = oracle.encode32(len(raw))
    assert hdr + parts.tobytes() == whole and int(sizes.sum()) == len(whole) - len(hdr)
    a, _ = oracle.compress_fragments(raw, len(raw), 0, 5)
    b, _ = oracle.compress_fragments(raw, len(raw), 5, nfrag - 5)
    assert hdr + a.tobytes() + b.tobytes() == whole


# ---- the reference's literal lookup tables (src/internal.jl:47-85), extracted by tests/golden/make_char_table.py ----
def _golden_char_table():
    import json
    import os
    from conftest import ROOT
    with open(os.path.join(ROOT, "tests", "golden", "char_table.json")) as f:
        g = json.load(f)
    assert len(g["char_table"]) == 256 and len(g["wordmask"]) == 5
    return g


def test_char_table_golden_matches_the_snappy_tag_format():
    """the committed table (extracted from the reference by tests/golden/make_char_table.py) holds, for every tag
    byte, what the Snappy format defines: entry = length | copy-offset high bits << 8 | trailer bytes << 11"""
    want = []
    for tag in range(256):
        kind, hi = tag & 3, tag >> 2
        if kind == 0:    # literal: length - 1 in the tag, or in 1..4 trailer bytes for 60..63
            want.append(hi + 1 if hi < 60 else 1 | (hi - 59) << 11)
        elif kind == 1:  # copy, 1 trailer byte: length 4..11, offset bits 8..10 in the tag
            want.append(4 + (hi & 7) | (tag >> 5) << 8 | 1 << 11)
        else:            # copy with a 2- or 4-byte offset trailer: length 1..64
            want.append(hi + 1 | (2 if kind == 2 else 4) << 11)
    g = _golden_char_table()
    assert g["char_table"] == want
    assert g["wordmask"] == [0, 0xFF, 0xFFFF, 0xFFFFFF, 0xFFFFFFFF]


def test_char_table_of_both_cpu_decoders_equals_the_reference_table(oracle):
    """oracle/snappy_oracle.c and oracle/py_restatement.py regenerate CHAR_TABLE by formula: all 256 entries must be
    the reference's literal ones"""
    import py_restatement
    g = _golden_char_table()
    assert oracle.char_table() == g["char_table"]
    assert [int(x) for x in py_restatement.CHAR_TABLE] == g["char_table"]


def test_char_table_of_the_cuda_decoders_equals_the_reference_table(tmp_path):
    """csrc/decompress.cuh evaluates CHAR_TABLE / WORDMASK arithmetically in decode_tag (exact decoder, parse
    kernels) and decode_tag_fast (indexed decoder): the real header, compiled for the CPU, against the literal table"""
    import os
    import subprocess
    from conftest import ROOT
    exe = str(tmp_path / "dump_char_table")
    subprocess.check_call(["g++", "-O1", "-std=c++17", "-DSB200_CPU_EMU", "-I" + os.path.join(ROOT, "tools", "cpu_warp"),
                           "-o", exe, os.path.join(ROOT, "tools", "cpu_warp", "dump_char_table.cpp")])
    lines = subprocess.run([exe], capture_output=True, text=True, check=True).stdout.splitlines()
    g = _golden_char_table()
    assert [int(x) for x in lines[0].split()] == g["char_table"]   # decode_tag
    assert [int(x) for x in lines[1].split()] == g["char_table"]   # decode_tag_fast
    assert [int(x) for x in lines[2].split()] == g["wordmask"]
    assert [int(x) for x in lines[3].split()] == g["wordmask"]
