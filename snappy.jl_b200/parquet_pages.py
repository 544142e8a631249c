"""Parquet-page adapter (SURVEY.md section 8(f)3): BASELINE config 4's real-world caller.

A Parquet column chunk is a run of pages, each `PageHeader` (Thrift compact protocol) followed by
`compressed_page_size` bytes; with the SNAPPY codec every page body is ONE raw Snappy stream (varint
length + elements) -- exactly the unit of the batched page API
(`snappy_b200_uncompress_batched_device`, one independent stream per page).  This module walks the
page headers of a file image, hands all SNAPPY page bodies to the GPU in one batched call, and
returns the decompressed pages; `compress_pages` is the writer-side twin (one stream per page).

Only the page headers are parsed here (host, a few hundred bytes per page); the file footer is read
with pyarrow, which is also what the tests use to WRITE the files.  Nothing on the data path runs on
the CPU.
"""
import struct

import numpy as np

SNAPPY = "SNAPPY"


# ---- Thrift compact protocol: just enough to read a PageHeader and know where it ends ------------
class _Reader:
    """Page headers come out of files: every length is checked against the bytes that are left, nesting is
    bounded, and read_page_header turns any malformed input into ValueError."""
    MAX_DEPTH = 16

    def __init__(self, buf, pos):
        self.b, self.p, self.depth = buf, pos, 0

    def _left(self):
        return len(self.b) - self.p

    def byte(self):
        v = self.b[self.p]
        self.p += 1
        return v

    def varint(self):
        v, s = 0, 0
        while True:
            c = self.byte()
            v |= (c & 0x7F) << s
            s += 7
            if not c & 0x80:
                return v
            if s > 63:
                raise ValueError("thrift compact: varint too long")

    def zigzag(self):
        v = self.varint()
        return (v >> 1) ^ -(v & 1)

    def value(self, t, in_container=False):
        if t in (1, 2):                      # BOOLEAN_TRUE / BOOLEAN_FALSE (in a struct the value lives in the type)
            return (self.byte() == 1) if in_container else (t == 1)
        if t == 3:
            return self.byte()
        if t in (4, 5, 6):                   # i16 / i32 / i64
            return self.zigzag()
        if t == 7:
            v = struct.unpack_from("<d", self.b, self.p)[0]
            self.p += 8
            return v
        if t == 8:                           # binary / string
            n = self.varint()
            if n > self._left():
                raise ValueError("thrift compact: string runs past the buffer")
            v = bytes(self.b[self.p:self.p + n])
            self.p += n
            return v
        if t in (9, 10):                     # list / set
            h = self.byte()
            n, et = h >> 4, h & 0x0F
            if n == 15:
                n = self.varint()
            if n > self._left():             # every element takes at least one byte
                raise ValueError("thrift compact: list runs past the buffer")
            return [self.value(et, True) for _ in range(n)]
        if t == 11:                          # map
            n = self.varint()
            if n == 0:
                return {}
            if 2 * n > self._left():
                raise ValueError("thrift compact: map runs past the buffer")
            kv = self.byte()
            return {self.value(kv >> 4, True): self.value(kv & 0x0F, True) for _ in range(n)}
        if t == 12:
            return self.struct()
        raise ValueError("thrift compact: unknown type %d" % t)

    def struct(self):
        self.depth += 1
        if self.depth > self.MAX_DEPTH:
            raise ValueError("thrift compact: nesting too deep")
        out, fid = {}, 0
        while True:
            h = self.byte()
            if h == 0:
                self.depth -= 1
                return out
            delta, t = h >> 4, h & 0x0F
            fid = fid + delta if delta else self.zigzag()
            out[fid] = self.value(t)


DATA_PAGE, INDEX_PAGE, DICTIONARY_PAGE, DATA_PAGE_V2 = 0, 1, 2, 3


def read_page_header(buf, pos):
    """PageHeader at buf[pos:]: returns (fields, header_length).  fields: 1 type, 2 uncompressed_page_size,
    3 compressed_page_size, 5 data_page_header, 7 dictionary_page_header, 8 data_page_header_v2."""
    r = _Reader(buf, pos)
    try:
        f = r.struct()
    except (IndexError, struct.error, TypeError) as e:
        raise ValueError("malformed page header: %s" % e) from None
    for need in (1, 2, 3):
        if not isinstance(f.get(need), int) or f[need] < 0:
            raise ValueError("malformed page header: field %d" % need)
    return f, r.p - pos


def list_pages(file_bytes):
    """All pages of all column chunks of a Parquet file image.  Returns a list of dicts:
    codec, kind, header (offset of the PageHeader), body (offset of the page body in the file), compressed (bytes of the SNAPPY stream
    inside the body), stream (offset of that stream), uncompressed (its decoded length), prefix (bytes
    of the body that are stored uncompressed in front of it: the levels of a v2 data page)."""
    import io
    import pyarrow.parquet as pq
    buf = memoryview(file_bytes)
    md = pq.ParquetFile(io.BytesIO(bytes(file_bytes))).metadata
    pages = []
    for rg in range(md.num_row_groups):
        for ci in range(md.num_columns):
            col = md.row_group(rg).column(ci)
            pos = col.dictionary_page_offset if col.has_dictionary_page and col.dictionary_page_offset else col.data_page_offset
            end = pos + col.total_compressed_size
            while pos < end:
                f, hl = read_page_header(buf, pos)
                body = pos + hl
                csize, usize, kind = f[3], f[2], f[1]
                prefix, compressed = 0, True
                if kind == DATA_PAGE_V2:
                    h2 = f[8]
                    prefix = h2.get(5, 0) + h2.get(6, 0)       # definition + repetition level bytes
                    compressed = h2.get(7, True)
                # the sizes come from the file: nothing below may let the decode kernel read past the image or
                # take a negative / >= 2 GiB length (in_sizes and out_caps are 32-bit in the batched C ABI)
                if not isinstance(prefix, int) or not (0 <= prefix <= csize and prefix <= usize):
                    raise ValueError("page at %d: level bytes (%r) exceed the page sizes (%d compressed, %d "
                                     "uncompressed)" % (pos, prefix, csize, usize))
                if csize >= 1 << 31 or usize >= 1 << 31:
                    raise ValueError("page at %d: size of 2 GiB or more (%d compressed, %d uncompressed)"
                                     % (pos, csize, usize))
                if body + csize > len(buf):
                    raise ValueError("page at %d: body [%d, %d) runs past the end of the file image (%d bytes)"
                                     % (pos, body, body + csize, len(buf)))
                pages.append({"codec": col.compression if compressed else "UNCOMPRESSED", "kind": kind,
                              "header": pos, "body": body, "prefix": prefix, "stream": body + prefix,
                              "compressed": csize - prefix, "uncompressed": usize - prefix})
                pos = body + csize
    return pages


def uncompress_pages(file_bytes, pages=None):
    """Decode every SNAPPY page body of the file on the GPU with ONE batched call.
    Returns (pages, out, out_offsets): page i's decoded bytes are out[out_offsets[i] : + uncompressed]
    (numpy uint8; pages with another codec are skipped and get offset -1)."""
    import torch
    from . import device
    if pages is None:
        pages = list_pages(file_bytes)
    sel = [p for p in pages if p["codec"] == SNAPPY and p["compressed"] > 0]
    for p in sel:  # a caller-supplied page list gets the same checks as list_pages applies
        if not (0 <= p["stream"] and p["stream"] + p["compressed"] <= len(file_bytes) and
                0 <= p["uncompressed"] < 1 << 31 and p["compressed"] < 1 << 31):
            raise ValueError("page stream [%d, +%d) -> %d bytes does not fit the file image (%d bytes)"
                             % (p["stream"], p["compressed"], p["uncompressed"], len(file_bytes)))
    offs = np.full(len(pages), -1, dtype=np.int64)
    if not sel:
        return pages, np.empty(0, dtype=np.uint8), offs
    d_file = torch.from_numpy(np.frombuffer(bytes(file_bytes), dtype=np.uint8).copy()).cuda()
    in_off = torch.tensor([p["stream"] for p in sel], dtype=torch.int64, device="cuda")
    in_sz = torch.tensor([p["compressed"] for p in sel], dtype=torch.int32, device="cuda")
    caps = np.array([p["uncompressed"] for p in sel], dtype=np.int64)
    out_off_np = np.concatenate([[0], np.cumsum((caps + 15) // 16 * 16)[:-1]])
    out = torch.zeros(int(((caps + 15) // 16 * 16).sum()), dtype=torch.uint8, device="cuda")
    got_sizes, statuses = device.uncompress_batched_device(
        d_file, in_off, in_sz, out, torch.from_numpy(out_off_np).cuda(),
        torch.from_numpy(caps.astype(np.int32)).cuda())
    st = statuses.cpu().numpy()
    if st.any():
        bad = int(np.nonzero(st)[0][0])
        from .api import SnappyError
        raise SnappyError(int(st[bad]), "page %d" % bad)
    if not np.array_equal(got_sizes.cpu().numpy().astype(np.int64), caps):
        from . import _abi
        from .api import SnappyError
        raise SnappyError(_abi.INVALID_INPUT, "page length differs from its header")
    k = 0
    for i, p in enumerate(pages):
        if p["codec"] == SNAPPY and p["compressed"] > 0:
            offs[i] = out_off_np[k]
            k += 1
    return pages, out.cpu().numpy(), offs


def validate_pages(file_bytes, pages=None):
    """Would uncompress_pages accept each page?  ONE batched validation call on the GPU (no output is allocated or
    written).  Returns (pages, statuses): statuses[i] is 0 or the reference's status 2..6 of page i's Snappy stream,
    INVALID_INPUT (2) as well when the stream's length disagrees with the page header's uncompressed size, and -1 for
    pages uncompress_pages does not decode (another codec, or no compressed bytes)."""
    import torch
    from . import _abi, device
    if pages is None:
        pages = list_pages(file_bytes)
    sel = [i for i, p in enumerate(pages) if pages[i]["codec"] == SNAPPY and pages[i]["compressed"] > 0]
    for i in sel:
        p = pages[i]
        if not (0 <= p["stream"] and p["stream"] + p["compressed"] <= len(file_bytes) and p["compressed"] < 1 << 31):
            raise ValueError("page stream [%d, +%d) does not fit the file image (%d bytes)"
                             % (p["stream"], p["compressed"], len(file_bytes)))
    statuses = np.full(len(pages), -1, dtype=np.int32)
    if not sel:
        return pages, statuses
    d_file = torch.from_numpy(np.frombuffer(bytes(file_bytes), dtype=np.uint8).copy()).cuda()
    in_off = torch.tensor([pages[i]["stream"] for i in sel], dtype=torch.int64, device="cuda")
    in_sz = torch.tensor([pages[i]["compressed"] for i in sel], dtype=torch.int32, device="cuda")
    st, claimed = device.validate_batched_device(d_file, in_off, in_sz)
    st, claimed = st.cpu().numpy(), claimed.cpu().numpy().astype(np.uint32)
    for k, i in enumerate(sel):
        ok_len = int(claimed[k]) == pages[i]["uncompressed"]
        statuses[i] = _abi.INVALID_INPUT if st[k] == _abi.OK and not ok_len else st[k]
    return pages, statuses


def compress_pages(page_bytes):
    """Writer side: a list of uncompressed page bodies -> list of SNAPPY page bodies (bytes), one
    independent stream per page, all pages in ONE batched GPU call."""
    import torch
    from . import device
    if not page_bytes:
        return []
    sizes = np.array([len(p) for p in page_bytes], dtype=np.int64)
    in_off_np = np.concatenate([[0], np.cumsum((sizes + 15) // 16 * 16)[:-1]])
    flat = np.zeros(int(((sizes + 15) // 16 * 16).sum()), dtype=np.uint8)
    for p, o in zip(page_bytes, in_off_np):
        flat[o:o + len(p)] = np.frombuffer(p, dtype=np.uint8)
    out, out_off, out_sz = device.compress_batched_device(
        torch.from_numpy(flat).cuda(), torch.from_numpy(in_off_np).cuda(),
        torch.from_numpy(sizes.astype(np.int32)).cuda())
    o, oo, os_ = out.cpu().numpy(), out_off.cpu().numpy(), out_sz.cpu().numpy()
    return [o[int(a):int(a) + int(n)].tobytes() for a, n in zip(oo, os_)]
