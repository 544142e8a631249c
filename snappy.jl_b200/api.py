"""Host-side mirror of Snappy.jl's module interface (src/Snappy.jl:3-5,20,38,46,80-92).

Same names, same argument meaning, same failure behaviour as the reference: `compress(bytes)`,
`compress(str)`, `uncompress(bytes)` are the exports; `maxlength_compressed`,
`length_uncompressed`, `parse32`, `encode32`, `find_match_length` are the un-exported helpers the
reference's tests touch (test/runtests.jl:96,102,159-160,172).  Failures raise SnappyError (the
twin of Julia's ErrorException) carrying the reference's message.

Every call goes through the C ABI into the sm_100a kernels: the host-buffer entry points copy
host -> device, run the kernels and copy the result back.  Nothing here computes on the CPU
except the varint header helpers, which the reference also keeps on the host (varint.jl).
"""
import ctypes

import numpy as np

from . import _abi


class SnappyError(Exception):
    """Julia `ErrorException` twin: `str(e)` is the reference's message, `e.status` the C code."""

    def __init__(self, status, detail=None):
        msg = _abi.status_string(status)
        if detail and status in (_abi.CUDA_ERROR, _abi.NO_DEVICE):
            msg = "%s (%s)" % (msg, detail)
        super().__init__(msg)
        self.status = status


def _check(rc):
    if rc != _abi.OK:
        raise SnappyError(rc, _abi.last_error())


def _as_u8(data):
    if isinstance(data, str):  # compress(::String), src/Snappy.jl:38
        data = data.encode("utf-8")
    if isinstance(data, np.ndarray):
        return np.ascontiguousarray(data, dtype=np.uint8).reshape(-1)
    return np.frombuffer(bytes(data), dtype=np.uint8)


def _ptr(a):
    return ctypes.c_void_p(a.ctypes.data if a.size else 0)


def maxlength_compressed(sourcelen):
    """src/Snappy.jl:80-82."""
    return _abi.lib().snappy_b200_max_compressed_length(int(sourcelen))


def compress_np(data):
    """compress on a numpy uint8 array; returns a numpy uint8 array (no bytes() copy)."""
    a = _as_u8(data)
    if a.size > 0xFFFFFFFF:
        raise SnappyError(_abi.INPUT_TOO_LARGE)  # src/Snappy.jl:21
    out = np.empty(maxlength_compressed(a.size), dtype=np.uint8)  # :25
    n = ctypes.c_size_t(out.size)
    _check(_abi.lib().snappy_b200_compress(_ptr(a), a.size, _ptr(out), ctypes.byref(n)))
    return out[: n.value]  # resize!, :35


def compress(data):
    """Snappy.compress(::Vector{UInt8}) / compress(::String) -> bytes (src/Snappy.jl:20-38)."""
    return compress_np(data).tobytes()


def length_uncompressed(data):
    """src/Snappy.jl:90-92: (value, index past the varint) -- 0-based index here."""
    return parse32(data, 0)


def uncompress_np(data):
    a = _as_u8(data)
    claimed = ctypes.c_size_t(0)
    _check(_abi.lib().snappy_b200_uncompressed_length(_ptr(a), a.size, ctypes.byref(claimed)))
    out = np.zeros(claimed.value, dtype=np.uint8)  # src/Snappy.jl:48
    n = ctypes.c_size_t(out.size)
    _check(_abi.lib().snappy_b200_uncompress(_ptr(a), a.size, _ptr(out), ctypes.byref(n)))
    return out[: n.value]


def uncompress(data):
    """Snappy.uncompress(::Vector{UInt8}) -> bytes (src/Snappy.jl:46-52)."""
    return uncompress_np(data).tobytes()


def validate(data):
    """snappy_validate_compressed_buffer / IsValidCompressedBuffer: the status `uncompress(data)` would end with --
    0 when it would succeed, else the reference's status 2..6 (`SnappyError(status)` carries its message).  Nothing is
    decoded and no output is allocated; raises SnappyError only for CUDA / device problems."""
    a = _as_u8(data)
    rc = _abi.lib().snappy_b200_validate_compressed_buffer(_ptr(a), a.size)
    if rc >= _abi.BUFFER_TOO_SMALL:
        raise SnappyError(rc, _abi.last_error())
    return rc


def parse32(buf, offset=0):
    """varint.jl:12-37 with a 0-based offset: returns (value, index past the varint)."""
    a = _as_u8(buf)
    if offset < 0 or offset > a.size:
        raise SnappyError(_abi.BAD_VARINT)
    v = ctypes.c_uint32(0)
    hdr = ctypes.c_size_t(0)
    sub = a[offset:]
    _check(_abi.lib().snappy_b200_parse_header(_ptr(sub), sub.size, ctypes.byref(v), ctypes.byref(hdr)))
    return v.value, offset + hdr.value


def encode32(value):
    """varint.jl:46-69: the 1..5 bytes of the varint32."""
    buf = np.zeros(5, dtype=np.uint8)
    k = _abi.lib().snappy_b200_encode_header(int(value) & 0xFFFFFFFF, _ptr(buf))
    return buf[:k].tobytes()


def find_match_length(a, i1, i2, limit):
    """src/internal.jl:344-387, 0-based with `limit` exclusive (the reference: 1-based inclusive)."""
    arr = _as_u8(a)
    if not (0 <= i1 <= i2 <= limit <= arr.size):
        raise ValueError("find_match_length: need 0 <= i1 <= i2 <= limit <= len(a)")
    return _abi.lib().snappy_b200_find_match_length(_ptr(arr), i1, i2, limit)


# ---- side-index sidecar (SURVEY.md section 8(f)2; include/snappy_b200.h) --------------------------

def set_rules(rules):
    """Which compressor's bytes `compress` reproduces: 0 = Snappy.jl (the reference, default), 1 = libsnappy
    <= 1.1.7, 2 = Google snappy >= 1.1.9 (what pyarrow / current C++ consumers produce).  SURVEY.md 8(f)4."""
    if rules not in (0, 1, 2):
        raise ValueError("rules must be 0, 1 or 2")
    _abi.lib().snappy_b200_set_option(b"rules", int(rules))


def pack_index(index, uncompressed_len):
    """`index`: the nfrag + 1 fragment offsets of a stream (as returned by device.compress_device(...,
    want_index=True), on the host).  Returns the sidecar bytes that travel next to the stream."""
    idx = np.ascontiguousarray(np.asarray(index), dtype=np.uint64).reshape(-1)
    nfrag = idx.size - 1
    out = np.empty(_abi.lib().snappy_b200_index_pack_bound(nfrag), dtype=np.uint8)
    n = ctypes.c_size_t(out.size)
    _check(_abi.lib().snappy_b200_index_pack(_ptr(idx), nfrag, int(uncompressed_len), _ptr(out), ctypes.byref(n)))
    return out[: n.value].tobytes()


def unpack_index(sidecar):
    """Inverse of pack_index: (index as uint64 array of nfrag + 1 offsets, uncompressed_len, stream_len).
    Raises SnappyError("Invalid input.") for a malformed sidecar."""
    a = _as_u8(sidecar)
    nfrag = ctypes.c_size_t(0)
    ulen, slen = ctypes.c_uint64(0), ctypes.c_uint64(0)
    _check(_abi.lib().snappy_b200_index_unpack(_ptr(a), a.size, None, ctypes.byref(nfrag), ctypes.byref(ulen),
                                               ctypes.byref(slen)))
    idx = np.empty(nfrag.value + 1, dtype=np.uint64)
    cap = ctypes.c_size_t(nfrag.value)
    _check(_abi.lib().snappy_b200_index_unpack(_ptr(a), a.size, _ptr(idx), ctypes.byref(cap), ctypes.byref(ulen),
                                               ctypes.byref(slen)))
    return idx, ulen.value, slen.value
