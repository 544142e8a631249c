"""Device-resident entry points on torch uint8 CUDA tensors (torch is plumbing only: it owns the
device memory and the stream; all work happens in libsnappy_b200.so's sm_100a kernels).

These wrap the `_device`, `_batched_device` and `_shard_device` functions of
include/snappy_b200.h, which is what BASELINE.json's GB/s targets are quoted on.
"""
import ctypes

import torch

from . import _abi
from .api import SnappyError, _check, maxlength_compressed

FRAGMENT = 65536  # K_BLOCK_SIZE, src/internal.jl:31


def _dev_ptr(t):
    if t is None:
        return ctypes.c_void_p(0)
    if not t.is_cuda or not t.is_contiguous():
        raise ValueError("expected a contiguous CUDA tensor")
    return ctypes.c_void_p(t.data_ptr())


def _stream_ptr(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


def nfragments(n):
    return (n + FRAGMENT - 1) // FRAGMENT


def compress_device(src, out=None, want_index=False):
    """Compress the uint8 CUDA tensor `src` into one Snappy stream on the device.

    Returns (stream_tensor_view, frag_index or None).  `out` may be a preallocated uint8 CUDA
    tensor of at least maxlength_compressed(len(src)) bytes.  frag_index is the (nfrag+1) x
    uint64 side index of fragment offsets inside the stream."""
    n = src.numel()
    cap = maxlength_compressed(n)
    if out is None:
        out = torch.empty(cap, dtype=torch.uint8, device=src.device)
    elif out.numel() < cap:
        raise SnappyError(_abi.BUFFER_TOO_SMALL)
    index = None
    if want_index:
        index = torch.empty(nfragments(n) + 1, dtype=torch.int64, device=src.device)
    out_len = ctypes.c_size_t(0)
    with torch.cuda.device(src.device):
        _abi.lib().snappy_b200_init(src.device.index)
        _check(_abi.lib().snappy_b200_compress_device(
            _dev_ptr(src), n, _dev_ptr(out), out.numel(), ctypes.byref(out_len), _dev_ptr(index),
            _stream_ptr(src.device)))
    return out[: out_len.value], index


def uncompress_device(stream, out=None, index=None, claimed=None):
    """Uncompress a Snappy stream held in a uint8 CUDA tensor.  `index` is the optional side index
    from compress_device; `claimed` (uncompressed length) avoids a header read when known."""
    n = stream.numel()
    if out is None:
        if claimed is None:
            from .api import parse32
            claimed, _ = parse32(stream[: min(n, 5)].cpu().numpy(), 0)
        out = torch.empty(claimed, dtype=torch.uint8, device=stream.device)
    out_len = ctypes.c_size_t(0)
    with torch.cuda.device(stream.device):
        _abi.lib().snappy_b200_init(stream.device.index)
        _check(_abi.lib().snappy_b200_uncompress_device(
            _dev_ptr(stream), n, _dev_ptr(out), out.numel(), ctypes.byref(out_len), _dev_ptr(index),
            _stream_ptr(stream.device)))
    return out[: out_len.value]


def validate_device(stream, index=None):
    """Would uncompress_device(stream, index=index) succeed?  Returns (status, claimed): status 0 or the reference's
    2..6, exactly what uncompress_device reports with unlimited room; claimed is the header's length, None when the
    header does not parse.  No output is allocated; `index` (optional side index) cannot change the result."""
    claimed = ctypes.c_size_t(0)
    with torch.cuda.device(stream.device):
        _abi.lib().snappy_b200_init(stream.device.index)
        rc = _abi.lib().snappy_b200_validate_device(_dev_ptr(stream), stream.numel(), _dev_ptr(index),
                                                    ctypes.byref(claimed), _stream_ptr(stream.device))
    if rc >= _abi.BUFFER_TOO_SMALL:
        raise SnappyError(rc, _abi.last_error())
    return rc, (None if rc == _abi.BAD_VARINT else claimed.value)


def compress_shard_device(shard, total_len, out=None, want_sizes=False):
    """Compress a run of whole fragments of a stream whose total length is `total_len`
    (elements only, no varint header).  Returns (bytes_view, frag_sizes or None)."""
    n = shard.numel()
    cap = maxlength_compressed(n)
    if out is None:
        out = torch.empty(cap, dtype=torch.uint8, device=shard.device)
    sizes = None
    if want_sizes:
        sizes = torch.empty(max(nfragments(n), 1), dtype=torch.int32, device=shard.device)
    out_len = ctypes.c_size_t(0)
    with torch.cuda.device(shard.device):
        _abi.lib().snappy_b200_init(shard.device.index)
        _check(_abi.lib().snappy_b200_compress_shard_device(
            _dev_ptr(shard), n, int(total_len), _dev_ptr(out), out.numel(), ctypes.byref(out_len),
            _dev_ptr(sizes), _stream_ptr(shard.device)))
    return out[: out_len.value], (sizes[: nfragments(n)] if want_sizes else None)


def uncompress_shard_device(data, frag_offsets, out_len, out=None):
    """Decode fragments given their element byte ranges (frag_offsets: (nfrag+1) x int64, offsets
    into `data`); fragment i lands at out[i*65536:]."""
    nfrag = nfragments(out_len)
    if out is None:
        out = torch.empty(out_len, dtype=torch.uint8, device=data.device)
    if out_len == 0:
        return out
    with torch.cuda.device(data.device):
        _abi.lib().snappy_b200_init(data.device.index)
        _check(_abi.lib().snappy_b200_uncompress_shard_device(
            _dev_ptr(data), _dev_ptr(frag_offsets), nfrag, _dev_ptr(out), out_len,
            _stream_ptr(data.device)))
    return out


def _ptr_array(tensors):
    return (ctypes.c_void_p * len(tensors))(*[(t.data_ptr() if t is not None and t.numel() else 0) for t in tensors])


def compress_shards_device(shards, total_lens, want_sizes=True):
    """Batched compress_shard_device: all shards go through one kernel pass.
    Returns a list of (bytes_view, frag_sizes)."""
    count = len(shards)
    dev = shards[0].device
    outs = [torch.empty(maxlength_compressed(s.numel()), dtype=torch.uint8, device=dev) for s in shards]
    sizes = [torch.empty(max(nfragments(s.numel()), 1), dtype=torch.int32, device=dev) for s in shards]
    lens = (ctypes.c_size_t * count)(*[s.numel() for s in shards])
    totals = (ctypes.c_uint64 * count)(*[int(t) for t in total_lens])
    caps = (ctypes.c_size_t * count)(*[o.numel() for o in outs])
    out_lens = (ctypes.c_size_t * count)()
    for s in shards:
        if not s.is_cuda or not s.is_contiguous():
            raise ValueError("expected contiguous CUDA tensors")
    with torch.cuda.device(dev):
        _abi.lib().snappy_b200_init(dev.index)
        _check(_abi.lib().snappy_b200_compress_shards_device(
            _ptr_array(shards), lens, totals, count, _ptr_array(outs), caps, out_lens,
            _ptr_array(sizes) if want_sizes else None, _stream_ptr(dev)))
    return [(outs[k][: out_lens[k]], sizes[k][: nfragments(shards[k].numel())]) for k in range(count)]


def uncompress_shards_device(datas, frag_offsets, out_lens):
    """Batched uncompress_shard_device.  Returns the list of decoded runs."""
    count = len(datas)
    dev = datas[0].device
    outs = [torch.empty(int(n), dtype=torch.uint8, device=dev) for n in out_lens]
    lens = (ctypes.c_size_t * count)(*[int(n) for n in out_lens])
    with torch.cuda.device(dev):
        _abi.lib().snappy_b200_init(dev.index)
        _check(_abi.lib().snappy_b200_uncompress_shards_device(
            _ptr_array(datas), _ptr_array(frag_offsets), lens, count, _ptr_array(outs), _stream_ptr(dev)))
    return outs


def compress_batched_device(src, in_offsets, in_sizes, out=None, out_offsets=None):
    """One independent stream per page.  in_offsets int64[count], in_sizes int32[count] (device).
    Returns (out, out_offsets, out_sizes)."""
    count = in_sizes.numel()
    dev = src.device
    if out_offsets is None:
        sz = in_sizes.to(torch.int64)
        caps = 32 + sz + sz // 6
        caps = (caps + 15) // 16 * 16
        out_offsets = torch.cumsum(caps, 0) - caps
        total = int(caps.sum().item())
        out = torch.empty(total, dtype=torch.uint8, device=dev)
    out_sizes = torch.zeros(count, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _abi.lib().snappy_b200_init(dev.index)
        _check(_abi.lib().snappy_b200_compress_batched_device(
            _dev_ptr(src), _dev_ptr(in_offsets), _dev_ptr(in_sizes), count, _dev_ptr(out),
            _dev_ptr(out_offsets), _dev_ptr(out_sizes), _stream_ptr(dev)))
    return out, out_offsets, out_sizes


def uncompress_batched_device(data, in_offsets, in_sizes, out, out_offsets, out_caps):
    """Inverse of compress_batched_device.  Returns (out_sizes, statuses) device tensors."""
    count = in_sizes.numel()
    dev = data.device
    out_sizes = torch.zeros(count, dtype=torch.int32, device=dev)
    statuses = torch.zeros(count, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _abi.lib().snappy_b200_init(dev.index)
        _check(_abi.lib().snappy_b200_uncompress_batched_device(
            _dev_ptr(data), _dev_ptr(in_offsets), _dev_ptr(in_sizes), count, _dev_ptr(out),
            _dev_ptr(out_offsets), _dev_ptr(out_caps), _dev_ptr(out_sizes), _dev_ptr(statuses),
            _stream_ptr(dev)))
    return out_sizes, statuses


def validate_batched_device(data, in_offsets, in_sizes):
    """Validation form of uncompress_batched_device (no output).  Returns (statuses, claimed) int32 device tensors:
    per page what uncompress_batched_device reports with unlimited room, and the header's length (0 when it does not
    parse)."""
    count = in_sizes.numel()
    dev = data.device
    claimed = torch.zeros(count, dtype=torch.int32, device=dev)
    statuses = torch.zeros(count, dtype=torch.int32, device=dev)
    with torch.cuda.device(dev):
        _abi.lib().snappy_b200_init(dev.index)
        _check(_abi.lib().snappy_b200_validate_batched_device(
            _dev_ptr(data), _dev_ptr(in_offsets), _dev_ptr(in_sizes), count, _dev_ptr(claimed), _dev_ptr(statuses),
            _stream_ptr(dev)))
    return statuses, claimed


def last_kernel_ms(which):
    """Device time of the dominant kernel of the last compress (0) / uncompress (1) call."""
    return float(_abi.lib().snappy_b200_last_kernel_ms(which))


def last_launch_count(which):
    return int(_abi.lib().snappy_b200_last_launch_count(which))


def set_option(name, value):
    _abi.lib().snappy_b200_set_option(name.encode(), int(value))
