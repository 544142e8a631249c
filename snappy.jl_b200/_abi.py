"""ctypes binding of libsnappy_b200.so (include/snappy_b200.h).

This is the Python twin of the Julia `ccall` stubs in snappy.jl_b200/julia/Snappy.jl: the same
C entry points, the same argument order.  There is no fallback of any kind -- if the shared
library is missing the import fails, and if no sm_100 device is usable every compute call
returns SNAPPY_B200_NO_DEVICE, which the callers raise as SnappyError.
"""
import ctypes
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
# SNAPPY_B200_LIB: another build of the same library (A/B experiments); default: the in-tree build
LIB_PATH = os.environ.get("SNAPPY_B200_LIB") or os.path.join(_HERE, "libsnappy_b200.so")

OK = 0
INPUT_TOO_LARGE = 1
INVALID_INPUT = 2
CORRUPT_COPY_OFFSET = 3
CORRUPT_COPY_LENGTH = 4
CORRUPT_LITERAL = 5
BAD_VARINT = 6
BUFFER_TOO_SMALL = 7
CUDA_ERROR = 8
NO_DEVICE = 9
BAD_ARGUMENT = 10

_vp = ctypes.c_void_p
_sz = ctypes.c_size_t
_szp = ctypes.POINTER(ctypes.c_size_t)

# name -> (restype, argtypes); one entry per function declared in include/snappy_b200.h
SIGNATURES = {
    "snappy_b200_status_string": (ctypes.c_char_p, [ctypes.c_int]),
    "snappy_b200_last_error": (ctypes.c_char_p, []),
    "snappy_b200_init": (ctypes.c_int, [ctypes.c_int]),
    "snappy_b200_shutdown": (None, []),
    "snappy_b200_max_compressed_length": (_sz, [_sz]),
    "snappy_b200_compress": (ctypes.c_int, [_vp, _sz, _vp, _szp]),
    "snappy_b200_uncompressed_length": (ctypes.c_int, [_vp, _sz, _szp]),
    "snappy_b200_uncompress": (ctypes.c_int, [_vp, _sz, _vp, _szp]),
    "snappy_b200_validate_compressed_buffer": (ctypes.c_int, [_vp, _sz]),
    "snappy_b200_validate_device": (ctypes.c_int, [_vp, _sz, _vp, _szp, _vp]),
    "snappy_b200_validate_batched_device": (ctypes.c_int, [_vp, _vp, _vp, _sz, _vp, _vp, _vp]),
    "snappy_b200_compress_device": (ctypes.c_int, [_vp, _sz, _vp, _sz, _szp, _vp, _vp]),
    "snappy_b200_uncompress_device": (ctypes.c_int, [_vp, _sz, _vp, _sz, _szp, _vp, _vp]),
    "snappy_b200_compress_batched_device": (ctypes.c_int, [_vp, _vp, _vp, _sz, _vp, _vp, _vp, _vp]),
    "snappy_b200_uncompress_batched_device": (ctypes.c_int,
                                              [_vp, _vp, _vp, _sz, _vp, _vp, _vp, _vp, _vp, _vp]),
    "snappy_b200_compress_shard_device": (ctypes.c_int,
                                          [_vp, _sz, ctypes.c_uint64, _vp, _sz, _szp, _vp, _vp]),
    "snappy_b200_uncompress_shard_device": (ctypes.c_int, [_vp, _vp, _sz, _vp, _sz, _vp]),
    "snappy_b200_compress_shards_device": (ctypes.c_int, [_vp, _vp, _vp, _sz, _vp, _vp, _vp, _vp, _vp]),
    "snappy_b200_uncompress_shards_device": (ctypes.c_int, [_vp, _vp, _vp, _sz, _vp, _vp]),
    "snappy_b200_comm_unique_id": (ctypes.c_int, [_vp]),
    "snappy_b200_comm_create": (ctypes.c_int, [_vp, ctypes.c_int, ctypes.c_int, ctypes.POINTER(_vp)]),
    "snappy_b200_comm_create_loopback": (ctypes.c_int, [ctypes.c_int, ctypes.POINTER(_vp)]),
    "snappy_b200_comm_destroy": (None, [_vp]),
    "snappy_b200_comm_info": (ctypes.c_int, [_vp, ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int),
                                             ctypes.POINTER(ctypes.c_int)]),
    "snappy_b200_comm_compress": (ctypes.c_int, [_vp, _vp, _vp, _vp, _sz, _vp, _vp, _vp, _vp]),
    "snappy_b200_comm_uncompress": (ctypes.c_int, [_vp, _vp, _vp, _vp, _vp, _sz, _vp, _vp, _vp]),
    "snappy_b200_encode_header": (ctypes.c_int, [ctypes.c_uint32, _vp]),
    "snappy_b200_parse_header": (ctypes.c_int, [_vp, _sz, ctypes.POINTER(ctypes.c_uint32), _szp]),
    "snappy_b200_find_match_length": (_sz, [_vp, _sz, _sz, _sz]),
    "snappy_b200_last_kernel_ms": (ctypes.c_float, [ctypes.c_int]),
    "snappy_b200_last_launch_count": (ctypes.c_int, [ctypes.c_int]),
    "snappy_b200_set_option": (None, [ctypes.c_char_p, ctypes.c_int]),
    "snappy_b200_get_option": (ctypes.c_int, [ctypes.c_char_p]),
    "snappy_b200_debug_trace": (ctypes.c_size_t, [ctypes.c_void_p, ctypes.c_size_t]),
    "snappy_b200_index_pack_bound": (ctypes.c_size_t, [ctypes.c_size_t]),
    "snappy_b200_index_pack": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_uint64, ctypes.c_void_p,
                                              ctypes.POINTER(ctypes.c_size_t)]),
    "snappy_b200_index_unpack": (ctypes.c_int, [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_void_p,
                                                ctypes.POINTER(ctypes.c_size_t), ctypes.POINTER(ctypes.c_uint64),
                                                ctypes.POINTER(ctypes.c_uint64)]),
}

_lib = None


def lib():
    """Load libsnappy_b200.so (once).  Raises OSError if it was not built -- by design."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise OSError(
                "libsnappy_b200.so is not built (%s); run `python -c 'import __graft_entry__ as g; "
                "g.build()'` or `make -C snappy.jl_b200/csrc`.  There is no CPU fallback." % LIB_PATH)
        L = ctypes.CDLL(LIB_PATH)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = res
            fn.argtypes = args
        _lib = L
    return _lib


def status_string(code):
    return lib().snappy_b200_status_string(int(code)).decode()


def last_error():
    return lib().snappy_b200_last_error().decode()
