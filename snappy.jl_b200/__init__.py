"""snappy.jl_b200 -- B200-native (sm_100a) drop-in for Snappy.jl's compress / uncompress path.

The directory name carries a dot, so it is imported through the root shim `snappy_jl_b200`
(`import snappy_jl_b200 as Snappy`).  Exports mirror src/Snappy.jl:3-5: `compress`, `uncompress`;
the helpers the reference's tests reach into are available under the same names.

No CPU fallback: importing the codec entry points loads libsnappy_b200.so, and every compute call
fails with SnappyError when no sm_100 GPU is usable.
"""
from . import _abi
from .api import (SnappyError, pack_index, unpack_index, set_rules, compress, compress_np, encode32, find_match_length,
                  length_uncompressed, maxlength_compressed, parse32, uncompress, uncompress_np, validate)

K_BLOCK_SIZE = 65536          # src/internal.jl:31
K_INPUT_MARGIN_BYTES = 15     # src/internal.jl:32
K_MAX_HASH_TABLE_SIZE = 16384  # src/internal.jl:33

__all__ = ["compress", "uncompress"]  # src/Snappy.jl:3-5
