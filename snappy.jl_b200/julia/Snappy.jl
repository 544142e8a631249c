# Snappy.jl -- drop-in replacement for krm01/Snappy.jl's module file (src/Snappy.jl) whose
# compress / uncompress run on a B200 through libsnappy_b200.so.
#
# Same exports and same helper names as the reference module:
#   compress(::Vector{UInt8}), compress(::String), uncompress(::Vector{UInt8})      (Snappy.jl:3-5,20,38,46)
#   maxlength_compressed, length_uncompressed                                       (Snappy.jl:80-92)
#   parse32, encode32!, find_match_length  -- the names test/runtests.jl reaches into (:96,:102,:159-160,:172)
# Every ccall below has the shape of the reference's own FFI example, test/libsnappy.jl:5-30
# (caller allocates both buffers, passes a Ref{Csize_t} capacity, resize!s to the returned length).
# Failures raise ErrorException with the reference's messages (error(...) at Snappy.jl:21,50,
# internal.jl:499,505,518, varint.jl:36).  varint.jl stays host-side Julia, as in the reference.
#
# NOTE: there is no Julia in the build image, so this file has not been executed there; the Python
# ctypes twin (snappy.jl_b200/_abi.py + api.py) makes exactly the same C calls and is what the test
# suite drives.  Written for Julia >= 1.0 syntax.
module Snappy

export compress, uncompress

const LIB = get(ENV, "SNAPPY_B200_LIB", "libsnappy_b200")

include("varint.jl")   # parse32 / encode32!: host-side, same interface as the reference src/varint.jl

# status -> the reference's message (include/snappy_b200.h)
function _check(status::Cint)
    status == 0 && return nothing
    msg = unsafe_string(ccall((:snappy_b200_status_string, LIB), Cstring, (Cint,), status))
    if status >= 8   # CUDA / device problems carry a detail string
        detail = unsafe_string(ccall((:snappy_b200_last_error, LIB), Cstring, ()))
        msg = string(msg, " (", detail, ")")
    end
    error(msg)
end

"""
    maxlength_compressed(sourcelen::Integer)

Return the maximum possible output size (in bytes) for a given input.
"""
maxlength_compressed(sourcelen::Integer) =
    Int(ccall((:snappy_b200_max_compressed_length, LIB), Csize_t, (Csize_t,), sourcelen))

"""
    compress(input::Vector{UInt8})

Compress a byte array; the stream is byte-identical to the pure-Julia Snappy.jl's.
"""
function compress(input::Vector{UInt8})
    length(input) > typemax(UInt32) && error("Input too large.")
    output = Vector{UInt8}(undef, maxlength_compressed(length(input)))
    outlen = Ref{Csize_t}(length(output))
    GC.@preserve input output begin
        _check(ccall((:snappy_b200_compress, LIB), Cint,
                     (Ptr{UInt8}, Csize_t, Ptr{UInt8}, Ref{Csize_t}),
                     input, length(input), output, outlen))
    end
    return resize!(output, outlen[])
end
compress(input::String) = compress(Vector{UInt8}(codeunits(input)))

"""
    length_uncompressed(input::Vector{UInt8})

Read uncompressed length encoded as a varint32 from the start of the array.
"""
length_uncompressed(input::Vector{UInt8}) = parse32(input, firstindex(input))

"""
    uncompress(input::Vector{UInt8})

Uncompress a snappy encoded byte array.
"""
function uncompress(input::Vector{UInt8})
    output_size, _ = length_uncompressed(input)          # throws "Could not decode varint32."
    output = zeros(UInt8, output_size)
    outlen = Ref{Csize_t}(length(output))
    GC.@preserve input output begin
        _check(ccall((:snappy_b200_uncompress, LIB), Cint,
                     (Ptr{UInt8}, Csize_t, Ptr{UInt8}, Ref{Csize_t}),
                     input, length(input), output, outlen))
    end
    return output
end

"""
    validate(input::Vector{UInt8}) -> Int

The status `uncompress(input)` would end with, without decoding: 0 when it would succeed, else the reference's
status 2..6 (`snappy_b200_status_string` gives its message).  No output buffer.  Device problems raise.
"""
function validate(input::Vector{UInt8})
    status = GC.@preserve input begin
        ccall((:snappy_b200_validate_compressed_buffer, LIB), Cint, (Ptr{UInt8}, Csize_t), input, length(input))
    end
    status >= 7 && _check(status)
    return Int(status)
end

# test/runtests.jl:172 calls Snappy.find_match_length(c, i1, i2, limit) with 1-based indices and an
# inclusive limit; the C helper is 0-based with an exclusive limit.
function find_match_length(a::Vector{UInt8}, i1::Integer, i2::Integer, limit::Integer)
    GC.@preserve a begin
        return Int(ccall((:snappy_b200_find_match_length, LIB), Csize_t,
                         (Ptr{UInt8}, Csize_t, Csize_t, Csize_t), a, i1 - 1, i2 - 1, limit))
    end
end

# Side-index sidecar (include/snappy_b200.h): `index` holds the nfrag + 1 fragment offsets a
# device-resident compress returned; the sidecar travels next to the stream and lets a consumer take
# the indexed decoder (snappy_b200_uncompress_device with d_frag_index) without the parse.
function pack_index(index::Vector{UInt64}, uncompressed_len::Integer)
    nfrag = length(index) - 1
    out = Vector{UInt8}(undef, ccall((:snappy_b200_index_pack_bound, LIB), Csize_t, (Csize_t,), nfrag))
    outlen = Ref{Csize_t}(length(out))
    GC.@preserve index out begin
        _check(ccall((:snappy_b200_index_pack, LIB), Cint,
                     (Ptr{UInt64}, Csize_t, UInt64, Ptr{UInt8}, Ref{Csize_t}),
                     index, nfrag, uncompressed_len, out, outlen))
    end
    resize!(out, outlen[])
end

function unpack_index(sidecar::Vector{UInt8})
    nfrag = Ref{Csize_t}(0)
    ulen = Ref{UInt64}(0)
    slen = Ref{UInt64}(0)
    GC.@preserve sidecar begin
        _check(ccall((:snappy_b200_index_unpack, LIB), Cint,
                     (Ptr{UInt8}, Csize_t, Ptr{UInt64}, Ref{Csize_t}, Ref{UInt64}, Ref{UInt64}),
                     sidecar, length(sidecar), C_NULL, nfrag, ulen, slen))
        index = Vector{UInt64}(undef, nfrag[] + 1)
        _check(ccall((:snappy_b200_index_unpack, LIB), Cint,
                     (Ptr{UInt8}, Csize_t, Ptr{UInt64}, Ref{Csize_t}, Ref{UInt64}, Ref{UInt64}),
                     sidecar, length(sidecar), index, nfrag, ulen, slen))
        return index, ulen[], slen[]
    end
end

# Which compressor's bytes `compress` reproduces (include/snappy_b200.h, option "rules"): 0 = Snappy.jl
# (src/internal.jl, the default), 1 = libsnappy <= 1.1.7, 2 = Google snappy >= 1.1.9.
set_rules(rules::Integer) = ccall((:snappy_b200_set_option, LIB), Cvoid, (Cstring, Cint), "rules", rules)

# Optional: pick the device / create the context up front (otherwise lazy on first call).
init(device::Integer = -1) = _check(ccall((:snappy_b200_init, LIB), Cint, (Cint,), device))

end
