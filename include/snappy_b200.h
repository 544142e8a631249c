/*
 * include/snappy_b200.h -- C ABI of libsnappy_b200.so: the B200-native (sm_100a) drop-in for
 * Snappy.jl's compress / uncompress hot path.
 *
 * The reference (krm01/Snappy.jl) has no FFI of its own; its exported Julia API
 * (src/Snappy.jl:3-5,20,38,46) is the boundary, and its own model of an FFI call for this path
 * is test/libsnappy.jl:5-30 (ccall into the snappy-c interface).  The four host-buffer entry
 * points below have exactly that shape so that the same ccall stubs bind to them
 * (INTEGRATION.md shows the Julia side).  Everything is plain pointers and sizes.
 *
 * Stream format: varint32(uncompressed length) followed by Snappy elements; the compressed bytes
 * are identical to what Snappy.jl's compress() produces for the same input.
 *
 * There is no CPU fallback: every compute entry point returns SNAPPY_B200_NO_DEVICE /
 * SNAPPY_B200_CUDA_ERROR when no sm_100 GPU is usable.
 */
#ifndef SNAPPY_B200_H
#define SNAPPY_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* Status codes.  1..6 map one-to-one onto the reference's error(...) sites. */
typedef enum {
    SNAPPY_B200_OK = 0,
    SNAPPY_B200_INPUT_TOO_LARGE = 1,     /* src/Snappy.jl:21     "Input too large." */
    SNAPPY_B200_INVALID_INPUT = 2,       /* src/Snappy.jl:50     "Invalid input." */
    SNAPPY_B200_CORRUPT_COPY_OFFSET = 3, /* src/internal.jl:499  "Invalid input: corrupt copy offset" */
    SNAPPY_B200_CORRUPT_COPY_LENGTH = 4, /* src/internal.jl:505  "Invalid input: corrupt copy length" */
    SNAPPY_B200_CORRUPT_LITERAL = 5,     /* src/internal.jl:518  "Invalid input: corrupt literal" */
    SNAPPY_B200_BAD_VARINT = 6,          /* src/varint.jl:36     "Could not decode varint32." */
    SNAPPY_B200_BUFFER_TOO_SMALL = 7,    /* caller's output buffer is smaller than required */
    SNAPPY_B200_CUDA_ERROR = 8,          /* a CUDA runtime call or kernel failed */
    SNAPPY_B200_NO_DEVICE = 9,           /* no CUDA device / not an sm_100 part */
    SNAPPY_B200_BAD_ARGUMENT = 10
} snappy_b200_status;

/* The reference's message for a status (exact strings of the error(...) calls above). */
const char *snappy_b200_status_string(int status);
/* Detail of the last failure on the calling thread (CUDA error text etc.). */
const char *snappy_b200_last_error(void);

/* Select the device (default: current device / $SNAPPY_B200_DEVICE) and create the context.
 * Optional -- every entry point initialises lazily.  Thread-safe. */
int snappy_b200_init(int device);
void snappy_b200_shutdown(void);

/* ---- host-buffer API: replaces test/libsnappy.jl:7,9-12 and :20-28 one for one ------------ */

/* Snappy.maxlength_compressed (src/Snappy.jl:80-82): 32 + n + n/6.
 * ccall twin: snappy_max_compressed_length (test/libsnappy.jl:7). */
size_t snappy_b200_max_compressed_length(size_t source_length);

/* Snappy.compress(::Vector{UInt8}) (src/Snappy.jl:20-36).  in/out are HOST pointers.
 * *out_len: in = capacity of `out` (>= max_compressed_length(n)), out = compressed length.
 * ccall twin: snappy_compress (test/libsnappy.jl:9-12). */
int snappy_b200_compress(const uint8_t *in, size_t n, uint8_t *out, size_t *out_len);

/* Snappy.length_uncompressed (src/Snappy.jl:90-92 -> varint.jl:12-37).  Host only, no GPU.
 * ccall twin: snappy_uncompressed_length (test/libsnappy.jl:20-23). */
int snappy_b200_uncompressed_length(const uint8_t *in, size_t n, size_t *result);

/* Snappy.uncompress (src/Snappy.jl:46-52).  in/out are HOST pointers.
 * *out_len: in = capacity of `out` (>= uncompressed_length), out = uncompressed length.
 * ccall twin: snappy_uncompress (test/libsnappy.jl:25-28). */
int snappy_b200_uncompress(const uint8_t *in, size_t n, uint8_t *out, size_t *out_len);

/* snappy_validate_compressed_buffer / IsValidCompressedBuffer: would snappy_b200_uncompress accept `in`?  Returns
 * exactly the status uncompress returns when the output capacity is unlimited: SNAPPY_B200_OK or one of the
 * reference's statuses 2..6 (never BUFFER_TOO_SMALL); 8..10 for device problems only.  Takes no output buffer and
 * writes nothing: the stream is judged on the GPU from its element headers and output positions (DESIGN.md section 4,
 * "Validation").  `in` is a HOST pointer (pinned or pageable).
 * ccall twin: snappy_validate_compressed_buffer (snappy-c). */
int snappy_b200_validate_compressed_buffer(const uint8_t *in, size_t n);

/* ---- device-resident API (the GB/s targets are quoted on these) --------------------------- */

/* Same as snappy_b200_compress but d_in / d_out are DEVICE pointers; `stream` is a cudaStream_t
 * (NULL = default stream).  out_cap >= max_compressed_length(n).
 * d_frag_index (optional, device, (nfrag+1) x uint64): side index -- byte offset inside the
 * stream of each 64 KiB fragment's first element; entry nfrag = total stream length.
 * nfrag = ceil(n / 65536).  The call synchronises `stream` before returning *out_len. */
int snappy_b200_compress_device(const uint8_t *d_in, size_t n, uint8_t *d_out, size_t out_cap,
                                size_t *out_len, uint64_t *d_frag_index, void *stream);

/* Same as snappy_b200_uncompress on DEVICE pointers.  d_frag_index (optional): the side index
 * written by snappy_b200_compress_device; NULL = arbitrary stream (segmented speculative parse).
 * A wrong index cannot change the result: the indexed path validates every fragment and falls
 * back to the index-free path on any inconsistency.  Synchronises `stream`. */
int snappy_b200_uncompress_device(const uint8_t *d_in, size_t n, uint8_t *d_out, size_t out_cap,
                                  size_t *out_len, const uint64_t *d_frag_index, void *stream);

/* snappy_b200_validate_compressed_buffer on DEVICE memory.  d_frag_index (optional): a side index as for
 * uncompress_device; right or wrong, it cannot change the result.  *uncompressed_len (optional) receives the claimed
 * length when the header parses.  Device memory: the parse's O(n / parse chunk) plus 17 bytes per claimed 64 KiB
 * fragment, never an output of `claimed` bytes.
 * Synchronises `stream`. */
int snappy_b200_validate_device(const uint8_t *d_in, size_t n, const uint64_t *d_frag_index,
                                size_t *uncompressed_len, void *stream);

/* ---- batched API: many independent streams (Parquet-page-like), one stream per page ------- */

/* Page i is d_in + in_offsets[i], in_sizes[i] bytes; its stream (own varint header, own table
 * size -- src/Snappy.jl:26-27 apply per page) is written at d_out + out_offsets[i] where the
 * caller reserved max_compressed_length(in_sizes[i]) bytes; out_sizes[i] receives its length.
 * All arrays are DEVICE arrays of `count` entries.  Synchronises `stream`. */
int snappy_b200_compress_batched_device(const uint8_t *d_in, const uint64_t *d_in_offsets,
                                        const uint32_t *d_in_sizes, size_t count, uint8_t *d_out,
                                        const uint64_t *d_out_offsets, uint32_t *d_out_sizes,
                                        void *stream);

/* Inverse: stream i is d_in + in_offsets[i] (in_sizes[i] bytes); its bytes go to
 * d_out + out_offsets[i], out_caps[i] = room there; out_sizes[i] receives the length and
 * d_statuses[i] the per-page snappy_b200_status.  Returns OK when the batch ran; per-page
 * failures are reported in d_statuses only. */
int snappy_b200_uncompress_batched_device(const uint8_t *d_in, const uint64_t *d_in_offsets,
                                          const uint32_t *d_in_sizes, size_t count, uint8_t *d_out,
                                          const uint64_t *d_out_offsets, const uint32_t *d_out_caps,
                                          uint32_t *d_out_sizes, int32_t *d_statuses, void *stream);

/* Validation form of uncompress_batched_device: d_statuses[i] = what uncompress_batched_device reports for page i
 * with unlimited room (never BUFFER_TOO_SMALL), d_claimed[i] = the page's claimed length (0 when its header does not
 * parse).  No output.  DEVICE arrays of `count` entries.  Synchronises `stream`. */
int snappy_b200_validate_batched_device(const uint8_t *d_in, const uint64_t *d_in_offsets,
                                        const uint32_t *d_in_sizes, size_t count, uint32_t *d_claimed,
                                        int32_t *d_statuses, void *stream);

/* ---- shard API: multi-GPU sharding on whole-fragment boundaries --------------------------- */

/* Compress a contiguous run of whole 64 KiB fragments of a stream whose TOTAL length is
 * total_len (the hash-table size comes from the total, src/Snappy.jl:27).  d_shard holds
 * shard_len bytes starting at a multiple of 65536 inside the stream; only the last shard may
 * be ragged.  Writes the compacted element bytes of the shard (NO varint header) to d_out and
 * its length to *out_len; the caller concatenates the shards behind
 * snappy_b200_encode_header(total_len).  d_frag_sizes (optional, device, one uint32 per fragment
 * of the shard) receives each fragment's compressed size.  Synchronises `stream`. */
int snappy_b200_compress_shard_device(const uint8_t *d_shard, size_t shard_len, uint64_t total_len,
                                      uint8_t *d_out, size_t out_cap, size_t *out_len,
                                      uint32_t *d_frag_sizes, void *stream);

/* Decode fragments of a stream given their element byte ranges: fragment i of the shard is
 * d_in[frag_offsets[i] .. frag_offsets[i+1]) and decodes to d_out + i*65536 (the last one may
 * be short: out_len total bytes expected).  Used by each rank on its own slice. */
int snappy_b200_uncompress_shard_device(const uint8_t *d_in, const uint64_t *d_frag_offsets,
                                        size_t nfrag, uint8_t *d_out, size_t out_len, void *stream);

/* Batched forms of the two shard calls: `count` shards (runs of whole fragments, possibly of
 * different streams) go through ONE kernel pass, which is what keeps the GPU full when a rank
 * holds many small shards (8 streams x 1/8 each).  The arrays are HOST arrays of `count` entries
 * whose pointer members are DEVICE pointers; d_frag_sizes (and its entries) may be NULL. */
int snappy_b200_compress_shards_device(const uint8_t *const *d_shards, const size_t *shard_lens,
                                       const uint64_t *total_lens, size_t count,
                                       uint8_t *const *d_outs, const size_t *out_caps,
                                       size_t *out_lens, uint32_t *const *d_frag_sizes, void *stream);
int snappy_b200_uncompress_shards_device(const uint8_t *const *d_ins,
                                         const uint64_t *const *d_frag_offsets,
                                         const size_t *out_lens, size_t count,
                                         uint8_t *const *d_outs, void *stream);

/* ---- multi-GPU communicator: the sharded path with its exchange steps inside the library -------------------
 * (SURVEY.md 8(e); replaces the implicit contiguous write of src/Snappy.jl:25-35 across GPUs.)
 * One process per GPU.  Stream s of a call is OWNED by rank s mod world; rank r holds, of every stream, the run of
 * whole 64 KiB fragments that whole-fragment sharding gives it: with nfrag = ceil(total/65536), the first
 * nfrag mod world ranks hold nfrag/world + 1 fragments, the others nfrag/world, in rank order.
 * Exchange steps, all on the caller's stream: ncclAllGather of the compressed byte counts, then every fragment is
 * stored straight into the owner's buffer through a peer-mapped pointer (cudaIpc, NVLink), side-index entries
 * included; uncompress loads each rank's compressed range from the owner the same way.  NCCL is bound at run time
 * (the copy already loaded in the process, else libnccl.so.2). */
typedef struct snappy_b200_comm snappy_b200_comm;

/* Rank 0 makes the 128-byte id (ncclGetUniqueId); the host's own plumbing (torch.distributed, MPI.jl, a file)
 * carries it to the other ranks. */
int snappy_b200_comm_unique_id(uint8_t id[128]);
/* Collective over `world` processes, each on its own GPU (the calling thread's device).  world == 1 needs no id. */
int snappy_b200_comm_create(const uint8_t id[128], int rank, int world, snappy_b200_comm **out);
/* A world whose `world` ranks all live in this process on the current device: no NCCL, no IPC; per-rank argument
 * arrays then carry world x nstreams entries, rank-major.  What a single GPU uses to push many streams through one
 * kernel pass (world = 1), and what lets one GPU run the exact multi-rank data path (tests). */
int snappy_b200_comm_create_loopback(int world, snappy_b200_comm **out);
void snappy_b200_comm_destroy(snappy_b200_comm *comm);
int snappy_b200_comm_info(const snappy_b200_comm *comm, int *world, int *nlocal, int *rank0);

/* Collective.  d_shards / shard_lens: nlocal x nstreams entries (rank-major): the local ranks' runs of every stream
 * (device pointers; NULL / 0 where a rank's run is empty).  total_lens[nstreams]: the same on every rank.
 * For every stream owned by a local rank: out_streams[s] = device pointer to the assembled stream (header +
 * elements), out_index[s] = its side index (nfrag + 1 offsets); both point into the communicator's arena and stay
 * valid until the next call on it.  out_lens[s] is set for EVERY stream.  Other entries are NULL.
 * Bytes are identical to snappy_b200_compress_device on the whole stream.  Synchronises `stream`. */
int snappy_b200_comm_compress(snappy_b200_comm *comm, const uint8_t *const *d_shards, const size_t *shard_lens,
                              const uint64_t *total_lens, size_t nstreams, uint8_t **out_streams, size_t *out_lens,
                              uint64_t **out_index, void *stream);

/* Collective inverse.  For streams owned by a local rank: d_streams[s] / stream_lens[s] (any device memory, or the
 * pointers comm_compress returned) and optionally d_index[s] (NULL, or d_index == NULL: the owner parses its stream).
 * d_outs: nlocal x nstreams device pointers; each receives that rank's run of the stream (the output stays
 * sharded).  statuses (optional, nstreams): the reference's status per stream, agreed by all ranks
 * (src/internal.jl:499,505,518, src/Snappy.jl:50); BAD_ARGUMENT marks a valid stream that cannot be decoded in
 * shards (elements straddling 64 KiB output boundaries): decode it on one GPU.  Returns the first non-OK status. */
int snappy_b200_comm_uncompress(snappy_b200_comm *comm, const uint8_t *const *d_streams, const size_t *stream_lens,
                                const uint64_t *const *d_index, const uint64_t *total_lens, size_t nstreams,
                                uint8_t *const *d_outs, int *statuses, void *stream);

/* varint.jl:46-69 / :12-37 on the host (the stream header). Returns bytes written (1..5). */
int snappy_b200_encode_header(uint32_t value, uint8_t out[5]);
int snappy_b200_parse_header(const uint8_t *in, size_t n, uint32_t *value, size_t *header_len);

/* Host helper mirroring Snappy.find_match_length (src/internal.jl:344-387), which the
 * reference's tests call directly (test/runtests.jl:172).  0-based, `limit` exclusive. */
size_t snappy_b200_find_match_length(const uint8_t *a, size_t i1, size_t i2, size_t limit);

/* ---- side-index sidecar (SURVEY.md section 8(f)2) ----------------------------------------
 * The side index (nfrag + 1 offsets of the 64 KiB fragments inside a stream) lets any consumer
 * take the indexed decoder without the parse.  It cannot travel inside the stream (the format has
 * no room: a reference decoder would read a trailer as elements), so it travels NEXT to it, as a
 * small self-describing blob:
 *   "SB2IDX1\0" | u32 nfrag | u32 reserved | u64 uncompressed_len | u64 stream_len |
 *   varint(index[0]) varint(index[1]-index[0]) ... varint(index[nfrag]-index[nfrag-1]) | u32 fnv1a
 * All host code, no GPU.  A sidecar that does not match its stream can never change a result:
 * the indexed decoder validates every fragment and falls back to the index-free paths. */
size_t snappy_b200_index_pack_bound(size_t nfrag);
/* index: HOST array of nfrag + 1 offsets (index[0] = header length, index[nfrag] = stream length).
 * *out_len: in = capacity, out = bytes written. */
int snappy_b200_index_pack(const uint64_t *index, size_t nfrag, uint64_t uncompressed_len,
                           uint8_t *out, size_t *out_len);
/* *nfrag: in = capacity of index in fragments (index holds capacity + 1 entries), out = fragments.
 * Returns SNAPPY_B200_INVALID_INPUT for a malformed / truncated / checksum-failing sidecar. */
int snappy_b200_index_unpack(const uint8_t *in, size_t n, uint64_t *index, size_t *nfrag,
                             uint64_t *uncompressed_len, uint64_t *stream_len);

/* ---- instrumentation (bench.py roofline) ------------------------------------------------- */

/* Device time, in milliseconds, of the dominant kernel of the last compress (which=0) or
 * uncompress (which=1) call on this thread's context, measured with CUDA events recorded on
 * the launching stream around that kernel; and the number of kernels that call launched. */
float snappy_b200_last_kernel_ms(int which);
int snappy_b200_last_launch_count(int which);
/* Selects kernel variants for A/B testing (0 = default).  See DESIGN.md.
 * One option changes the BYTES the compressor emits (SURVEY.md 8(f)4, appendix B.4):
 *   "rules" = 0  Snappy.jl's rules (src/internal.jl:127-329): the reference, default;
 *           = 1  libsnappy <= 1.1.7 (ip_limit n-15, 60-byte literal with the short tag, table per fragment);
 *           = 2  Google snappy >= 1.1.9 (as 1, bucket = (hash >> 17) & mask, up to 32768 buckets): byte-identical
 *                to the C++ library current consumers link (checked against pyarrow's bundled codec).
 * Every setting produces a valid Snappy stream that any decoder (this one, Snappy.jl, libsnappy) accepts. */
void snappy_b200_set_option(const char *name, int value);
/* Current value of an option, or -1 for a name this build does not know.  "experiments" reads 1 in a build that
 * also holds the measured-and-rejected kernel designs (make -C snappy.jl_b200/csrc exp), 0 in the product build. */
int snappy_b200_get_option(const char *name);
/* With option "trace" = 1 the compress warps record when they began and finished every fragment (globaltimer ns;
 * begin carries the table placement in bit 0, end the SM number in its low 8 bits): 2 x uint64 per fragment of the
 * calling thread's last compress call.  Returns the fragments copied.  tools/trace_frags.py turns it into the
 * utilisation timeline and the length of the launch's tail. */
size_t snappy_b200_debug_trace(uint64_t *out, size_t max_frags);

#ifdef __cplusplus
}
#endif
#endif
