// decompress.cuh -- Snappy raw-format decoder kernels for sm_100a, following the reference's
// decoder semantics (src/Snappy.jl:46-52, src/internal.jl:411-527) including its quirks
// (strict `ip < last` loop bound, zero-padded trailer, UInt32 literal-length wrap-around).
#pragma once
#include "common.cuh"

namespace sb200 {

struct DecodeResult {
    int status;        // ST_* of the first failing element in stream order (ST_OK if none)
    u32 fallback;      // indexed path: some fragment was inconsistent with the side index
    u64 produced;      // output bytes produced
    u64 err_op;        // output position at which the error fired
};

// One element header decoded from its tag byte `c` and the (zero-padded) 4 bytes behind it.
// CHAR_TABLE (src/internal.jl:47-80) is evaluated arithmetically: bits 0-7 length,
// 8-10 offset high bits, 11-13 extra bytes; WORDMASK (:83-85) becomes a shift.
struct Element {
    u32 len;      // literal: byte count (mod 2^32); copy: 1..64
    u32 offset;   // copy offset (0 for literals)
    u32 extra;    // bytes after the tag that belong to the header
    bool is_copy;
};

__device__ __forceinline__ Element decode_tag(u32 c, u32 tag4) {
    Element e;
    const u32 kind = c & 3, hi = c >> 2;
    if (kind == 0) {
        e.is_copy = false;
        e.offset = 0;
        if (hi < 60) {
            e.extra = 0;
            e.len = hi + 1;
        } else {
            e.extra = hi - 59;
            u32 mask = (e.extra == 4) ? 0xffffffffu : ((1u << (8 * e.extra)) - 1);
            e.len = 1 + (tag4 & mask);  // src/internal.jl:462, UInt32 arithmetic wraps
        }
    } else if (kind == 1) {
        e.is_copy = true;
        e.extra = 1;
        e.len = 4 + (hi & 7);
        e.offset = ((c >> 5) << 8) + (tag4 & 0xff);
    } else if (kind == 2) {
        e.is_copy = true;
        e.extra = 2;
        e.len = hi + 1;
        e.offset = tag4 & 0xffff;
    } else {
        e.is_copy = true;
        e.extra = 4;
        e.len = hi + 1;
        e.offset = tag4;
    }
    return e;
}

// tag byte at ip and the next 4 bytes, zero-padded past `end` (src/internal.jl:426-430)
__device__ __forceinline__ void load_tag(const u8* __restrict__ in, u64 ip, u64 end, u32& c,
                                         u32& tag4) {
    if (ip + 12 <= end) {
        // three aligned 32-bit words cover the 5 bytes at any misalignment of the address
        const uintptr_t pa = reinterpret_cast<uintptr_t>(in + ip);
        const u32* w = reinterpret_cast<const u32*>(pa & ~(uintptr_t)3);
        const u32 sh = (u32)(pa & 3) * 8;
        u32 w0 = __ldg(w), w1 = __ldg(w + 1), w2 = __ldg(w + 2);
        u32 lo = __funnelshift_r(w0, w1, sh);
        u32 hi = __funnelshift_r(w1, w2, sh);
        c = lo & 0xff;
        tag4 = __funnelshift_r(lo, hi, 8);
    } else {
        c = in[ip];
        tag4 = 0;
#pragma unroll
        for (int k = 0; k < 4; k++)
            if (ip + 1 + k < end) tag4 |= (u32)in[ip + 1 + k] << (8 * k);
    }
}

// warp-cooperative copies -----------------------------------------------------------------
__device__ __forceinline__ void warp_copy_literal(u8* __restrict__ dst, const u8* __restrict__ src,
                                                  u64 len, u32 lane) {
    warp_copy_forward<true>(dst, src, len, lane);
}

// out[op+i] = out[op-offset+i], ascending i (src/internal.jl:477-481): for offset < len the
// source pattern of `offset` bytes repeats, so byte i reads op - offset + (i mod offset).
__device__ __forceinline__ void warp_copy_backref(u8* out, u64 op, u32 offset, u32 len, u32 lane) {
    const u8* src = out + (op - offset);
    u8* dst = out + op;
    if (offset >= len) {
        // the last source group of 16 may end above the copy's first byte only if offset < len + 15: then
        // the vector body would read bytes it is about to write, so it needs offset >= 16 as well
        if (offset >= 16) warp_copy_forward<false>(dst, src, len, lane);
        else
            for (u32 i = lane; i < len; i += 32) dst[i] = src[i];
    } else {
        for (u32 i = lane; i < len; i += 32) dst[i] = src[i % offset];
    }
}

// Exact serial decoder: one warp walks a stream element by element, reproducing the
// reference's status for every input (first error in stream order).  Used for arbitrary streams
// until the speculative parse has produced an index, and as the arbiter whenever the fast paths
// see anything inconsistent.  `ip0` is the first byte after the varint header.
// Range form: elements from *ip up to (not including) ip_stop, output position *op; returns the status of the first
// failing element (ST_OK if none).  The whole-stream decoder is the range [ip0, L) from op = 0 plus the final length
// check (src/Snappy.jl:50).
// kWrite = false: validation only -- the same walk, the same checks and the same op, but no byte is written and `out`
// is never touched (it may be null).
template <bool kWrite = true>
__device__ __forceinline__ int decode_exact_range(const u8* __restrict__ in, u64 L, u64& ip, u64 ip_stop,
                                                  u8* __restrict__ out, u64 n, u64& op, u32 lane) {
    while (ip < ip_stop && ip + 1 < L) {  // src/internal.jl:416
        u32 c, tag4;
        load_tag(in, ip, L, c, tag4);
        ip += 1;
        Element e = decode_tag(c, tag4);
        ip += e.extra;
        if (e.is_copy) {
            if (e.offset == 0 || (u64)e.offset > op) return ST_CORRUPT_COPY_OFFSET;  // :499
            if (n - op < e.len) return ST_CORRUPT_COPY_LENGTH;                       // :505
            if (kWrite) warp_copy_backref(out, op, e.offset, e.len, lane);
            op += e.len;
        } else {
            // avail_in may be negative when the header bytes ran past the end (:517-518)
            long long avail_in = (long long)L - (long long)ip;
            if (n - op < (u64)e.len || avail_in < (long long)e.len) return ST_CORRUPT_LITERAL;
            if (kWrite) warp_copy_literal(out + op, in + ip, e.len, lane);
            op += e.len;
            ip += e.len;
        }
        if (kWrite) __syncwarp();
    }
    return ST_OK;
}

template <bool kWrite = true>
__device__ __forceinline__ int decode_exact_warp(const u8* __restrict__ in, u64 L, u64 ip0,
                                                 u8* __restrict__ out, u64 n, u32 lane,
                                                 u64& produced) {
    u64 ip = ip0, op = 0;
    int status = decode_exact_range<kWrite>(in, L, ip, L, out, n, op, lane);
    if (status == ST_OK && op != n) status = ST_INVALID_INPUT;  // src/Snappy.jl:50
    produced = op;
    return status;
}

__global__ void __launch_bounds__(32)
k_decode_serial(const u8* __restrict__ in, u64 L, u64 ip0, u8* __restrict__ out, u64 n,
                DecodeResult* __restrict__ res) {
    const u32 lane = lane_id();
    u64 produced;
    int status = decode_exact_warp(in, L, ip0, out, n, lane, produced);
    if (lane == 0) {
        res->status = status;
        res->produced = produced;
        res->err_op = produced;
    }
}

// Status-only twin of k_decode_serial (snappy_b200_validate_*): no output buffer.
__global__ void __launch_bounds__(32)
k_validate_serial(const u8* __restrict__ in, u64 L, u64 ip0, u64 n, DecodeResult* __restrict__ res) {
    const u32 lane = lane_id();
    u64 produced;
    int status = decode_exact_warp<false>(in, L, ip0, nullptr, n, lane, produced);
    if (lane == 0) {
        res->status = status;
        res->produced = produced;
        res->err_op = produced;
    }
}

// Indexed decoder: one warp per 64 KiB output fragment, whose elements are
// in[frag_off[f] .. frag_off[f+1]) (side index from the compressor, or from the parse kernels).
// Elements are parsed 32 at a time (warp-uniform walk; lane k keeps element k), then executed
// lane-per-element in dependency rounds: an element may run once every output byte it reads lies
// below the `frontier` (the destination of the first unfinished element of the batch).
// Anything that is not a clean, self-contained fragment sets res->fallback and the caller reruns
// the exact serial decoder, so a wrong index can never change the result.
constexpr u32 kDecodeWarpsPerCta = 2;   // small CTAs: finished warps free their slot sooner (5.60 -> 5.53 ms)

// Decode the self-contained element run in[ip .. ie) into o[0 .. on).  Returns false when the run
// is not clean (bad element, reaches before o, does not end exactly at ie / on).
//
// Window-parallel parse: the 32 lanes decode the 32 byte positions base .. base+31 as if each were
// a tag (loop header of decompress_all_tags!, src/internal.jl:416-439, evaluated for every byte at
// once); the real chain inside the window is then the set of positions reachable from lane 0,
// found by pointer doubling on "position + element size" (5 rounds of reduce-or + shuffle).  The
// element that leaves the window gives the next window's base, so long literals are skipped in one
// hop.  A warp scan over the chain's lengths gives every element its output offset.
// Execution: short elements (<= kShortElem bytes) run one per lane, in dependency rounds: an
// element may go once every output byte it reads lies below the destination of the first
// unfinished element; long elements are copied by the whole warp when they become the first
// unfinished one (incremental_copy! / copy_literal!, src/internal.jl:477-527).
constexpr u32 kShortElem = 16;
// The window walk reads the stream front to back, 30-100 bytes per window, and 8 % of the decoder's warp time sits on
// the first use of a window's tag words (profiles/r02q_prof_decode.txt).  Build switch: one lane asks for the line
// kDecodePrefetch bytes ahead.  Measured 0 / 256 / 512 / 1024 bytes ahead into L2, 512 into L1: 4.78 / 4.79 / 4.71 /
// 4.78 / 4.79 ms per GiB (profiles/r02r_decode_variants.txt): within noise, so off.
#ifndef SB200_DECODE_PREFETCH
#define SB200_DECODE_PREFETCH 0
#endif
constexpr u32 kDecodePrefetch = SB200_DECODE_PREFETCH;

// branch-free form of decode_tag for the window parse (same fields; CHAR_TABLE / WORDMASK of
// src/internal.jl:47-85 evaluated arithmetically)
__device__ __forceinline__ void decode_tag_fast(u32 c, u32 tag4, u32& len, u32& offset, u32& extra,
                                                bool& is_copy) {
    const u32 kind = c & 3u, hi = c >> 2;
    extra = (kind == 0) ? (hi >= 60 ? hi - 59 : 0u) : (kind == 3 ? 4u : kind);
    const u32 mask = (extra >= 4) ? 0xffffffffu : ((1u << (8u * extra)) - 1u);
    const u32 v = tag4 & mask;
    is_copy = kind != 0;
    len = (kind == 0) ? (hi >= 60 ? 1u + v : hi + 1u) : (kind == 1 ? 4u + (hi & 7u) : hi + 1u);
    offset = (kind == 1) ? (((c >> 5) << 8) | v) : v;
}

// kWrite = false: the window parse, chain, scan and every check, without the execute loop (validation; `o` unused).
template <bool kWrite = true>
__device__ __forceinline__ bool decode_fast_warp(const u8* __restrict__ in, u64 ip, const u64 ie,
                                                 u8* __restrict__ o, const u32 on, const u32 lane) {
    if (ie - ip > 0xfffffff0ull) return false;
    const u8* __restrict__ src = in + ip;   // all positions below are relative to the run start
    const u32 nin = (u32)(ie - ip);
    u32 base = 0, op = 0;
    while (base < nin) {
        // ---- decode all 32 byte positions of the window
        const u32 p = base + lane;
        const bool inb = p < nin;
        const u32 rem = inb ? nin - p : 1u;  // bytes from p to the end of the run (>= 1)
#ifndef SB200_CPU_EMU
        if (kDecodePrefetch && lane == 0 && base + kDecodePrefetch < nin)
#ifdef SB200_DECODE_PREFETCH_L1
            asm volatile("prefetch.global.L1 [%0];" ::"l"(src + base + kDecodePrefetch));
#else
            asm volatile("prefetch.global.L2 [%0];" ::"l"(src + base + kDecodePrefetch));
#endif
#endif
        u32 c = 0, tag4 = 0;
        if (inb) {
            if (rem >= 12) {
                // three aligned words cover the 5 bytes at any misalignment of the address
                const uintptr_t pa = reinterpret_cast<uintptr_t>(src + p);
                const u32* w = reinterpret_cast<const u32*>(pa & ~(uintptr_t)3);
                const u32 sh = (u32)pa << 3;
                const u32 w0 = __ldg(w), w1 = __ldg(w + 1), w2 = __ldg(w + 2);
                const u32 lo = __funnelshift_r(w0, w1, sh), hi = __funnelshift_r(w1, w2, sh);
                c = lo & 0xffu;
                tag4 = __funnelshift_r(lo, hi, 8);
            } else {
                c = src[p];
#pragma unroll
                for (u32 k = 0; k < 4; k++)
                    if (1 + k < rem) tag4 |= (u32)src[p + 1 + k] << (8 * k);  // zero-padded, :426-430
            }
        }
        u32 elen0, eoff, extra;
        bool is_copy;
        decode_tag_fast(c, tag4, elen0, eoff, extra, is_copy);
        // element size, saturated to "one past the end of the run" when it does not fit
        const u32 hdr = 1u + extra;
        const bool fits = hdr <= rem && (is_copy || elen0 <= rem - hdr);
        const u32 size = fits ? hdr + (is_copy ? 0u : elen0) : rem + 1u;
        // 32: leaves the window (also when the element ends at or past the end: the run is over)
        u32 jump = (size >= 32u - lane || size >= rem) ? 32u : lane + size;
        const bool leaves = jump == 32u;
        // ---- positions reachable from lane 0 (the chain enters every window at its first byte)
        // (every element is at least 2 bytes long, so the chain has at most 16 positions in a window:
        // 4 rounds of doubling reach hops 0..15)
        u32 R = 1u;
#pragma unroll
        for (int r = 0; r < 4; r++) {
            const u32 m = (((R >> lane) & 1u) && jump < 32u) ? (1u << jump) : 0u;
            R |= __reduce_or_sync(kFullMask, m);
            const u32 j2 = __shfl_sync(kFullMask, jump, jump & 31u);
            jump = (jump < 32u) ? j2 : 32u;
        }
        const bool mine = (R >> lane) & 1u;
        // ---- validate the chain's elements (anything odd: let the exact decoder decide)
        bool bad = mine && (!inb || !fits || elen0 == 0 || elen0 > on);
        const u32 elen = mine ? elen0 : 0u;
        u32 incl = bad ? 0u : elen;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const u32 t = __shfl_up_sync(kFullMask, incl, d);
            if (lane >= (u32)d) incl += t;
        }
        const u32 total = __shfl_sync(kFullMask, incl, 31);
        const u32 dst = op + incl - elen;
        bad = bad || (mine && is_copy && (eoff == 0 || eoff > dst));
        const u32 exitm = __ballot_sync(kFullMask, mine && leaves);
        if (__any_sync(kFullMask, bad) || exitm == 0 || total > on - op) return false;
        const u32 nbase = __shfl_sync(kFullMask, p + size, (u32)__ffs((int)exitm) - 1u);
        if (!kWrite) {
            op += total;
            base = nbase;
            continue;
        }
        // ---- execute
        const u32 lsrc = p + hdr;  // literal bytes start behind the header
        // highest output byte (exclusive) the element reads; literals read none
        const u32 need = (mine && is_copy) ? (dst - eoff + min(elen, eoff)) : 0u;
        u32 pending = R;
        while (pending) {
            const u32 f = (u32)__ffs((int)pending) - 1u;
            const u32 frontier = __shfl_sync(kFullMask, dst, f);
            const u32 flen = __shfl_sync(kFullMask, elen, f);
            if (flen > kShortElem) {
                const u32 fcopy = __shfl_sync(kFullMask, (u32)is_copy, f);
                const u32 fx = __shfl_sync(kFullMask, is_copy ? eoff : lsrc, f);
                if (fcopy) warp_copy_backref(o, frontier, fx, flen, lane);
                else warp_copy_literal(o + frontier, src + fx, flen, lane);
                __syncwarp();
                pending &= ~(1u << f);
                continue;
            }
            const bool ready = ((pending >> lane) & 1u) && elen <= kShortElem && need <= frontier;
            if (ready) {
                u8* d = o + dst;
                if (is_copy && eoff < elen) {
                    const u8* s = o + (dst - eoff);
                    for (u32 i = 0, k = 0; i < elen; i++) {  // pattern of `offset` bytes repeats
                        d[i] = s[k];
                        k = (k + 1 == eoff) ? 0 : k + 1;
                    }
                } else {
                    // <= 16 source bytes through the aligned words that hold them (only words with at least
                    // one wanted byte are read), then one predicated byte store per position: no loop
                    const uintptr_t sa = reinterpret_cast<uintptr_t>(is_copy ? o + (dst - eoff) : src + lsrc);
                    const u32* w = reinterpret_cast<const u32*>(sa & ~(uintptr_t)3);
                    const u32 sh = (u32)sa << 3;
                    const u32 last = (((u32)sa & 3u) + elen - 1u) >> 2;  // index of the last word needed (0..4)
                    u32 w0, w1 = 0, w2 = 0, w3 = 0, w4 = 0;
                    if (is_copy) {  // output bytes written earlier in this kernel: coherent loads
                        w0 = w[0];
                        if (last >= 1) w1 = w[1];
                        if (last >= 2) w2 = w[2];
                        if (last >= 3) w3 = w[3];
                        if (last >= 4) w4 = w[4];
                    } else {  // input: read-only path
                        w0 = __ldg(w);
                        if (last >= 1) w1 = __ldg(w + 1);
                        if (last >= 2) w2 = __ldg(w + 2);
                        if (last >= 3) w3 = __ldg(w + 3);
                        if (last >= 4) w4 = __ldg(w + 4);
                    }
                    const u32 b0 = __funnelshift_r(w0, w1, sh), b1 = __funnelshift_r(w1, w2, sh),
                              b2 = __funnelshift_r(w2, w3, sh), b3 = __funnelshift_r(w3, w4, sh);
#pragma unroll
                    for (u32 i = 0; i < 16; i++) {
                        const u32 word = i < 4 ? b0 : (i < 8 ? b1 : (i < 12 ? b2 : b3));
                        if (i < elen) d[i] = (u8)(word >> (8 * (i & 3)));
                    }
                }
            }
            __syncwarp();
            pending &= ~__ballot_sync(kFullMask, ready);
        }
        op += total;
        base = nbase;
    }
    return base == nin && op == on;
}

// in_begin / in_end: the element bytes of the whole stream are in[in_begin .. in_end); the index
// must start at in_begin and end at in_end.
// One entry per shard for the batched shard API (fragments [frag_begin, frag_begin + nfrag) of the
// launch): element bytes of fragment i are in[frag_off[i] .. frag_off[i+1]), output at out + i*65536.
struct DecodeDesc {
    const u8* in;
    const u64* frag_off;
    u8* out;
    u64 out_len;
    u32 frag_begin, nfrag;
    u32* flag;   // optional: raised when a fragment of THIS shard is not clean (besides res->fallback)
};

template <int kMinBlocks>
__global__ void __launch_bounds__(kDecodeWarpsPerCta * 32, kMinBlocks * 4 / kDecodeWarpsPerCta)
k_decode_fragments(const u8* __restrict__ in, const u64* __restrict__ frag_off, u32 nfrag, u32 first,
                   u32 count, u64 in_begin, u64 in_end, u8* __restrict__ out, u64 out_len,
                   DecodeResult* __restrict__ res, const DecodeDesc* __restrict__ descs = nullptr,
                   u32 ndesc = 0, const u64* __restrict__ out_start = nullptr, u8* __restrict__ tile_flags = nullptr) {
    // fragments [first, first + count) of the nfrag the index describes (ranges let the host
    // overlap the device->host copy of finished output with the decoding of the rest)
    const u32 lane = lane_id();
    const u32 local = blockIdx.x * kDecodeWarpsPerCta + (threadIdx.x >> 5);
    if (local >= count) return;
    u32 f = first + local;
    u32* shard_flag = nullptr;
    if (descs) {  // batched shards: find the shard, take its own arrays and bounds
        u32 k = 0;
        while (k + 1 < ndesc && descs[k + 1].frag_begin <= f) k++;
        shard_flag = descs[k].flag;
        in = descs[k].in;
        frag_off = descs[k].frag_off;
        out = descs[k].out;
        out_len = descs[k].out_len;
        nfrag = descs[k].nfrag;
        f -= descs[k].frag_begin;
        in_begin = frag_off[0];
        in_end = frag_off[nfrag];
    }
    const u64 ip = frag_off[f];
    const u64 ie = frag_off[f + 1];
    // out_start (index built by the parse for a foreign stream): tile f begins at the element that covers output
    // byte f * 65536 -- a literal may straddle the boundary -- so tiles start where out_start says
    const u64 ob = out_start ? out_start[f] : (u64)f * kBlockSize;
    u64 oe = out_start ? out_start[f + 1] : ob + kBlockSize;
    if (oe > out_len) oe = out_len;
    const u32 on = (oe >= ob && oe - ob <= 0xffffffffull) ? (u32)(oe - ob) : 0u;
    bool ok = (ie >= ip) && (ie <= in_end) && (f != 0 || ip == in_begin) &&
              (f != nfrag - 1 || ie == in_end) && (oe >= ob) && (ob <= out_len);
    if (ok) ok = decode_fast_warp(in, ip, ie, out + ob, on, lane);
    if (!ok && lane == 0) {
        atomicOr(&res->fallback, 1u);
        if (shard_flag) atomicOr(shard_flag, 1u);
        if (tile_flags) tile_flags[f] = 1;
    }
}

// Validation over a side index: one warp per 64 KiB fragment with the per-fragment rules of k_decode_fragments
// (fragment 0 starts behind the header, the last ends at in_end, fragment f is exactly in[frag_off[f] ..
// frag_off[f+1]) with exactly its output length, no copy reaches before the fragment), but no output: a fragment that
// is not clean raises res->fallback and the index-free chain decides.
__global__ void __launch_bounds__(kDecodeWarpsPerCta * 32)
k_validate_fragments(const u8* __restrict__ in, const u64* __restrict__ frag_off, u32 nfrag, u64 in_begin,
                     u64 in_end, u64 out_len, DecodeResult* __restrict__ res) {
    const u32 lane = lane_id();
    const u32 f = blockIdx.x * kDecodeWarpsPerCta + (threadIdx.x >> 5);
    if (f >= nfrag) return;
    const u64 ip = frag_off[f];
    const u64 ie = frag_off[f + 1];
    const u64 ob = (u64)f * kBlockSize;
    u64 oe = ob + kBlockSize;
    if (oe > out_len) oe = out_len;
    const u32 on = oe >= ob ? (u32)(oe - ob) : 0u;
    bool ok = (ie >= ip) && (ie <= in_end) && (f != 0 || ip == in_begin) && (f != nfrag - 1 || ie == in_end) &&
              (oe >= ob);
    if (ok) ok = decode_fast_warp<false>(in, ip, ie, nullptr, on, lane);
    if (!ok && lane == 0) atomicOr(&res->fallback, 1u);
}

// Status arbiter, bounded: only the tiles the parallel decoder rejected (tile_flags) are decoded again, one warp,
// element by element with the reference's checks (decode_exact_range), in stream order.  Every tile before the first
// rejected one passed the (stricter) clean-tile validation, so its bytes are final and the reference accepts it too:
// the first error this walk meets is the reference's first error.  A rejected tile that decodes fine in whole-stream
// terms (a copy that reaches into an earlier tile) is simply complete afterwards.  The walk goes on through the
// following tiles until it stands exactly on the start of a tile that was not rejected.
template <bool kWrite>
__device__ __forceinline__ void serial_tiles_walk(const u8* __restrict__ in, u64 L, const u64* __restrict__ index,
                                                  const u64* __restrict__ out_start, u32 nfrag,
                                                  const u8* __restrict__ tile_flags, u8* __restrict__ out, u64 n,
                                                  DecodeResult* __restrict__ res) {
    const u32 lane = lane_id();
    int status = ST_OK;
    u64 ip = 0, op = 0;
    bool ran_to_end = false;
    u32 f = 0;
    while (f < nfrag && status == ST_OK) {
        if (!tile_flags[f]) {
            f++;
            continue;
        }
        // a known start: this tile's own index entry, else the nearest earlier one (tile 0 starts behind the header)
        u32 s = f;
        while (s > 0 && index[s] >= L) s--;
        ip = index[s];
        op = out_start ? out_start[s] : (u64)s * kBlockSize;
        u32 cur = s;
        for (;;) {
            // one element at a time, so that the walk can stop on a tile start
            u64 stop = ip + 1;
            status = decode_exact_range<kWrite>(in, L, ip, stop, out, n, op, lane);
            if (status != ST_OK) break;
            if (ip + 1 >= L) {  // end of the stream (a lone trailing byte is ignored, src/internal.jl:416)
                ran_to_end = true;
                break;
            }
            while (cur + 1 < nfrag && op >= (out_start ? out_start[cur + 1] : (u64)(cur + 1) * kBlockSize)) cur++;
            const u64 ts = out_start ? out_start[cur] : (u64)cur * kBlockSize;
            if (cur > f && op == ts && ip == index[cur] && !tile_flags[cur]) break;  // back on a good tile
        }
        if (ran_to_end || status != ST_OK) break;
        f = cur;
    }
    if (status == ST_OK && ran_to_end && op != n) status = ST_INVALID_INPUT;  // src/Snappy.jl:50
    if (lane == 0) {
        res->status = status;
        res->produced = op;
        res->err_op = op;
    }
}

__global__ void __launch_bounds__(32)
k_decode_serial_tiles(const u8* __restrict__ in, u64 L, const u64* __restrict__ index,
                      const u64* __restrict__ out_start, u32 nfrag, const u8* __restrict__ tile_flags,
                      u8* __restrict__ out, u64 n, DecodeResult* __restrict__ res) {
    serial_tiles_walk<true>(in, L, index, out_start, nfrag, tile_flags, out, n, res);
}

// Status-only twin (validation): the same walk from the same starts with the same checks, tracking op only.
__global__ void __launch_bounds__(32)
k_validate_serial_tiles(const u8* __restrict__ in, u64 L, const u64* __restrict__ index,
                        const u64* __restrict__ out_start, u32 nfrag, const u8* __restrict__ tile_flags, u64 n,
                        DecodeResult* __restrict__ res) {
    serial_tiles_walk<false>(in, L, index, out_start, nfrag, tile_flags, nullptr, n, res);
}

// Batched pages: one warp per independent stream (own varint header).  Fast path first; the exact
// decoder arbitrates anything unusual so the per-page status equals the reference's.
__device__ __forceinline__ int parse_varint_dev(const u8* __restrict__ in, u64 L, u32& value, u32& hdr) {
    u32 result = 0;
    for (u32 i = 0; i < 5; i++) {  // src/varint.jl:12-37
        if (i >= L) return ST_BAD_VARINT;
        u32 b = in[i];
        result |= (b & 0x7f) << (7 * i);
        if (i < 4 ? (b < 0x80) : (b < 0x10)) {
            value = result;
            hdr = i + 1;
            return ST_OK;
        }
    }
    return ST_BAD_VARINT;
}

__global__ void __launch_bounds__(kDecodeWarpsPerCta * 32)
k_decode_pages(const u8* __restrict__ in, const u64* __restrict__ in_off,
               const u32* __restrict__ in_size, u32 count, u8* __restrict__ out,
               const u64* __restrict__ out_off, const u32* __restrict__ out_cap,
               u32* __restrict__ out_size, int* __restrict__ statuses) {
    const u32 lane = lane_id();
    const u32 pg = blockIdx.x * kDecodeWarpsPerCta + (threadIdx.x >> 5);
    if (pg >= count) return;
    const u8* pin = in + in_off[pg];
    const u64 L = in_size[pg];
    u8* pout = out + out_off[pg];
    u32 claimed = 0, hdr = 0;
    int status = parse_varint_dev(pin, L, claimed, hdr);
    if (status == ST_OK && claimed > out_cap[pg]) status = 7;  // SNAPPY_B200_BUFFER_TOO_SMALL
    if (status == ST_OK) {
        bool ok = (claimed <= kBlockSize) && decode_fast_warp(pin, hdr, L, pout, claimed, lane);
        if (!ok) {
            u64 produced;
            __syncwarp();
            status = decode_exact_warp(pin, L, hdr, pout, claimed, lane, produced);
        }
    }
    if (lane == 0) {
        statuses[pg] = status;
        out_size[pg] = (status == ST_OK) ? claimed : 0;
    }
}

// Status-only twin of k_decode_pages (snappy_b200_validate_batched_device): no output, no capacity; writes the claimed
// length (0 when the header does not parse) and the reference's status of every page.
__global__ void __launch_bounds__(kDecodeWarpsPerCta * 32)
k_validate_pages(const u8* __restrict__ in, const u64* __restrict__ in_off, const u32* __restrict__ in_size, u32 count,
                 u32* __restrict__ claimed_out, int* __restrict__ statuses) {
    const u32 lane = lane_id();
    const u32 pg = blockIdx.x * kDecodeWarpsPerCta + (threadIdx.x >> 5);
    if (pg >= count) return;
    const u8* pin = in + in_off[pg];
    const u64 L = in_size[pg];
    u32 claimed = 0, hdr = 0;
    int status = parse_varint_dev(pin, L, claimed, hdr);
    if (status == ST_OK) {
        bool ok = (claimed <= kBlockSize) && decode_fast_warp<false>(pin, hdr, L, nullptr, claimed, lane);
        if (!ok) {
            u64 produced;
            __syncwarp();
            status = decode_exact_warp<false>(pin, L, hdr, nullptr, claimed, lane, produced);
        }
    }
    if (lane == 0) {
        statuses[pg] = status;
        claimed_out[pg] = status == ST_BAD_VARINT ? 0u : claimed;
    }
}

}  // namespace sb200
