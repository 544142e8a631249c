// run_decode_parsed.cpp -- runs the REAL index-free decode chain (snappy.jl_b200/csrc/parse.cuh + decompress.cuh) on
// the CPU (cuda_shim.h) for arbitrary, typically corrupt, streams and checks the status -- and the bytes when the status
// is OK -- against the oracle's decoder (sjo_uncompress_ex).  TEST INFRASTRUCTURE ONLY (tests/test_decode_corruption.py,
// tools/cpu_warp/fuzz.py).  Every file is a STREAM.
//
//   mode "parsed": uncompress_device_locked without a side index, kernel for kernel (snappy_b200.cu):
//       parse_varint + out_cap check                       uncompress_device_locked   (:1131-1143)
//       relaxed parse, counters initialised as the product  build_index_segment        (:962-995)
//       first_err / total != claimed verdicts (path 1)      decode_parsed_locked       (:1049-1058)
//       clean cuts when CLEAN_CUTS=1 (default)              decode_parsed_locked       (:1061-1082)
//       k_first_missing -> tvalid                           decode_parsed_locked       (:1083-1095)
//       k_decode_fragments with tile flags (path 1)         decode_parsed_locked       (:1096-1111)
//       k_decode_serial_tiles (path 2)                      decode_parsed_locked       (:1112-1124)
//       k_decode_serial when nothing came of the parse      uncompress_device_locked   (:1154-1155, path 3)
//     The multi-warp helpers (k_scan_sizes, k_suffix_min) are plain loops here.  Per stream: the status, the path (the
//     numbers of the option last_decode_path; "-" when the header alone decides) and "0 mismatches" or "MISMATCH".
//     The output buffer carries sentinel bytes behind `claimed` that no path may touch.  PSHIFT selects
//     parse_chunk_log2 (default 10).
//   mode "pages": every stream is one page of ONE k_decode_pages launch, plus two empty pages (status BAD_VARINT);
//     every fourth non-empty page gets out_cap = claimed - 1 (status BUFFER_TOO_SMALL).  Per page: status, out_size,
//     the bytes on OK, and nothing written at or past out_cap (sentinels up to the next page's slot).
//   mode "validate": validate_device_locked (snappy_b200.cu), kernel for kernel, with a NULL output pointer: the
//     status-only kernels must never write.  IDX_SUFFIX=.x: the side index of stream F is read from F.x (nfrag + 1
//     little-endian u64) when that file exists (path 0, k_validate_fragments).  Per stream: the validation status, the
//     `parsed` mode's status for the same stream, the path, "step3" when a complete error-free parse decided alone,
//     and "0 mismatches" when both statuses equal the oracle's.
//   mode "validate-pages": every stream as one page of ONE k_validate_pages launch (no output), plus two empty pages.
//     Per page: status and claimed length against the oracle.
//   g++ -O1 -std=c++17 -DSB200_CPU_EMU -Itools/cpu_warp tools/cpu_warp/run_decode_parsed.cpp oracle.o
//   ./a.out parsed|pages|validate|validate-pages file...
#include "../../snappy.jl_b200/csrc/parse.cuh"

#include <string>
#include <vector>

extern "C" {
#include "../../oracle/snappy_oracle.h"
}

namespace sb200 {
u8 smem[1024] __attribute__((aligned(128)));
}
using namespace sb200;
using cpu_warp::launch_independent_threads;

constexpr u8 kSentinel = 0xEE;
constexpr size_t kGuard = 256;  // sentinel bytes behind every output

static void as_warp(u32 block, u32 tid_base, u32 block_dim) {
    cpu_warp::W().block = block;
    cpu_warp::W().tid_base = tid_base;
    cpu_warp::W().block_dim = block_dim;
}

struct FragArgs {
    const u8* in;
    const u64* idx;
    u32 nfrag, count;
    u64 hdr, n;
    u8* out;
    u64 claimed;
    DecodeResult* res;
    const u64* ost;
    u8* tf;
};
static void entry_fragments(void* p) {
    const FragArgs& a = *(const FragArgs*)p;
    k_decode_fragments<8>(a.in, a.idx, a.nfrag, 0u, a.count, a.hdr, a.n, a.out, a.claimed, a.res, nullptr, 0u, a.ost, a.tf);
}
struct TileArgs {
    const u8* in;
    u64 n;
    const u64 *idx, *ost;
    u32 nfrag;
    const u8* tf;
    u8* out;
    u64 claimed;
    DecodeResult* res;
};
static void entry_serial_tiles(void* p) {
    const TileArgs& a = *(const TileArgs*)p;
    k_decode_serial_tiles(a.in, a.n, a.idx, a.ost, a.nfrag, a.tf, a.out, a.claimed, a.res);
}
struct SerialArgs {
    const u8* in;
    u64 n, hdr;
    u8* out;
    u64 claimed;
    DecodeResult* res;
};
static void entry_serial(void* p) {
    const SerialArgs& a = *(const SerialArgs*)p;
    k_decode_serial(a.in, a.n, a.hdr, a.out, a.claimed, a.res);
}
struct PageArgs {
    const u8* in;
    const u64* in_off;
    const u32* in_size;
    u32 count;
    u8* out;
    const u64* out_off;
    const u32* out_cap;
    u32* out_size;
    int* statuses;
};
static void entry_pages(void* p) {
    const PageArgs& a = *(const PageArgs*)p;
    k_decode_pages(a.in, a.in_off, a.in_size, a.count, a.out, a.out_off, a.out_cap, a.out_size, a.statuses);
}
struct VFragArgs {
    const u8* in;
    const u64* idx;
    u32 nfrag;
    u64 hdr, n, claimed;
    DecodeResult* res;
};
static void entry_validate_fragments(void* p) {
    const VFragArgs& a = *(const VFragArgs*)p;
    k_validate_fragments(a.in, a.idx, a.nfrag, a.hdr, a.n, a.claimed, a.res);
}
static void entry_validate_tiles(void* p) {
    const TileArgs& a = *(const TileArgs*)p;
    k_validate_serial_tiles(a.in, a.n, a.idx, a.ost, a.nfrag, a.tf, a.claimed, a.res);
}
static void entry_validate_serial(void* p) {
    const SerialArgs& a = *(const SerialArgs*)p;
    k_validate_serial(a.in, a.n, a.hdr, a.claimed, a.res);
}
struct VPageArgs {
    const u8* in;
    const u64* in_off;
    const u32* in_size;
    u32 count;
    u32* claimed;
    int* statuses;
};
static void entry_validate_pages(void* p) {
    const VPageArgs& a = *(const VPageArgs*)p;
    k_validate_pages(a.in, a.in_off, a.in_size, a.count, a.claimed, a.statuses);
}

// decode_parsed_locked (snappy_b200.cu:1027-1125) + its fall-back to k_decode_serial; returns the status, *path as
// last_decode_path reports it
// build_index_segment (snappy_b200.cu:945-1009), relaxed form, the whole stream as one segment; idx / ost seeded as
// decode_parsed_locked seeds them (:1040-1045)
struct Parse {
    u32 nfrag, nchunk;
    std::vector<u64> idx, ost, out_off;
    std::vector<u8> arena;
    ParseArrays pa;
    u64 pflags, total, first_err;
};
static void parse_stream(const u8* in, u64 n, u64 hdr, u32 claimed, u32 pshift, Parse& P) {
    const u32 nfrag = P.nfrag = (u32)(((u64)claimed + kBlockSize - 1) / kBlockSize);
    P.idx.assign(nfrag + 1, ~0ull);
    P.ost.assign(nfrag + 1, ~0ull);
    std::vector<u64>& idx = P.idx;
    std::vector<u64>& ost = P.ost;
    idx[0] = hdr;
    ost[0] = 0;
    const u64 pchunk = 1ull << pshift, body = n - hdr;
    const u32 nchunk = P.nchunk = (u32)((body + pchunk - 1) / pchunk);
    P.arena.assign(ParseArrays::bytes(nchunk) + 64, 0);
    ParseArrays& pa = P.pa;
    pa.carve(P.arena.data(), nchunk);
    memset(pa.counters, 0, 64);                    // :962
    memset((u8*)pa.counters + 16, 0xff, 8);        // :963 first failing element: none yet
    const u32 pgrid = (nchunk + kParseThreads - 1) / kParseThreads, lgrid = (nchunk + 255) / 256;
    launch_independent_threads(pgrid, kParseThreads, k_parse_guess, in, n, hdr, nchunk, pa, n, pshift);
    launch_independent_threads(pgrid, kParseThreads, k_parse_bridge, in, n, hdr, nchunk, pa, n, pshift);
    std::vector<u32> next_orig(pa.next_a, pa.next_a + nchunk);
    u32 *nx = pa.next_a, *nx2 = pa.next_b;
    for (u32 span = 1; span < nchunk; span <<= 1) {
        launch_independent_threads(lgrid, 256u, k_parse_reach, nchunk, (const u32*)nx, nx2, pa.reach);
        u32* t = nx;
        nx = nx2;
        nx2 = t;
    }
    launch_independent_threads(lgrid, 256u, k_parse_reach, nchunk, (const u32*)nx, nx2, pa.reach);
    launch_independent_threads(pgrid, kParseThreads, k_parse_entries, in, n, hdr, nchunk, pa, (const u32*)next_orig.data(), 0, n, pshift);
    launch_independent_threads(pgrid, kParseThreads, k_parse_entries, in, n, hdr, nchunk, pa, (const u32*)next_orig.data(), 1, n, pshift);
    launch_independent_threads(pgrid, kParseThreads, k_parse_final, in, n, hdr, nchunk, pa, n, pshift);
    std::vector<u64>& out_off = P.out_off;  // k_scan_sizes: exclusive scan, total behind the end
    out_off.assign(nchunk + 1, 0);
    for (u32 k = 0; k < nchunk; k++) out_off[k + 1] = out_off[k] + pa.outb[k];
    launch_independent_threads(pgrid, kParseThreads, k_build_index, in, n, hdr, nchunk, pa, (const u64*)out_off.data(), idx.data(),
                               nfrag, n, (u64)0, pshift, ost.data(), 1u, (u64)claimed);
    u64 h4[4];
    k_parse_report(pa.counters, out_off.data() + nchunk, h4);
    P.pflags = h4[0];
    P.total = h4[2];
    P.first_err = h4[3];
}

// k_first_missing -> tvalid (snappy_b200.cu:1083-1095)
static u32 tiles_valid(const std::vector<u64>& idx, u32 nfrag, u64 n) {
    u32 first = nfrag + 1;
    launch_independent_threads((nfrag + 1 + 255) / 256, 256u, k_first_missing, (const u64*)idx.data(), nfrag, n, &first);
    u32 tvalid = first == 0 ? 0u : (first > nfrag ? nfrag : first - 1);
    if (first <= nfrag && first > 0 && tvalid > 0) tvalid = first - 1;
    return tvalid;
}

static int decode_parsed(const u8* in, u64 n, u64 hdr, u32 claimed, u8* out, u32 pshift, bool clean_cuts, int* path) {
    const u32 nfrag = (u32)(((u64)claimed + kBlockSize - 1) / kBlockSize);
    DecodeResult res{};
    if (nfrag == 0 || n <= hdr) {  // :1030 -> whole-stream serial decoder (:1154-1155)
        *path = 3;
        SerialArgs a{in, n, hdr, out, claimed, &res};
        as_warp(0, 0, 32);
        cpu_warp::run_warp(entry_serial, &a);
        return res.status;
    }
    Parse P;
    parse_stream(in, n, hdr, claimed, pshift, P);
    std::vector<u64>& idx = P.idx;
    std::vector<u64>& ost = P.ost;
    std::vector<u64>& out_off = P.out_off;
    ParseArrays& pa = P.pa;
    const u32 nchunk = P.nchunk, pgrid = (nchunk + kParseThreads - 1) / kParseThreads;
    const u64 pflags = P.pflags, total = P.total, first_err = P.first_err;
    std::vector<u8> tf(nfrag + 64, 0);
    // ---- the parse's verdicts (:1049-1058)
    *path = 1;
    if (first_err != ~0ull) return (int)(first_err & 7);
    if (!(pflags & (PF_ANOMALY | PF_BROKEN)) && total != claimed) return ST_INVALID_INPUT;
    ost[nfrag] = claimed;
    const bool complete = !(pflags & (PF_ANOMALY | PF_BROKEN)) && total == claimed;
    if (complete && (pflags & PF_NOT_CLEAN) && nfrag > 1 && clean_cuts) {  // :1061-1082
        std::vector<u64> low(nchunk, 0), sfx(nchunk, ~0ull);
        launch_independent_threads(pgrid, kParseThreads, k_cut_low, in, n, hdr, nchunk, pa, (const u64*)out_off.data(), n, pshift, low.data());
        u64 run = ~0ull;  // k_suffix_min
        for (u32 k = nchunk; k-- > 0;) {
            sfx[k] = run;
            run = low[k] < run ? low[k] : run;
        }
        launch_independent_threads((nfrag - 1 + kParseThreads - 1) / kParseThreads, kParseThreads, k_cut_tiles, in, n, hdr, nchunk, pa,
                                   (const u64*)out_off.data(), (const u64*)sfx.data(), n, pshift, nfrag, idx.data(), ost.data());
        k_cut_fill(nfrag, idx.data(), ost.data());
    }
    const u32 tvalid = complete ? nfrag : tiles_valid(idx, nfrag, n);  // :1083-1095
    // ---- the tiles (:1096-1111)
    if (tvalid) {
        FragArgs a{in, idx.data(), nfrag, tvalid, hdr, n, out, claimed, &res, ost.data(), tf.data()};
        for (u32 f = 0; f < tvalid; f++) {  // warp (f % warps-per-CTA) of CTA f / warps-per-CTA
            as_warp(f / kDecodeWarpsPerCta, (f % kDecodeWarpsPerCta) * 32, kDecodeWarpsPerCta * 32);
            cpu_warp::run_warp(entry_fragments, &a);
        }
    }
    if (!res.fallback && complete) return ST_OK;
    // ---- the bounded serial walk (:1112-1124)
    *path = 2;
    for (u32 f = tvalid; f < nfrag; f++) tf[f] = 1;
    if (!complete) tf[nfrag - 1] = 1;
    res = DecodeResult{};
    TileArgs t{in, n, idx.data(), ost.data(), nfrag, tf.data(), out, claimed, &res};
    as_warp(0, 0, 32);
    cpu_warp::run_warp(entry_serial_tiles, &t);
    return res.status;
}

// validate_device_locked: path 0 (side index), 1 (the parse decides), 2 (status-only tile walk), 3 (whole-stream
// walk).  No output pointer anywhere: a write would fault.  *step3: a complete, error-free parse said OK on its own.
static int validate(const u8* in, u64 n, u64 hdr, u32 claimed, const std::vector<u64>* index, u32 pshift, int* path,
                    bool* step3) {
    const u32 nfrag = (u32)(((u64)claimed + kBlockSize - 1) / kBlockSize);
    DecodeResult res{};
    *step3 = false;
    if (index && nfrag > 0) {  // validate_indexed_locked
        *path = 0;
        VFragArgs a{in, index->data(), nfrag, hdr, n, claimed, &res};
        for (u32 f = 0; f < nfrag; f++) {
            as_warp(f / kDecodeWarpsPerCta, (f % kDecodeWarpsPerCta) * 32, kDecodeWarpsPerCta * 32);
            cpu_warp::run_warp(entry_validate_fragments, &a);
        }
        if (!res.fallback) return ST_OK;
        res = DecodeResult{};
    }
    if (nfrag == 0 || n <= hdr) {  // validate_exact_locked
        *path = 3;
        SerialArgs a{in, n, hdr, nullptr, claimed, &res};
        as_warp(0, 0, 32);
        cpu_warp::run_warp(entry_validate_serial, &a);
        return res.status;
    }
    Parse P;  // validate_parsed_locked
    parse_stream(in, n, hdr, claimed, pshift, P);
    *path = 1;
    if (P.first_err != ~0ull) return (int)(P.first_err & 7);
    if (!(P.pflags & (PF_ANOMALY | PF_BROKEN))) {
        *step3 = P.total == claimed;
        return P.total == claimed ? ST_OK : ST_INVALID_INPUT;
    }
    *path = 2;
    P.ost[nfrag] = claimed;
    const u32 tvalid = tiles_valid(P.idx, nfrag, n);
    std::vector<u8> tf(nfrag + 64, 0);
    for (u32 f = tvalid; f < nfrag; f++) tf[f] = 1;
    tf[nfrag - 1] = 1;
    TileArgs t{in, n, P.idx.data(), P.ost.data(), nfrag, tf.data(), nullptr, claimed, &res};
    as_warp(0, 0, 32);
    cpu_warp::run_warp(entry_validate_tiles, &t);
    return res.status;
}

// the oracle's status of uncompress (sjo_uncompress_ex into a buffer of the claimed length)
static int oracle_status(const u8* s, size_t n) {
    u32 claimed = 0;
    size_t hdr = 0;
    const int hst = sjo_parse32(s, n, 0, &claimed, &hdr);
    if (hst != SJO_OK) return hst;
    std::vector<u8> want((size_t)claimed + 64);
    size_t wl = claimed, werr = 0;
    return sjo_uncompress_ex(s, n, want.data(), &wl, &werr);
}

static std::vector<u8> slurp(const char* path) {
    FILE* fp = fopen(path, "rb");
    if (!fp) {
        perror(path);
        exit(2);
    }
    fseek(fp, 0, SEEK_END);
    const size_t sz = (size_t)ftell(fp);
    fseek(fp, 0, SEEK_SET);
    std::vector<u8> b(sz);
    if (sz && fread(b.data(), 1, sz, fp) != sz) exit(2);
    fclose(fp);
    return b;
}

static bool sentinels_intact(const u8* p, size_t len) {
    for (size_t i = 0; i < len; i++)
        if (p[i] != kSentinel) return false;
    return true;
}

static int run_parsed(int argc, char** argv) {
    const u32 pshift = getenv("PSHIFT") ? (u32)atoi(getenv("PSHIFT")) : kParseChunkLog2;
    const bool clean_cuts = !getenv("CLEAN_CUTS") || atoi(getenv("CLEAN_CUTS")) != 0;
    int failed = 0;
    for (int ai = 2; ai < argc; ai++) {
        std::vector<u8> s = slurp(argv[ai]);
        const size_t sz = s.size();
        // the stream in a 256-aligned buffer, as a fresh device allocation holds it
        u8* in = (u8*)aligned_alloc(256, (sz + 64 + 255) & ~(size_t)255);
        memset(in, 0, sz + 64);
        if (sz) memcpy(in, s.data(), sz);
        u32 claimed = 0;
        size_t hdr = 0;
        const int hrc = sjo_parse32(in, sz, 0, &claimed, &hdr);
        std::vector<u8> want((size_t)claimed + 64);
        size_t wl = claimed, werr = 0;
        const int wrc = sjo_uncompress_ex(in, sz, want.data(), &wl, &werr);
        int got = hrc, path = -1;
        bool bytes_ok = true, guard_ok = true;
        if (hrc == SJO_OK) {
            u8* out = (u8*)aligned_alloc(256, ((size_t)claimed + kGuard + 255) & ~(size_t)255);
            memset(out, kSentinel, (size_t)claimed + kGuard);
            got = decode_parsed(in, sz, hdr, claimed, out, pshift, clean_cuts, &path);
            if (got == SJO_OK && wrc == SJO_OK) bytes_ok = memcmp(out, want.data(), claimed) == 0;
            guard_ok = sentinels_intact(out + claimed, kGuard);
            free(out);
        }
        const bool ok = got == wrc && bytes_ok && guard_ok;
        char ps[8];
        if (path < 0) snprintf(ps, sizeof ps, "-");
        else snprintf(ps, sizeof ps, "%d", path);
        printf("%s: status %d (oracle %d) path %s%s%s: %s\n", argv[ai], got, wrc, ps, bytes_ok ? "" : " [bytes differ]",
               guard_ok ? "" : " [wrote past claimed]", ok ? "0 mismatches" : "MISMATCH");
        failed += !ok;
        free(in);
    }
    return failed ? 1 : 0;
}

static int run_pages(int argc, char** argv) {
    // one flat input buffer, page offsets 16-byte aligned (the Python wrapper's layout)
    std::vector<u64> in_off, out_off;
    std::vector<u32> in_size, out_cap;
    std::vector<int> want_status;
    std::vector<std::vector<u8>> want_bytes;
    std::vector<std::string> names;
    std::vector<u8> flat;
    u64 out_total = 0;
    auto add = [&](const std::string& name, const std::vector<u8>& s) {
        const u32 k = (u32)in_size.size();
        in_off.push_back(flat.size());
        in_size.push_back((u32)s.size());
        flat.insert(flat.end(), s.begin(), s.end());
        flat.resize((flat.size() + 15) & ~(size_t)15, 0);
        u32 claimed = 0;
        size_t hdr = 0;
        int st = sjo_parse32(s.data(), s.size(), 0, &claimed, &hdr);
        u32 cap = claimed;
        std::vector<u8> want;
        if (st == SJO_OK) {
            if (k % 4 == 3 && claimed > 0) {
                cap = claimed - 1;
                st = SJO_BUFFER_TOO_SMALL;
            } else {
                want.resize((size_t)claimed + 64);
                size_t wl = claimed, werr = 0;
                st = sjo_uncompress_ex(s.data(), s.size(), want.data(), &wl, &werr);
            }
        }
        if (st == SJO_BAD_VARINT) cap = 0;  // no header, no claimed length: the whole slot must stay untouched
        out_off.push_back(out_total);
        out_cap.push_back(cap);
        out_total += ((u64)cap + kGuard + 15) & ~(u64)15;
        want_status.push_back(st);
        want_bytes.push_back(std::move(want));
        names.push_back(name);
    };
    add("(empty page)", {});
    for (int ai = 2; ai < argc; ai++) add(argv[ai], slurp(argv[ai]));
    add("(empty page)", {});
    flat.resize(flat.size() + 64, 0);
    const u32 count = (u32)in_size.size();
    std::vector<u8> out(out_total + 64, kSentinel);
    std::vector<u32> out_size(count, 0xdeadbeefu);
    std::vector<int> statuses(count, -1);
    PageArgs a{flat.data(), in_off.data(), in_size.data(), count, out.data(), out_off.data(), out_cap.data(), out_size.data(),
               statuses.data()};
    for (u32 i = 0; i < count; i++) {  // one launch: warp (i % warps-per-CTA) of CTA i / warps-per-CTA
        as_warp(i / kDecodeWarpsPerCta, (i % kDecodeWarpsPerCta) * 32, kDecodeWarpsPerCta * 32);
        cpu_warp::run_warp(entry_pages, &a);
    }
    int failed = 0;
    for (u32 i = 0; i < count; i++) {
        const u32 cap = out_cap[i];
        const bool st_ok = statuses[i] == want_status[i];
        const u32 want_size = want_status[i] == SJO_OK ? cap : 0u;
        const bool size_ok = out_size[i] == want_size;
        const bool bytes_ok = want_status[i] != SJO_OK || statuses[i] != SJO_OK ||
                              memcmp(out.data() + out_off[i], want_bytes[i].data(), cap) == 0;
        const u64 slot_end = i + 1 < count ? out_off[i + 1] : out_total;
        const bool guard_ok = sentinels_intact(out.data() + out_off[i] + cap, slot_end - out_off[i] - cap);
        const bool ok = st_ok && size_ok && bytes_ok && guard_ok;
        printf("%s: page %u status %d (oracle %d), out_size %u%s%s: %s\n", names[i].c_str(), i, statuses[i], want_status[i], out_size[i],
               bytes_ok ? "" : " [bytes differ]", guard_ok ? "" : " [wrote past out_cap]", ok ? "0 mismatches" : "MISMATCH");
        failed += !ok;
    }
    return failed ? 1 : 0;
}

static int run_validate(int argc, char** argv) {
    const u32 pshift = getenv("PSHIFT") ? (u32)atoi(getenv("PSHIFT")) : kParseChunkLog2;
    const char* suffix = getenv("IDX_SUFFIX");
    int failed = 0;
    for (int ai = 2; ai < argc; ai++) {
        std::vector<u8> s = slurp(argv[ai]);
        const size_t sz = s.size();
        u8* in = (u8*)aligned_alloc(256, (sz + 64 + 255) & ~(size_t)255);
        memset(in, 0, sz + 64);
        if (sz) memcpy(in, s.data(), sz);
        u32 claimed = 0;
        size_t hdr = 0;
        const int hrc = sjo_parse32(in, sz, 0, &claimed, &hdr);
        const int want = oracle_status(in, sz);
        std::vector<u64> index;
        bool have_index = false;
        if (suffix) {
            const std::string ip = std::string(argv[ai]) + suffix;
            if (FILE* fp = fopen(ip.c_str(), "rb")) {
                fclose(fp);
                std::vector<u8> raw = slurp(ip.c_str());
                index.resize(raw.size() / 8);
                memcpy(index.data(), raw.data(), index.size() * 8);
                have_index = true;
            }
        }
        int got = hrc, dec = hrc, path = -1, dpath = -1;
        bool step3 = false;
        if (hrc == SJO_OK) {
            const u32 nfrag = (u32)(((u64)claimed + kBlockSize - 1) / kBlockSize);
            if (have_index && index.size() != (size_t)nfrag + 1) {
                fprintf(stderr, "%s: index has %zu entries, want %u\n", argv[ai], index.size(), nfrag + 1);
                exit(2);
            }
            got = validate(in, sz, hdr, claimed, have_index ? &index : nullptr, pshift, &path, &step3);
            u8* out = (u8*)aligned_alloc(256, ((size_t)claimed + kGuard + 255) & ~(size_t)255);
            dec = decode_parsed(in, sz, hdr, claimed, out, pshift, true, &dpath);
            free(out);
        }
        const bool ok = got == want && dec == want;
        char ps[8];
        if (path < 0) snprintf(ps, sizeof ps, "-");
        else snprintf(ps, sizeof ps, "%d", path);
        printf("%s: status %d parsed %d (oracle %d) path %s%s: %s\n", argv[ai], got, dec, want, ps, step3 ? " step3" : "",
               ok ? "0 mismatches" : "MISMATCH");
        failed += !ok;
        free(in);
    }
    return failed ? 1 : 0;
}

static int run_validate_pages(int argc, char** argv) {
    std::vector<u64> in_off;
    std::vector<u32> in_size, want_claimed;
    std::vector<int> want_status;
    std::vector<std::string> names;
    std::vector<u8> flat;
    auto add = [&](const std::string& name, const std::vector<u8>& s) {
        in_off.push_back(flat.size());
        in_size.push_back((u32)s.size());
        flat.insert(flat.end(), s.begin(), s.end());
        flat.resize((flat.size() + 15) & ~(size_t)15, 0);
        u32 claimed = 0;
        size_t hdr = 0;
        const int hst = sjo_parse32(s.data(), s.size(), 0, &claimed, &hdr);
        want_claimed.push_back(hst == SJO_OK ? claimed : 0u);
        want_status.push_back(oracle_status(s.data(), s.size()));
        names.push_back(name);
    };
    add("(empty page)", {});
    for (int ai = 2; ai < argc; ai++) add(argv[ai], slurp(argv[ai]));
    add("(empty page)", {});
    flat.resize(flat.size() + 64, 0);
    const u32 count = (u32)in_size.size();
    std::vector<u32> claimed(count, 0xdeadbeefu);
    std::vector<int> statuses(count, -1);
    VPageArgs a{flat.data(), in_off.data(), in_size.data(), count, claimed.data(), statuses.data()};
    for (u32 i = 0; i < count; i++) {
        as_warp(i / kDecodeWarpsPerCta, (i % kDecodeWarpsPerCta) * 32, kDecodeWarpsPerCta * 32);
        cpu_warp::run_warp(entry_validate_pages, &a);
    }
    int failed = 0;
    for (u32 i = 0; i < count; i++) {
        const bool ok = statuses[i] == want_status[i] && claimed[i] == want_claimed[i];
        printf("%s: page %u status %d (oracle %d), claimed %u (header %u): %s\n", names[i].c_str(), i, statuses[i],
               want_status[i], claimed[i], want_claimed[i], ok ? "0 mismatches" : "MISMATCH");
        failed += !ok;
    }
    return failed ? 1 : 0;
}

int main(int argc, char** argv) {
    if (argc < 2) return 2;
    if (!strcmp(argv[1], "parsed")) return run_parsed(argc, argv);
    if (!strcmp(argv[1], "pages")) return run_pages(argc, argv);
    if (!strcmp(argv[1], "validate")) return run_validate(argc, argv);
    if (!strcmp(argv[1], "validate-pages")) return run_validate_pages(argc, argv);
    fprintf(stderr, "mode: parsed | pages | validate | validate-pages\n");
    return 2;
}
