// snappy_b200.cu -- C ABI (include/snappy_b200.h) + device buffer manager for libsnappy_b200.so.
//
// Host side of the drop-in boundary: what src/Snappy.jl:20-52 does around the codec kernels
// (length check, varint header, buffer sizing, final length, error mapping) lives here in C++;
// the codec itself runs only as sm_100a kernels (compress.cuh / decompress.cuh).  No CPU fallback.
#include "../../include/snappy_b200.h"

#include <cuda_profiler_api.h>
#include <cuda_runtime.h>

#include <atomic>
#include <chrono>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <condition_variable>
#include <mutex>
#include <thread>
#include <string>
#include <vector>

#include "compress.cuh"
#include "compress_chain.cuh"
#include "compress_pipe.cuh"
#ifdef SB200_EXPERIMENTS
#include "compress_wide.cuh"
#endif
#include "decompress.cuh"
#include "parse.cuh"
#include "schedule.cuh"

using namespace sb200;

namespace {

struct Bounce;  // pinned slots for pageable host buffers (defined with the host-buffer paths below)

thread_local std::string g_last_error;

struct DevBuf {
    void* p = nullptr;
    size_t cap = 0;
    // grow-only device allocation
    cudaError_t ensure(size_t bytes) {
        if (bytes <= cap) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
        size_t want = bytes + bytes / 8 + 4096;
        cudaError_t e = cudaMalloc(&p, want);
        if (e == cudaSuccess) cap = want;
        return e;
    }
    void release() {
        if (p) cudaFree(p);
        p = nullptr;
        cap = 0;
    }
};

constexpr int kMaxPipeChunks = 72;                 // 4 GiB / 64 MiB, plus slack
constexpr size_t kPinnedBytes = 64 * 1024;         // small pinned readback area of a lane
constexpr u32 kPageWindowMax = 8192;               // batched pages up to this size take the window-round page kernel
constexpr size_t kPinnedShardLens = 8192;          // offset of the per-shard lengths of the batched shard API (<= 4096 x u64)
constexpr size_t kPipeChunkFragsDefault = 4096;    // fragments per pipeline chunk (256 MiB)

struct Options {
    int compress_variant = 0;   // 0 = lane-speculative chain kernel, 1 = serial smem kernel, 2 = ring kernel
    int smem_chains = 6;        // persistent warps per SM with the table in shared memory
    int l2_reserve = 1;         // global-table warps stop pulling when fewer than l2_reserve x (smem warps) fragments remain
    int wide = 0;               // 2 or 4: warps per fragment of the wide window kernel (compress_wide.cuh); 0 = off
    int l2_persist = 0;         // 1 = pin the global hash tables in L2 (access policy window on the side stream)
    int rules = 0;              // emission rules: 0 = Snappy.jl (the reference, default), 1 = libsnappy <= 1.1.7,
                                // 2 = Google snappy >= 1.1.9 (byte-identical to pyarrow's bundled codec)
    int slowcont = 0;           // 1 = window kernel variant that extends long copies inside the hop loop (measured: 13.58 vs 13.12 ms, off)
    int window = 1;             // 1 = window-parallel kernel (compress_window.cuh), 0 = step-wise chain kernel
    int ring_smem = 2048;       // history ring per shared-table warp (bytes, power of two >= 1024)
    int ring_l2 = 1024;         // history ring per global-table warp
    int spec_smem = 32;         // copy end positions pre-probed per step by shared-table warps (1..32)
    int spec_l2 = 16;           // same for global-table warps (each probing lane costs an L1tex wavefront)
    int l2_chains = 14;         // warps per CTA of the global-table (L2) kernel, <= 20 (window kernel; <= 14 for the chain kernel)
    int l2_chains_big = 14;     // the same under rules = 2 (64 KiB tables; measured 4: 25.1, 8: 20.3, 10: 19.1, 14: 17.5 ms/GiB)
    int l2_ctas = 1;            // CTAs per SM of that kernel (1..3): l2_ctas x l2_chains extra chains per SM
    int decode_variant = 0;     // 0 = default, 1 = force exact serial decoder
    int decode_occupancy = 12;  // CTAs (of 4 warps) per SM the indexed decoder is compiled for: 8, 10 or 12
    int pipe_chunk_frags = (int)kPipeChunkFragsDefault;  // host-buffer API pipeline granularity
    int parse_chunk_log2 = (int)kParseChunkLog2;  // index-free parse: log2 of the compressed bytes per thread
    int overlap_compact = 0;    // device-resident compress: compaction per chunk while the rest still compresses (measured: 60.5 vs 61.3 GB/s, the compaction CTAs slow the persistent kernels more than they save: off)
    int uncompress_segments = 8;  // streamed host-buffer uncompress: segments the stream is parsed in (2, 4 or 8)
    int host_pipeline = 1;      // host-buffer API: overlap H2D / kernels / D2H in chunks
    int timing = 1;             // record CUDA events around the dominant kernel
    int trace = 0;              // 1 = the compress warps record begin / end time of every fragment (snappy_b200_debug_trace)
    int profile_range = 0;      // 1 = cudaProfilerStart/Stop around the concurrent compress kernels (ncu --replay-mode range)
    int mixed = 1;              // 1 = both table placements in ONE kernel, shared-table warps on the high warp numbers;
                                // 2 = the same with them on the low ones; 0 = two concurrent kernels (round 1)
    int two = 0;                // two-window round: 1 = global-table warps, 2 = shared-table warps, 3 = both (mixed kernel)
    int pipe = 0;               // pipelined round (compress_pipe.cuh): 1 = shared-table warps, 2 = global-table warps, 3 = both
    int unified = 0;            // merged kernel: one copy of the round's code for both table placements (run-time flag per warp)
    int l2_first = 0;           // mixed = 0 only: launch the global-table kernel before the shared-table kernel
    int pages_window = 1;       // batched pages <= 8 KiB: window-round kernel (0 = the serial page kernel for every size)
    int lpt = 1;                // compress: order the fragments by estimated cost, expensive first (k_estimate_cost)
    int clean_cuts = 1;         // index-free decode: re-tile at clean cuts when copies cross the 64 KiB boundaries (0: bounded serial walk only)
    int pin_host = 1;           // host-buffer API on pageable memory: register the caller's buffers for the call
};

Options g_opt;             // process-wide (snappy_b200_set_option / SNAPPY_B200_OPTIONS)
std::mutex g_opt_mu;

struct Context {
    std::mutex mu;
    bool ready = false;
    int device = -1;
    int lane = 0;
    int sm_count = 0;
    size_t l2_persist_max = 0, l2_window_max = 0;
    // scratch for compress
    DevBuf scratch, frag_sizes, frag_offsets, tail, gtables, descs, flags, order, trace;
    u32 trace_frags = 0;
    cudaStream_t side = nullptr;      // second stream for the global-table warps
    cudaStream_t s_h2d = nullptr, s_d2h = nullptr, s_comp = nullptr, s_pack = nullptr;  // host-buffer API pipeline
    cudaEvent_t ev_in[kMaxPipeChunks] = {}, ev_done[kMaxPipeChunks] = {};
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr;
    // scratch for decode
    DevBuf result, parse_a, parse_b, parse_c, parse_d, index, index_out, tile_flags;
    // staging for the host-buffer API
    DevBuf stage_in, stage_out;
    void* pinned = nullptr;  // small pinned readback area (kPinnedBytes)
    void* pinned_zero = nullptr;  // kTailPad zero bytes (pinned): pads go up through the copy engine
    Bounce* bounce = nullptr;         // pinned slots for pageable host buffers
    struct DownRange {
        size_t off, len;
        int ev;
    };
    std::vector<DownRange>* defer_down = nullptr;  // decode_launch: list the finished ranges instead of copying them
    cudaEvent_t ev[4] = {nullptr, nullptr, nullptr, nullptr};
    float last_ms[2] = {0.f, 0.f};
    int last_launches[2] = {0, 0};
    bool ev_pending[2] = {false, false};
    int last_path = 0;  // how the last uncompress decoded: 0 side index, 1 parse + tiles, 2 ... + bounded serial walk, 3 whole-stream serial
    Options& opt = g_opt;
};

// One Context (scratch buffers, streams, events) per device and LANE.  A call takes a free lane of the device it
// addresses, so that concurrent host threads (Threads.@threads over independent buffers, SURVEY.md 8(b)) run
// side by side instead of queueing on one mutex; a lane is created the first time every existing one is busy.
// Device selection: snappy_b200_init(d >= 0) binds the CALLING THREAD to device d; an unbound thread uses
// $SNAPPY_B200_DEVICE if set, else its current CUDA device (cudaGetDevice), which is what torch's
// `with torch.cuda.device(...)` sets.  Device pointers passed to a call must belong to that device.
constexpr int kMaxDevices = 16;
constexpr int kMaxLanes = 4;
struct DeviceSlot {
    std::mutex mu;               // guards lanes[] / nlanes / once
    std::mutex big;              // one streamed host pipeline (persistent kernels gated on copies) at a time
    Context* lanes[kMaxLanes] = {};
    int nlanes = 0;
    bool once = false;           // per-device one-time setup done (L2 set-aside, probe-offset table)
};
DeviceSlot g_dev[kMaxDevices];
thread_local int tl_device = -1;          // snappy_b200_init(d): this thread's device
thread_local Context* tl_last = nullptr;  // the context of this thread's last call (last_kernel_ms / launch_count)

int fail_cuda(cudaError_t e, const char* what) {
    char buf[256];
    snprintf(buf, sizeof buf, "%s: %s", what, cudaGetErrorString(e));
    g_last_error = buf;
    return SNAPPY_B200_CUDA_ERROR;
}

#define CU(call)                                              \
    do {                                                      \
        cudaError_t e__ = (call);                             \
        if (e__ != cudaSuccess) return fail_cuda(e__, #call); \
    } while (0)

// tuning knobs (snappy_b200_set_option / SNAPPY_B200_OPTIONS); caller holds g_opt_mu
void apply_option(const char* name, int value) {
    if (!name) return;
    if (!strcmp(name, "decode_variant")) g_opt.decode_variant = value;
#ifdef SB200_EXPERIMENTS  // kernel designs that were measured and lost (DESIGN.md section 4): not in the product build
    else if (!strcmp(name, "compress_variant")) g_opt.compress_variant = value;
    else if (!strcmp(name, "slowcont")) g_opt.slowcont = value != 0;
    else if (!strcmp(name, "window")) g_opt.window = value;
    else if (!strcmp(name, "wide")) g_opt.wide = value;
    else if (!strcmp(name, "two")) g_opt.two = value;
    else if (!strcmp(name, "pipe")) g_opt.pipe = value < 0 ? 0 : (value > 3 ? 3 : value);
    else if (!strcmp(name, "unified")) g_opt.unified = value != 0;
    else if (!strcmp(name, "l2_fetch")) {  // L2 fetch granularity in bytes (32, 64 or 128; the driver's default is 64): no effect measured
        if (value == 32 || value == 64 || value == 128) cudaDeviceSetLimit(cudaLimitMaxL2FetchGranularity, (size_t)value);
    }
#endif
    else if (!strcmp(name, "smem_chains")) g_opt.smem_chains = value < 0 ? 0 : (value > 7 ? 7 : value);
    else if (!strcmp(name, "l2_chains")) g_opt.l2_chains = value < 0 ? 0 : (value > 20 ? 20 : value);
    else if (!strcmp(name, "l2_chains_big")) g_opt.l2_chains_big = value < 0 ? 0 : (value > 20 ? 20 : value);
    else if (!strcmp(name, "spec_smem")) g_opt.spec_smem = value < 1 ? 1 : (value > 14 ? 14 : value);
    else if (!strcmp(name, "spec_l2")) g_opt.spec_l2 = value < 1 ? 1 : (value > 14 ? 14 : value);
    else if (!strcmp(name, "ring_smem") || !strcmp(name, "ring_l2")) {
        int r = 1024;
        while (r < value && r < 32768) r <<= 1;
        (name[5] == 's' ? g_opt.ring_smem : g_opt.ring_l2) = r;
    }
    else if (!strcmp(name, "parse_chunk_log2")) g_opt.parse_chunk_log2 = value < 9 ? 9 : (value > 16 ? 16 : value);
    else if (!strcmp(name, "l2_persist")) g_opt.l2_persist = value;
    else if (!strcmp(name, "overlap_compact")) g_opt.overlap_compact = value;
    else if (!strcmp(name, "uncompress_segments")) g_opt.uncompress_segments = value;
#ifdef SB200_EXPERIMENTS
    else if (!strcmp(name, "dbg_skip_emit")) {  // applies to the calling thread's current device
        const u32 v = (u32)value;
        cudaMemcpyToSymbol(g_dbg_skip_emit, &v, 4);
    }
#endif
    else if (!strcmp(name, "rules")) g_opt.rules = value < 0 ? 0 : (value > 2 ? 2 : value);
    else if (!strcmp(name, "l2_ctas")) g_opt.l2_ctas = value < 1 ? 1 : (value > 3 ? 3 : value);
    else if (!strcmp(name, "l2_reserve")) g_opt.l2_reserve = value;
    else if (!strcmp(name, "host_pipeline")) g_opt.host_pipeline = value;
    else if (!strcmp(name, "pipe_chunk_frags")) {
        // at most kMaxPipeChunks chunks for the largest stream (2^32 bytes = 65536 fragments)
        g_opt.pipe_chunk_frags = value < 1024 ? 1024 : value;
    }
    else if (!strcmp(name, "decode_occupancy")) g_opt.decode_occupancy = value;
    else if (!strcmp(name, "timing")) g_opt.timing = value;
    else if (!strcmp(name, "lpt")) g_opt.lpt = value;
    else if (!strcmp(name, "pages_window")) g_opt.pages_window = value;
    else if (!strcmp(name, "mixed")) g_opt.mixed = value;
    else if (!strcmp(name, "l2_first")) g_opt.l2_first = value;

    else if (!strcmp(name, "profile_range")) g_opt.profile_range = value;
    else if (!strcmp(name, "trace")) g_opt.trace = value;
    else if (!strcmp(name, "pin_host")) g_opt.pin_host = value;
    else if (!strcmp(name, "clean_cuts")) g_opt.clean_cuts = value != 0;
}

// Shared-memory opt-ins of the kernels (per device; the attributes live in the device's module).
int set_kernel_attributes() {
    CU(cudaFuncSetAttribute(k_compress_pages<false>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)kCompressSmemBytes));
    CU(cudaFuncSetAttribute(k_compress_pages<true>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)(kCompressSmemBytes + kMaxTableEntries * 2)));
    CU(cudaFuncSetAttribute(k_compress_window_mixed<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    CU(cudaFuncSetAttribute(k_compress_window_mixed<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
#ifdef SB200_EXPERIMENTS
    CU(cudaFuncSetAttribute(k_compress_window_mixed<false, false, false, 0, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    CU(cudaFuncSetAttribute(k_compress_window_mixed<false, false, false, 3, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    CU(cudaFuncSetAttribute(k_compress_window_mixed<false, false, false, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    CU(cudaFuncSetAttribute(k_compress_window_mixed<false, false, false, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    CU(cudaFuncSetAttribute(k_compress_window_mixed<false, false, false, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    CU(cudaFuncSetAttribute(k_compress_window_mixed<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    CU(cudaFuncSetAttribute(k_compress_window_mixed<false, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    CU(cudaFuncSetAttribute(k_compress_window_mixed<false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
#endif
    CU(cudaFuncSetAttribute(k_compress_pages_window<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    CU(cudaFuncSetAttribute(k_compress_pages_window<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    // both window kernels share the SMs: ask for the full shared-memory carve-out so that the global-table
    // CTAs fit next to the shared-table CTA
    CU(cudaFuncSetAttribute(k_compress_window<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    CU(cudaFuncSetAttribute(k_compress_window<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    CU(cudaFuncSetAttribute(k_compress_window<true>, cudaFuncAttributePreferredSharedMemoryCarveout,
                            cudaSharedmemCarveoutMaxShared));
    CU(cudaFuncSetAttribute(k_compress_window<false>, cudaFuncAttributePreferredSharedMemoryCarveout,
                            cudaSharedmemCarveoutMaxShared));
#ifdef SB200_EXPERIMENTS
    CU(cudaFuncSetAttribute(k_compress_window<true, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    CU(cudaFuncSetAttribute(k_compress_window<false, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    CU(cudaFuncSetAttribute(k_compress_window<true, false, false, true>, cudaFuncAttributePreferredSharedMemoryCarveout,
                            cudaSharedmemCarveoutMaxShared));
    CU(cudaFuncSetAttribute(k_compress_window<false, false, false, true>, cudaFuncAttributePreferredSharedMemoryCarveout,
                            cudaSharedmemCarveoutMaxShared));
#endif
    CU(cudaFuncSetAttribute(k_compress_window<true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    CU(cudaFuncSetAttribute(k_compress_window<false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    CU(cudaFuncSetAttribute(k_compress_window<true, true>, cudaFuncAttributePreferredSharedMemoryCarveout,
                            cudaSharedmemCarveoutMaxShared));
    CU(cudaFuncSetAttribute(k_compress_window<false, true>, cudaFuncAttributePreferredSharedMemoryCarveout,
                            cudaSharedmemCarveoutMaxShared));
#ifdef SB200_EXPERIMENTS
    CU(cudaFuncSetAttribute(k_compress_fragments_serial, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)kCompressSmemBytes));
    CU(cudaFuncSetAttribute(k_compress_fragments, cudaFuncAttributeMaxDynamicSharedMemorySize,
                            (int)kCompress2SmemBytes));
    CU(cudaFuncSetAttribute(k_compress_chain<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    CU(cudaFuncSetAttribute(k_compress_wide<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    CU(cudaFuncSetAttribute(k_compress_wide<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    CU(cudaFuncSetAttribute(k_compress_window<true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    CU(cudaFuncSetAttribute(k_compress_window<false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    CU(cudaFuncSetAttribute(k_compress_window<true, false, true>, cudaFuncAttributePreferredSharedMemoryCarveout,
                            cudaSharedmemCarveoutMaxShared));
    CU(cudaFuncSetAttribute(k_compress_window<false, false, true>, cudaFuncAttributePreferredSharedMemoryCarveout,
                            cudaSharedmemCarveoutMaxShared));
    CU(cudaFuncSetAttribute(k_compress_chain<true>, cudaFuncAttributePreferredSharedMemoryCarveout,
                            cudaSharedmemCarveoutMaxShared));
    CU(cudaFuncSetAttribute(k_compress_chain<false>, cudaFuncAttributePreferredSharedMemoryCarveout,
                            cudaSharedmemCarveoutMaxShared));
#endif
    return SNAPPY_B200_OK;
}

// Resolve the device a call on this thread addresses (see DeviceSlot above).
int resolve_device(int* device) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
        g_last_error = std::string("no CUDA device: ") + cudaGetErrorString(e);
        return SNAPPY_B200_NO_DEVICE;
    }
    int d = tl_device;
    if (d < 0) {
        const char* env = getenv("SNAPPY_B200_DEVICE");
        if (env) d = atoi(env);
        else if (cudaGetDevice(&d) != cudaSuccess) d = 0;
    }
    if (d < 0 || d >= count || d >= kMaxDevices) {
        char buf[96];
        snprintf(buf, sizeof buf, "device %d does not exist (%d CUDA devices)", d, count);
        g_last_error = buf;
        return SNAPPY_B200_BAD_ARGUMENT;
    }
    *device = d;
    return SNAPPY_B200_OK;
}

void parse_env_options() {
    // tuning knobs from the environment: SNAPPY_B200_OPTIONS="name=value,name=value" (see set_option)
    static bool done = false;
    std::unique_lock<std::mutex> lk(g_opt_mu);
    if (done) return;
    done = true;
    if (const char* env = getenv("SNAPPY_B200_OPTIONS")) {
        std::string e(env);
        size_t pos = 0;
        while (pos < e.size()) {
            size_t comma = e.find(',', pos);
            if (comma == std::string::npos) comma = e.size();
            const std::string kv = e.substr(pos, comma - pos);
            const size_t eq = kv.find('=');
            if (eq != std::string::npos) apply_option(kv.substr(0, eq).c_str(), atoi(kv.c_str() + eq + 1));
            pos = comma + 1;
        }
    }
}

void ctx_destroy(Context& c);
void bounce_destroy(Context& c);

// Create the streams, events and pinned areas of a lane (current device == `device`); slot.mu is held.
int ctx_init(Context& c, int device, DeviceSlot& slot) {
    if (c.ready) return SNAPPY_B200_OK;
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10) {
        char buf[128];
        snprintf(buf, sizeof buf, "device %d is sm_%d%d; libsnappy_b200 holds sm_100a code only", device,
                 prop.major, prop.minor);
        g_last_error = buf;
        return SNAPPY_B200_NO_DEVICE;
    }
    c.device = device;
    c.sm_count = prop.multiProcessorCount;
    c.l2_persist_max = (size_t)prop.persistingL2CacheMaxSize;
    c.l2_window_max = (size_t)prop.accessPolicyMaxWindowSize;
    if (!slot.once) {
        // L2 set-aside for persisting / evict_last lines, at its maximum (79 MiB on B200): the global hash tables
        // of the global-table compress warps are read and written with L2::evict_last hints and live there
        // (13.2 ms with the set-aside, 14.1 ms without; SNAPPY_B200_NO_PERSIST_LIMIT=1 leaves the device default)
        if (c.l2_persist_max && !getenv("SNAPPY_B200_NO_PERSIST_LIMIT"))
            cudaDeviceSetLimit(cudaLimitPersistingL2CacheSize, c.l2_persist_max);
        if (getenv("SNAPPY_B200_DEBUG"))
            fprintf(stderr, "[snappy_b200] device %d: L2 %d MiB, persisting max %zu MiB, window max %zu MiB\n", device,
                    prop.l2CacheSize >> 20, c.l2_persist_max >> 20, c.l2_window_max >> 20);
        int rc = set_kernel_attributes();
        if (rc != SNAPPY_B200_OK) return rc;
        k_init_probe_offsets<<<1, 32>>>();
        CU(cudaGetLastError());
        CU(cudaDeviceSynchronize());
        slot.once = true;
    }
    // a failure below leaves a half-built lane: release what exists, so that a retry starts clean
    struct Guard {
        Context& c;
        bool armed = true;
        ~Guard() { if (armed) ctx_destroy(c); }
    } guard{c};
    CU(cudaStreamCreateWithFlags(&c.side, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&c.s_h2d, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&c.s_d2h, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&c.s_comp, cudaStreamNonBlocking));
    CU(cudaStreamCreateWithFlags(&c.s_pack, cudaStreamNonBlocking));
    for (int i = 0; i < kMaxPipeChunks; i++) {
        CU(cudaEventCreateWithFlags(&c.ev_in[i], cudaEventDisableTiming));
        CU(cudaEventCreateWithFlags(&c.ev_done[i], cudaEventDisableTiming));
    }
    CU(cudaEventCreateWithFlags(&c.ev_fork, cudaEventDisableTiming));
    CU(cudaEventCreateWithFlags(&c.ev_join, cudaEventDisableTiming));
    CU(cudaMallocHost(&c.pinned, kPinnedBytes));
    CU(cudaMallocHost(&c.pinned_zero, kTailPad));
    memset(c.pinned_zero, 0, kTailPad);
    for (auto& ev : c.ev) CU(cudaEventCreate(&ev));
    CU(c.result.ensure(256));
    guard.armed = false;
    c.ready = true;
    return SNAPPY_B200_OK;
}

// Release everything a lane owns (current device == c.device).
void ctx_destroy(Context& c) {
    for (cudaStream_t* sp : {&c.side, &c.s_h2d, &c.s_d2h, &c.s_comp, &c.s_pack}) {
        if (*sp) cudaStreamDestroy(*sp);
        *sp = nullptr;
    }
    for (int i = 0; i < kMaxPipeChunks; i++) {
        if (c.ev_in[i]) cudaEventDestroy(c.ev_in[i]);
        if (c.ev_done[i]) cudaEventDestroy(c.ev_done[i]);
        c.ev_in[i] = c.ev_done[i] = nullptr;
    }
    if (c.ev_fork) cudaEventDestroy(c.ev_fork);
    if (c.ev_join) cudaEventDestroy(c.ev_join);
    c.ev_fork = c.ev_join = nullptr;
    for (DevBuf* b : {&c.descs, &c.tail, &c.gtables, &c.scratch, &c.frag_sizes, &c.frag_offsets, &c.result, &c.parse_a,
                      &c.parse_b, &c.parse_c, &c.parse_d, &c.index, &c.stage_in, &c.stage_out, &c.flags, &c.order, &c.trace, &c.index_out, &c.tile_flags})
        b->release();
    if (c.pinned) cudaFreeHost(c.pinned);
    if (c.pinned_zero) cudaFreeHost(c.pinned_zero);
    c.pinned = c.pinned_zero = nullptr;
    bounce_destroy(c);
    for (auto& ev : c.ev) {
        if (ev) cudaEventDestroy(ev);
        ev = nullptr;
    }
    c.ready = false;
}

// collect the event pair recorded around the dominant kernel of the last call
void harvest_timing(Context& c, int which) {
    if (c.ev_pending[which]) {
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, c.ev[2 * which], c.ev[2 * which + 1]) == cudaSuccess)
            c.last_ms[which] = ms;
        c.ev_pending[which] = false;
    }
}

// fragments of an n-byte stream; in 64 bits: (u32)n + 65535 wraps for streams within 64 KiB of 4 GiB
inline u32 frag_count(u64 n) { return (u32)((n + kBlockSize - 1) / kBlockSize); }

inline u32 table_shift(u64 total_len) {
    u32 entries = 256;  // alloc_hashtable, src/internal.jl:107-113
    while (entries < kMaxTableEntries && entries < total_len) entries <<= 1;
    u32 lg = 0;
    while ((1u << lg) < entries) lg++;
    return 32 - lg;  // src/internal.jl:128
}

int encode_varint(u32 v, u8* out) {  // src/varint.jl:46-69
    int k = 0;
    while (v >= 0x80) {
        out[k++] = (u8)(v | 0x80);
        v >>= 7;
    }
    out[k++] = (u8)v;
    return k;
}

int parse_varint(const u8* in, size_t n, u32* value, size_t* hdr) {  // src/varint.jl:12-37
    u32 result = 0;
    for (int i = 0; i < 5; i++) {
        if ((size_t)i >= n) return SNAPPY_B200_BAD_VARINT;
        u32 b = in[i];
        result |= (b & 0x7f) << (7 * i);
        if (i < 4 ? (b < 0x80) : (b < 0x10)) {
            *value = result;
            *hdr = (size_t)i + 1;
            return SNAPPY_B200_OK;
        }
    }
    return SNAPPY_B200_BAD_VARINT;
}

// Launch the chain compressor (compress_chain.cuh) over the fragments of d_in[0 .. len): the
// shared-memory-table warps on `st`, the global-table warps on the side stream (joined back).
constexpr size_t kTailSlot = kBlockSize + kTailPad + 256;

// padded copy of a shard's last fragment into tail slot `slot` (the chain kernel reads a few bytes
// past a fragment's end)
int stage_tail(Context& c, const u8* d_in, size_t len, size_t slot, cudaStream_t st) {
    const u32 nfrag = (u32)((len + kBlockSize - 1) / kBlockSize);
    const u64 tail_start = (u64)(nfrag - 1) * kBlockSize;
    const size_t tail_len = len - tail_start;
    u8* t = (u8*)c.tail.p + slot * kTailSlot;
    CU(cudaMemcpyAsync(t, d_in + tail_start, tail_len, cudaMemcpyDeviceToDevice, st));
    CU(cudaMemsetAsync(t + tail_len, 0, kTailPad, st));
    return SNAPPY_B200_OK;
}

// descs == nullptr: the fragments of d_in[0 .. len); else `nfrag_total` fragments described by the
// device array descs[ndesc] (tails already staged).
// streamed host-buffer path: the kernels wait for `ready` (fragments resident) and count finished
// fragments per chunk of `div` fragments in `done`; the caller stages the tail itself
struct Gate {
    const u32* ready = nullptr;
    u32* done = nullptr;
    u32 div = 1;
};

int launch_chain_kernels(Context& c, const u8* d_in, size_t len, u32 shift, u8* scratch, u32* sizes,
                         cudaStream_t st, int* launches, const ShardDesc* descs = nullptr, u32 ndesc = 0,
                         u32 nfrag_total = 0, const Gate* gate = nullptr) {
    const u32 nfrag = descs ? nfrag_total : (u32)((len + kBlockSize - 1) / kBlockSize);
    if (!descs && !gate) {
        CU(c.tail.ensure(kTailSlot));
        int rc = stage_tail(c, d_in, len, 0, st);
        if (rc != SNAPPY_B200_OK) return rc;
    }
    u32* counter = (u32*)((u8*)c.result.p + 64);
    // profile_range: the two concurrent kernels (and the counter reset they depend on) form one ncu range
    const bool prof = c.opt.profile_range != 0;
    if (prof) {
        CU(cudaStreamSynchronize(st));
        cudaProfilerStart();
    }
    CU(cudaMemsetAsync(counter, 0, 4, st));
    // fragment order: expensive first (schedule.cuh).  Not for the streamed host path (fragments become resident
    // in stream order) and pointless below a few fragments per warp.
    u64* trace = nullptr;
    if (c.opt.trace) {
        CU(c.trace.ensure((size_t)nfrag * 16));
        CU(cudaMemsetAsync(c.trace.p, 0, (size_t)nfrag * 16, st));
        trace = (u64*)c.trace.p;
        c.trace_frags = nfrag;
    }
    const u32* order = nullptr;
    if (c.opt.lpt && !gate && nfrag >= 2u * (u32)c.sm_count) {
        CU(c.order.ensure((size_t)nfrag * 5));
        u32* ord = (u32*)c.order.p;
        u8* cost = (u8*)(ord + nfrag);
        k_estimate_cost<<<(nfrag + kCostWarps - 1) / kCostWarps, kCostWarps * 32, 0, st>>>(d_in, (u64)len, nfrag, descs,
                                                                                         ndesc, cost);
        k_order_by_cost<<<1, 1024, 0, st>>>(cost, nfrag, ord);
        *launches += 2;
        order = ord;
    }
    // one CTA per SM, smem_chains warps each (fewer CTAs when there are fewer fragments)
    // rules != 0 (libsnappy's emission rules): always the window kernel, compiled with kLib; rules = 2 has
    // 64 KiB tables, so 3 shared-table warps per SM (and l2_chains_big global-table warps)
    const u32 rules = (u32)c.opt.rules;
    const u32 tab_bytes = (rules == 2 ? 2u : 1u) * kMaxTableEntries * 2u;
    u32 wa = (u32)c.opt.smem_chains;
    // (the step-wise chain kernel is compiled for <= 14 warps per CTA)
    u32 wb = (!c.opt.window && !rules && c.opt.l2_chains > 14) ? 14u : (u32)c.opt.l2_chains;
    if (rules == 2) {
        if (wa > 3) wa = 3;
        wb = (u32)c.opt.l2_chains_big;
    }
    u32 ctas_a = wa ? (nfrag + wa - 1) / wa : 0u;  // smem_chains == 0: global-table warps only (profiling)
    if (ctas_a > (u32)c.sm_count) ctas_a = (u32)c.sm_count;
    const u32 warps_a = ctas_a * wa;
    const u32 reserve = (u32)c.opt.l2_reserve * warps_a;
    const u32 ctas_b = (wb && (nfrag > warps_a + reserve || !wa)) ? (u32)(c.sm_count * c.opt.l2_ctas) : 0u;
    if (ctas_b) CU(c.gtables.ensure((size_t)ctas_b * wb * tab_bytes));
    if (ctas_b) CU(cudaEventRecord(c.ev_fork, st));
#ifdef SB200_EXPERIMENTS
    if (!rules && (c.opt.wide == 2 || c.opt.wide == 4)) {  // kW warps per fragment, shared tables only
        const u32 chains = (u32)c.opt.smem_chains, ra = (u32)c.opt.ring_smem;
        u32 ctas = (nfrag + chains - 1) / chains;
        if (ctas > (u32)c.sm_count) ctas = (u32)c.sm_count;
        if (c.opt.wide == 4)
            k_compress_wide<4><<<ctas, chains * 128, (size_t)chains * (kMaxTableEntries * 2 + ra + kRingMirror + sizeof(WideCtl<4>)), st>>>(
                d_in, (u64)len, nfrag, shift, (const u8*)c.tail.p, scratch, sizes, counter, descs, ndesc, ra);
        else
            k_compress_wide<2><<<ctas, chains * 64, (size_t)chains * (kMaxTableEntries * 2 + ra + kRingMirror + sizeof(WideCtl<2>)), st>>>(
                d_in, (u64)len, nfrag, shift, (const u8*)c.tail.p, scratch, sizes, counter, descs, ndesc, ra);
        *launches += 1;
        return SNAPPY_B200_OK;
    }
#endif
    const bool window = c.opt.window != 0 || rules != 0;
    (void)window;
    const u32 ra = (u32)c.opt.ring_smem, rb = (u32)c.opt.ring_l2;
    WindowArgs A;
    memset(&A, 0, sizeof A);
    A.g_in = d_in;
    A.shard_len = (u64)len;
    A.nfrag = nfrag;
    A.shift = shift;
    A.tail_copy = (const u8*)c.tail.p;
    A.scratch = scratch;
    A.frag_sizes = sizes;
    A.counter = counter;
    A.gtables = (u16*)c.gtables.p;
    A.reserve = reserve;
    A.descs = descs;
    A.ndesc = ndesc;
    A.ready = gate ? gate->ready : nullptr;
    A.done = gate ? gate->done : nullptr;
    A.done_div = gate ? gate->div : 1u;
    A.lib_rules = rules;
    A.order = order;
    A.trace = trace;
    const size_t smem_a = (size_t)wa * (tab_bytes + ra + kRingMirror), smem_b = (size_t)wb * (rb + kRingMirror);
    bool plain = true;
#ifdef SB200_EXPERIMENTS
    plain = !(window && c.opt.slowcont) && window;
#endif
    if (plain && ctas_a && ctas_b && c.opt.mixed && c.opt.l2_ctas == 1 && wa + wb <= 20 && smem_a + smem_b <= 227 * 1024) {
        // the default: both table placements in one CTA per SM (the global-table rows of `gtables` are indexed by
        // CTA, so the grid is the shared-table grid: one CTA per SM)
        const u32 sf = c.opt.mixed == 2 ? 1u : 0u;
        const dim3 grid((unsigned)c.sm_count), block((wa + wb) * 32);
        const size_t sm = smem_a + smem_b;
        // option `two`: the two-window round for the global-table warps (1), the shared-table warps (2), both (3)
        if (rules)
            k_compress_window_mixed<true><<<grid, block, sm, st>>>(A, wa, wb, ra, rb, sf);
#ifdef SB200_EXPERIMENTS
        // the pipelined round (compress_pipe.cuh) and the one-copy-of-the-code kernel: exact, measured, not faster
        // (profiles/r02h_pipelined_round.md: the loads are hidden, but the round needs 33-40 % more instructions)
        else if (c.opt.unified && c.opt.pipe)
            k_compress_window_mixed<false, false, false, 3, true><<<grid, block, sm, st>>>(A, wa, wb, ra, rb, sf);
        else if (c.opt.unified)
            k_compress_window_mixed<false, false, false, 0, true><<<grid, block, sm, st>>>(A, wa, wb, ra, rb, sf);
        else if (c.opt.pipe == 1)
            k_compress_window_mixed<false, false, false, 1><<<grid, block, sm, st>>>(A, wa, wb, ra, rb, sf);
        else if (c.opt.pipe == 2)
            k_compress_window_mixed<false, false, false, 2><<<grid, block, sm, st>>>(A, wa, wb, ra, rb, sf);
        else if (c.opt.pipe == 3)
            k_compress_window_mixed<false, false, false, 3><<<grid, block, sm, st>>>(A, wa, wb, ra, rb, sf);
        // measured slower (profiles/r02g_sweep_two_window.txt): 16.4 / 13.0 / 18.8 ms against 12.6 ms
        else if (c.opt.two == 1)
            k_compress_window_mixed<false, false, true><<<grid, block, sm, st>>>(A, wa, wb, ra, rb, sf);
        else if (c.opt.two == 2)
            k_compress_window_mixed<false, true, false><<<grid, block, sm, st>>>(A, wa, wb, ra, rb, sf);
        else if (c.opt.two == 3)
            k_compress_window_mixed<false, true, true><<<grid, block, sm, st>>>(A, wa, wb, ra, rb, sf);
#endif
        else
            k_compress_window_mixed<false><<<grid, block, sm, st>>>(A, wa, wb, ra, rb, sf);
        *launches += 1;
        if (prof) {
            CU(cudaStreamSynchronize(st));
            cudaProfilerStop();
        }
        return SNAPPY_B200_OK;
    }
    const bool l2_first = c.opt.l2_first != 0 && ctas_a && ctas_b;
    if (ctas_b && l2_first) CU(cudaStreamWaitEvent(c.side, c.ev_fork, 0));
    auto launch_b = [&]() -> int {
        if (c.opt.l2_persist && c.l2_persist_max && c.l2_window_max) {
            // keep the global hash tables resident in L2: they are the randomly read-and-written state, the
            // fragment bytes stream through the rest of the cache
            cudaStreamAttrValue av;
            memset(&av, 0, sizeof av);
            size_t bytes = (size_t)ctas_b * wb * kMaxTableEntries * 2;
            if (bytes > c.l2_window_max) bytes = c.l2_window_max;
            av.accessPolicyWindow.base_ptr = c.gtables.p;
            av.accessPolicyWindow.num_bytes = bytes;
            av.accessPolicyWindow.hitRatio = bytes <= c.l2_persist_max ? 1.0f : (float)c.l2_persist_max / (float)bytes;
            av.accessPolicyWindow.hitProp = cudaAccessPropertyPersisting;
            av.accessPolicyWindow.missProp = cudaAccessPropertyStreaming;
            CU(cudaStreamSetAttribute(c.side, cudaStreamAttributeAccessPolicyWindow, &av));
        }
        if (rules)
            k_compress_window<false, true><<<ctas_b, wb * 32, smem_b, c.side>>>(A, rb);
#ifdef SB200_EXPERIMENTS
        else if (window && c.opt.slowcont)
            k_compress_window<false, false, true><<<ctas_b, wb * 32, smem_b, c.side>>>(A, rb);
        else if (!window)
            k_compress_chain<false><<<ctas_b, wb * 32, 0, c.side>>>(
                d_in, (u64)len, nfrag, shift, (const u8*)c.tail.p, scratch, sizes, counter,
                (u16*)c.gtables.p, (u32)c.opt.spec_l2, reserve, descs, ndesc);
#endif
#ifdef SB200_EXPERIMENTS
        else if (c.opt.pipe & 2)
            k_compress_window<false, false, false, true><<<ctas_b, wb * 32, smem_b, c.side>>>(A, rb);
#endif
        else
            k_compress_window<false><<<ctas_b, wb * 32, smem_b, c.side>>>(A, rb);
        return SNAPPY_B200_OK;
    };
    if (ctas_b && l2_first) {  // experiment: the global-table CTAs take the lower warp slots of every SM
        int r = launch_b();
        if (r != SNAPPY_B200_OK) return r;
    }
    if (ctas_a) {
        if (rules)
            k_compress_window<true, true><<<ctas_a, wa * 32, smem_a, st>>>(A, ra);
#ifdef SB200_EXPERIMENTS
        else if (window && c.opt.slowcont)
            k_compress_window<true, false, true><<<ctas_a, wa * 32, smem_a, st>>>(A, ra);
        else if (!window)
            k_compress_chain<true><<<ctas_a, wa * 32, (size_t)wa * kMaxTableEntries * 2, st>>>(
                d_in, (u64)len, nfrag, shift, (const u8*)c.tail.p, scratch, sizes, counter, nullptr,
                (u32)c.opt.spec_smem, 0u, descs, ndesc);
#endif
#ifdef SB200_EXPERIMENTS
        else if (c.opt.pipe & 1)
            k_compress_window<true, false, false, true><<<ctas_a, wa * 32, smem_a, st>>>(A, ra);
#endif
        else
            k_compress_window<true><<<ctas_a, wa * 32, smem_a, st>>>(A, ra);
    }
    *launches += 1;
    if (ctas_b) {
        if (!l2_first) {
            CU(cudaStreamWaitEvent(c.side, c.ev_fork, 0));
            int r = launch_b();
            if (r != SNAPPY_B200_OK) return r;
        }
        CU(cudaEventRecord(c.ev_join, c.side));
        CU(cudaStreamWaitEvent(st, c.ev_join, 0));
        *launches += 1;
    }
    if (prof) {
        CU(cudaStreamSynchronize(st));
        cudaProfilerStop();
    }
    return SNAPPY_B200_OK;
}

// Compress the fragments of one shard into d_out + base (elements only) and return the number of
// bytes behind d_out (base + elements).  d_index (optional): nfrag+1 stream offsets.
int compress_shard_locked(Context& c, const u8* d_in, size_t shard_len, u64 total_len, u8* d_out,
                          u64 base, u64* total_out, u64* d_index, u32* d_frag_sizes_out,
                          cudaStream_t st) {
    const u32 nfrag = (u32)((shard_len + kBlockSize - 1) / kBlockSize);
    c.last_launches[0] = 0;
    if (nfrag == 0) {
        *total_out = base;
        if (d_index) {
            u64* h = (u64*)c.pinned;
            h[0] = base;
            CU(cudaMemcpyAsync(d_index, h, 8, cudaMemcpyHostToDevice, st));
            CU(cudaStreamSynchronize(st));
        }
        return SNAPPY_B200_OK;
    }
    CU(c.scratch.ensure((size_t)nfrag * kSlotStride));
    CU(c.frag_sizes.ensure((size_t)nfrag * sizeof(u32)));
    CU(c.frag_offsets.ensure(((size_t)nfrag + 1) * sizeof(u64)));
    const u32 shift = table_shift(total_len);
    u8* scratch = (u8*)c.scratch.p;
    u32* sizes = (u32*)c.frag_sizes.p;
    u64* offs = (u64*)c.frag_offsets.p;

    int launches = 0;
    if (c.opt.compress_variant == 0 && c.opt.window && !c.opt.wide && c.opt.overlap_compact && nfrag >= 4096) {
        // compaction overlapped with compression: the persistent kernels count finished fragments per chunk
        // of 1024; a scan + compaction per chunk, enqueued on a second stream, waits for its count, so only
        // the last chunk's compaction is left when the compress kernels end
        const size_t cf = 1024;
        const int nchunks = (int)((nfrag + cf - 1) / cf);
        if (nchunks > kMaxPipeChunks) return SNAPPY_B200_BAD_ARGUMENT;
        CU(c.frag_offsets.ensure(((size_t)nfrag + 2) * sizeof(u64)));
        offs = (u64*)c.frag_offsets.p;
        CU(c.flags.ensure(64 + (size_t)kMaxPipeChunks * 4));
        CU(c.tail.ensure(kTailSlot));
        u64* running = offs + nfrag + 1;
        u32* d_done = (u32*)((u8*)c.flags.p + 64);
        u64* h_tot = (u64*)((u8*)c.pinned + 2048);
        u64* h_base = (u64*)((u8*)c.pinned + 96);
        *h_base = base;
        CU(cudaMemsetAsync(c.flags.p, 0, 64 + (size_t)nchunks * 4, st));
        CU(cudaMemcpyAsync(running, h_base, 8, cudaMemcpyHostToDevice, st));
        int rc = stage_tail(c, d_in, shard_len, 0, st);
        if (rc != SNAPPY_B200_OK) return rc;
        CU(cudaEventRecord(c.ev_in[0], st));
        CU(cudaStreamWaitEvent(c.s_pack, c.ev_in[0], 0));
        Gate gate;
        gate.done = d_done;
        gate.div = (u32)cf;
        if (c.opt.timing) CU(cudaEventRecord(c.ev[0], st));
        rc = launch_chain_kernels(c, d_in, shard_len, shift, scratch, sizes, st, &launches, nullptr, 0, 0, &gate);
        if (rc != SNAPPY_B200_OK) return rc;
        if (c.opt.timing) {
            CU(cudaEventRecord(c.ev[1], st));
            c.ev_pending[0] = true;
        }
        for (int i = 0; i < nchunks; i++) {
            const size_t f0 = (size_t)i * cf;
            const u32 nf = (u32)((nfrag - f0 < cf) ? (nfrag - f0) : cf);
            k_scan_chunk<<<1, 256, 0, c.s_pack>>>(sizes + f0, nf, offs + f0, running, d_done + i, nf, h_tot + i);
            k_compact<<<nf, 256, 0, c.s_pack>>>(scratch + f0 * kSlotStride, sizes + f0, offs + f0, d_out);
            launches += 2;
        }
        CU(cudaEventRecord(c.ev_done[0], c.s_pack));
        CU(cudaStreamWaitEvent(st, c.ev_done[0], 0));
        c.last_launches[0] = launches;
        CU(cudaGetLastError());
        if (d_index)
            CU(cudaMemcpyAsync(d_index, offs, ((size_t)nfrag + 1) * 8, cudaMemcpyDeviceToDevice, st));
        if (d_frag_sizes_out)
            CU(cudaMemcpyAsync(d_frag_sizes_out, sizes, (size_t)nfrag * 4, cudaMemcpyDeviceToDevice, st));
        CU(cudaStreamSynchronize(st));
        harvest_timing(c, 0);
        *total_out = ((volatile u64*)h_tot)[nchunks - 1];
        return SNAPPY_B200_OK;
    }
    if (c.opt.compress_variant == 0 || c.opt.rules) {
        if (c.opt.timing) CU(cudaEventRecord(c.ev[0], st));
        int rc = launch_chain_kernels(c, d_in, shard_len, shift, scratch, sizes, st, &launches);
        if (rc != SNAPPY_B200_OK) return rc;
    }
#ifdef SB200_EXPERIMENTS
    else {
        if (c.opt.timing) CU(cudaEventRecord(c.ev[0], st));
        if (c.opt.compress_variant == 1)
            k_compress_fragments_serial<<<nfrag, 32, kCompressSmemBytes, st>>>(d_in, (u64)shard_len, shift,
                                                                              scratch, sizes);
        else
            k_compress_fragments<<<nfrag, 64, kCompress2SmemBytes, st>>>(d_in, (u64)shard_len, shift,
                                                                        scratch, sizes);
        launches = 1;
    }
#endif
    if (c.opt.timing) {
        CU(cudaEventRecord(c.ev[1], st));
        c.ev_pending[0] = true;
    }
    k_scan_sizes<<<1, 1024, 0, st>>>(sizes, nfrag, base, offs);
    k_compact<<<nfrag, 256, 0, st>>>(scratch, sizes, offs, d_out);
    c.last_launches[0] = launches + 2;
    CU(cudaGetLastError());
    u64* h = (u64*)c.pinned;
    CU(cudaMemcpyAsync(h, offs + nfrag, 8, cudaMemcpyDeviceToHost, st));
    if (d_index)
        CU(cudaMemcpyAsync(d_index, offs, ((size_t)nfrag + 1) * 8, cudaMemcpyDeviceToDevice, st));
    if (d_frag_sizes_out)
        CU(cudaMemcpyAsync(d_frag_sizes_out, sizes, (size_t)nfrag * 4, cudaMemcpyDeviceToDevice, st));
    CU(cudaStreamSynchronize(st));
    harvest_timing(c, 0);
    *total_out = h[0];
    return SNAPPY_B200_OK;
}

int compress_device_locked(Context& c, const u8* d_in, size_t n, u8* d_out, size_t out_cap,
                           size_t* out_len, u64* d_index, cudaStream_t st) {
    if (n > 0xffffffffull) return SNAPPY_B200_INPUT_TOO_LARGE;  // src/Snappy.jl:21
    if (out_cap < snappy_b200_max_compressed_length(n)) return SNAPPY_B200_BUFFER_TOO_SMALL;
    u8* hdr = (u8*)c.pinned + 64;
    const int k = encode_varint((u32)n, hdr);  // src/Snappy.jl:26
    CU(cudaMemcpyAsync(d_out, hdr, (size_t)k, cudaMemcpyHostToDevice, st));
    u64 total = 0;
    int rc = compress_shard_locked(c, d_in, n, n, d_out, (u64)k, &total, d_index, nullptr, st);
    if (rc != SNAPPY_B200_OK) return rc;
    *out_len = (size_t)total;
    return SNAPPY_B200_OK;
}

// run the exact serial decoder over the whole stream
int decode_exact_locked(Context& c, const u8* d_in, size_t n, size_t hdr, u8* d_out, u32 claimed,
                        cudaStream_t st) {
    DecodeResult* res = (DecodeResult*)c.result.p;
    k_decode_serial<<<1, 32, 0, st>>>(d_in, (u64)n, (u64)hdr, d_out, (u64)claimed, res);
    c.last_launches[1] += 1;
    CU(cudaGetLastError());
    DecodeResult* h = (DecodeResult*)((u8*)c.pinned + 128);
    CU(cudaMemcpyAsync(h, res, sizeof(DecodeResult), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return h->status;
}

// decode with a device-resident index of nfrag+1 offsets; returns OK, or -1 when the fast path
// declined (caller falls back)
// Enqueue the indexed decoder for fragments [fa, fb) on `st`; with host_out, in ranges of
// pipe_chunk_frags fragments, each followed by its device-to-host copy on the copy stream (*ri counts
// the events used).  No synchronisation.
int decode_launch(Context& c, const u8* d_in, size_t n, size_t hdr, u8* d_out, u32 claimed, const u64* d_index,
                  cudaStream_t st, u32 fa, u32 fb, u8* host_out, int* ri, u32 range = 0,
                  const u64* out_start = nullptr, u8* tile_flags = nullptr) {
    const u32 nfrag = frag_count(claimed);
    DecodeResult* res = (DecodeResult*)c.result.p;
    const bool ranged = host_out != nullptr;
    const u32 step = ranged ? (range ? range : (u32)c.opt.pipe_chunk_frags) : (fb - fa);
    for (u32 f0 = fa; f0 < fb; f0 += step) {
        const u32 cnt = (fb - f0 < step) ? (fb - f0) : step;
        const u32 grid = (cnt + kDecodeWarpsPerCta - 1) / kDecodeWarpsPerCta;
        if (c.opt.decode_occupancy == 12)
            k_decode_fragments<12><<<grid, kDecodeWarpsPerCta * 32, 0, st>>>(d_in, d_index, nfrag, f0, cnt, (u64)hdr,
                                                                             (u64)n, d_out, (u64)claimed, res, nullptr,
                                                                             0u, out_start, tile_flags);
        else if (c.opt.decode_occupancy == 10)
            k_decode_fragments<10><<<grid, kDecodeWarpsPerCta * 32, 0, st>>>(d_in, d_index, nfrag, f0, cnt, (u64)hdr,
                                                                             (u64)n, d_out, (u64)claimed, res, nullptr,
                                                                             0u, out_start, tile_flags);
        else
            k_decode_fragments<8><<<grid, kDecodeWarpsPerCta * 32, 0, st>>>(d_in, d_index, nfrag, f0, cnt, (u64)hdr,
                                                                            (u64)n, d_out, (u64)claimed, res, nullptr,
                                                                            0u, out_start, tile_flags);
        c.last_launches[1] += 1;
        if (ranged) {
            if (*ri >= kMaxPipeChunks) return fail_cuda(cudaErrorInvalidValue, "decode_launch: too many ranges");
            const size_t ob = (size_t)f0 * kBlockSize;
            const size_t ol = ((size_t)claimed - ob < (size_t)cnt * kBlockSize) ? ((size_t)claimed - ob)
                                                                                 : (size_t)cnt * kBlockSize;
            CU(cudaEventRecord(c.ev_done[*ri], st));
            if (c.defer_down) {  // pageable destination: the caller drains the range through the bounce slots
                c.defer_down->push_back(Context::DownRange{ob, ol, *ri});
            } else {
                CU(cudaStreamWaitEvent(c.s_d2h, c.ev_done[*ri], 0));
                CU(cudaMemcpyAsync(host_out + ob, d_out + ob, ol, cudaMemcpyDeviceToHost, c.s_d2h));
            }
            *ri += 1;
        }
    }
    return SNAPPY_B200_OK;
}

// Wait for the decoder and read its verdict: OK, or -1 when some fragment was inconsistent with the index.
int decode_finish(Context& c, cudaStream_t st, bool ranged) {
    DecodeResult* res = (DecodeResult*)c.result.p;
    CU(cudaStreamSynchronize(c.s_pack));  // streamed path: the decoder runs there
    if (c.opt.timing) {
        CU(cudaEventRecord(c.ev[3], st));
        c.ev_pending[1] = true;
    }
    CU(cudaGetLastError());
    DecodeResult* h = (DecodeResult*)((u8*)c.pinned + 128);
    CU(cudaMemcpyAsync(h, res, sizeof(DecodeResult), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (ranged) CU(cudaStreamSynchronize(c.s_d2h));
    harvest_timing(c, 1);
    return h->fallback ? -1 : SNAPPY_B200_OK;
}

int decode_indexed_locked(Context& c, const u8* d_in, size_t n, size_t hdr, u8* d_out, u32 claimed,
                          const u64* d_index, cudaStream_t st, u8* host_out = nullptr,
                          bool* host_copied = nullptr) {
    const u32 nfrag = frag_count(claimed);
    if (nfrag == 0) return -1;
    CU(cudaMemsetAsync(c.result.p, 0, sizeof(DecodeResult), st));
    if (c.opt.timing) CU(cudaEventRecord(c.ev[2], st));
    // host-buffer API: decode in ranges and send each finished range down while the next decodes
    const bool ranged = host_out && c.opt.host_pipeline && nfrag > (u32)c.opt.pipe_chunk_frags;
    int ri = 0;
    int rc = decode_launch(c, d_in, n, hdr, d_out, claimed, d_index, st, 0, nfrag, ranged ? host_out : nullptr, &ri);
    if (rc != SNAPPY_B200_OK) return rc;
    rc = decode_finish(c, st, ranged);
    if (rc != SNAPPY_B200_OK) return rc;
    if (ranged && host_copied) *host_copied = true;
    return SNAPPY_B200_OK;
}

// Segmented speculative parse (parse.cuh) of the segment [hdr, E) of the stream d_in[0 .. n): hdr is
// an element start, elements may run past E.  Writes the side-index entries of the 64 KiB output
// boundaries inside the segment into c.index (nfrag + 1 entries for the whole stream), given that
// the segments before it produced out_base bytes.  *seg_exit = first element start >= E (n at the
// end of the stream), *seg_out = output bytes of the segment.  Returns 0 when the index entries are
// ready, -1 when the stream is not fragment-clean or shows any anomaly (the exact serial decoder then
// decides), or a CUDA error status (> 0).
int build_index_segment(Context& c, const u8* d_in, size_t n, size_t hdr, size_t E, u64 out_base, u32 nfrag,
                        cudaStream_t st, u64* seg_exit, u64* seg_out, u64* out_start = nullptr,
                        u64* flags_out = nullptr, u64 out_total = 0, u64* first_err = nullptr) {
    if (nfrag == 0 || E <= hdr) return -1;
    const u64 body = E - hdr;
    const u32 pshift = (u32)c.opt.parse_chunk_log2;
    const u64 pchunk = 1ull << pshift;
    if (body / pchunk >= 0x7ffffff0ull) return -1;
    const u32 nchunk = (u32)((body + pchunk - 1) / pchunk);
    CU(c.parse_a.ensure(ParseArrays::bytes(nchunk)));
    CU(c.parse_c.ensure(((size_t)nchunk + 1) * 8));  // output offsets
    CU(c.index.ensure(((size_t)nfrag + 1) * 8));
    ParseArrays pa;
    pa.carve(c.parse_a.p, nchunk);
    u64* out_off = (u64*)c.parse_c.p;
    u32* h = (u32*)((u8*)c.pinned + 1024);

    CU(cudaMemsetAsync(pa.counters, 0, 64, st));
    CU(cudaMemsetAsync((u8*)pa.counters + 16, 0xff, 8, st));  // first failing element: none yet
    const u32 pgrid = (nchunk + kParseThreads - 1) / kParseThreads;
    const u32 lgrid = (nchunk + 255) / 256;
    k_parse_guess<<<pgrid, kParseThreads, 0, st>>>(d_in, (u64)n, (u64)hdr, nchunk, pa, (u64)E, pshift);
    k_parse_bridge<<<pgrid, kParseThreads, 0, st>>>(d_in, (u64)n, (u64)hdr, nchunk, pa, (u64)E, pshift);
    c.last_launches[1] += 2;
    // pointer doubling: after r rounds everything within 2^r hops of chunk 0 is marked
    u32* nx = pa.next_a;
    u32* nx2 = pa.next_b;
    // keep the original successor array for the broken-chain check: doubling works on copies
    CU(c.parse_b.ensure((size_t)nchunk * 4));
    u32* next_orig = (u32*)c.parse_b.p;
    CU(cudaMemcpyAsync(next_orig, pa.next_a, (size_t)nchunk * 4, cudaMemcpyDeviceToDevice, st));
    for (u32 span = 1; span < nchunk; span <<= 1) {
        k_parse_reach<<<lgrid, 256, 0, st>>>(nchunk, nx, nx2, pa.reach);
        u32* t = nx;
        nx = nx2;
        nx2 = t;
        c.last_launches[1] += 1;
    }
    k_parse_reach<<<lgrid, 256, 0, st>>>(nchunk, nx, nx2, pa.reach);
    k_parse_entries<<<pgrid, kParseThreads, 0, st>>>(d_in, (u64)n, (u64)hdr, nchunk, pa, next_orig, 0, (u64)E, pshift);
    k_parse_entries<<<pgrid, kParseThreads, 0, st>>>(d_in, (u64)n, (u64)hdr, nchunk, pa, next_orig, 1, (u64)E, pshift);
    k_parse_final<<<pgrid, kParseThreads, 0, st>>>(d_in, (u64)n, (u64)hdr, nchunk, pa, (u64)E, pshift);
    k_scan_sizes<<<1, 1024, 0, st>>>(pa.outb, nchunk, 0, out_off);
    k_build_index<<<pgrid, kParseThreads, 0, st>>>(d_in, (u64)n, (u64)hdr, nchunk, pa, out_off, (u64*)c.index.p, nfrag,
                                                  (u64)E, out_base, pshift, out_start, out_start ? 1u : 0u, out_total);
    c.last_launches[1] += 6;
    CU(cudaGetLastError());
    volatile u64* h3 = (volatile u64*)h;
    k_parse_report<<<1, 1, 0, st>>>(pa.counters, out_off + nchunk, (u64*)h);
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(st));
    const u64 flags = h3[0], ex = h3[1], total = h3[2];
    if (getenv("SNAPPY_B200_DEBUG"))
        fprintf(stderr, "[snappy_b200] parse [%zu, %zu): nchunk=%u flags=%u out=%llu exit=%llu\n", hdr, E, nchunk,
                (unsigned)flags, (unsigned long long)total, (unsigned long long)ex);
    *seg_exit = ex;
    *seg_out = total;
    if (first_err) *first_err = h3[3];
    if (flags_out) {  // relaxed whole-stream mode: the caller decides what the flags mean
        *flags_out = flags;
        return 0;
    }
    if (flags != 0) return -1;
    return 0;
}

// The whole stream as one segment.
int build_index_locked(Context& c, const u8* d_in, size_t n, size_t hdr, u32 claimed, cudaStream_t st) {
    const u32 nfrag = frag_count(claimed);
    if (nfrag == 0 || n <= hdr) return -1;
    u64 ex = 0, total = 0;
    const int rc = build_index_segment(c, d_in, n, hdr, n, 0, nfrag, st, &ex, &total);
    if (rc != 0) return rc;
    return total == claimed ? 0 : -1;
}

// Arbitrary stream, no usable side index.  The parse builds the tile index (relaxed: a literal may straddle a 64 KiB
// boundary); the indexed decoder runs over every tile whose both ends are known and marks the tiles it rejects; the
// bounded serial walk (k_decode_serial_tiles) then decodes only those, and everything behind the point where the
// parse lost the chain, with the reference's checks.  So a corrupt 1 GiB stream costs the parallel decode of its good
// prefix plus one tile of serial work, and the status is the reference's.  Returns a status (>= 0), or -1: nothing
// usable came out of the parse (caller: whole-stream serial decoder).
int decode_parsed_locked(Context& c, const u8* d_in, size_t n, size_t hdr, u8* d_out, u32 claimed, cudaStream_t st,
                         u8* host_out, bool* host_copied) {
    const u32 nfrag = frag_count(claimed);
    if (nfrag == 0 || n <= hdr) return -1;
    CU(c.index.ensure(((size_t)nfrag + 1) * 8));
    CU(c.index_out.ensure(((size_t)nfrag + 1) * 8));
    CU(c.tile_flags.ensure((size_t)nfrag + 64));
    u64* idx = (u64*)c.index.p;
    u64* ost = (u64*)c.index_out.p;
    u8* tf = (u8*)c.tile_flags.p;
    CU(cudaMemsetAsync(idx, 0xff, ((size_t)nfrag + 1) * 8, st));
    CU(cudaMemsetAsync(ost, 0xff, ((size_t)nfrag + 1) * 8, st));
    CU(cudaMemsetAsync(tf, 0, (size_t)nfrag + 64, st));
    u64* hseed = (u64*)((u8*)c.pinned + 3072);  // tile 0 starts behind the header whatever the parse finds
    hseed[0] = hdr;
    hseed[1] = 0;
    hseed[2] = claimed;
    CU(cudaMemcpyAsync(idx, hseed, 8, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ost, hseed + 1, 8, cudaMemcpyHostToDevice, st));
    u64 ex = 0, total = 0, pflags = 0, first_err = ~0ull;
    int rc = build_index_segment(c, d_in, n, hdr, n, 0, nfrag, st, &ex, &total, ost, &pflags, (u64)claimed, &first_err);
    if (rc != 0) return rc;
    if (first_err != ~0ull) {
        // an element the reference rejects, found by the parse (header + output position decide, not data): its
        // status, at once -- the reference stops there too and hands out nothing
        c.last_path = 1;
        return (int)(first_err & 7);
    }
    if (!(pflags & (PF_ANOMALY | PF_BROKEN)) && total != claimed) {
        c.last_path = 1;
        return SNAPPY_B200_INVALID_INPUT;  // every element is fine, the lengths do not add up (src/Snappy.jl:50)
    }
    CU(cudaMemcpyAsync(ost + nfrag, hseed + 2, 8, cudaMemcpyHostToDevice, st));
    const bool complete = !(pflags & (PF_ANOMALY | PF_BROKEN)) && total == claimed;
    if (complete && (pflags & PF_NOT_CLEAN) && nfrag > 1 && c.opt.clean_cuts) {
        // copies reach across the 64 KiB boundaries: move every tile start back to the nearest clean cut (parse.cuh),
        // so that the tiles are self-contained again wherever the stream allows it.  The parse arrays of
        // build_index_segment (entries, output offsets per chunk) are still in place.
        const u32 pshift = (u32)c.opt.parse_chunk_log2;
        const u64 pchunk = 1ull << pshift;
        const u32 nchunk = (u32)(((u64)(n - hdr) + pchunk - 1) / pchunk);
        ParseArrays pa;
        pa.carve(c.parse_a.p, nchunk);
        const u64* out_off = (const u64*)c.parse_c.p;
        CU(c.parse_d.ensure((size_t)nchunk * 16));
        u64* low = (u64*)c.parse_d.p;
        u64* sfx = low + nchunk;
        const u32 pgrid = (nchunk + kParseThreads - 1) / kParseThreads;
        k_cut_low<<<pgrid, kParseThreads, 0, st>>>(d_in, (u64)n, (u64)hdr, nchunk, pa, out_off, (u64)n, pshift, low);
        k_suffix_min<<<1, 1024, 0, st>>>(low, nchunk, sfx);
        k_cut_tiles<<<(nfrag - 1 + kParseThreads - 1) / kParseThreads, kParseThreads, 0, st>>>(
            d_in, (u64)n, (u64)hdr, nchunk, pa, out_off, sfx, (u64)n, pshift, nfrag, idx, ost);
        k_cut_fill<<<1, 32, 0, st>>>(nfrag, idx, ost);
        c.last_launches[1] += 4;
        CU(cudaGetLastError());
    }
    u32 tvalid = nfrag;  // tiles [0, tvalid) have both ends in the index
    if (!complete) {
        u32* d_first = (u32*)((u8*)c.result.p + 128);
        u32* h_first = (u32*)((u8*)c.pinned + 3104);
        *h_first = nfrag + 1;
        CU(cudaMemcpyAsync(d_first, h_first, 4, cudaMemcpyHostToDevice, st));
        k_first_missing<<<(nfrag + 1 + 255) / 256, 256, 0, st>>>(idx, nfrag, (u64)n, d_first);
        CU(cudaMemcpyAsync(h_first, d_first, 4, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        const u32 first = *h_first;  // index[first] was never written (<= nfrag when the chain broke)
        tvalid = first == 0 ? 0u : (first > nfrag ? nfrag : first - 1);
        if (first <= nfrag && first > 0 && tvalid > 0) tvalid = first - 1;
    }
    CU(cudaMemsetAsync(c.result.p, 0, sizeof(DecodeResult), st));
    if (c.opt.timing) CU(cudaEventRecord(c.ev[2], st));
    // host-buffer API: ranged device-to-host copies only when the tiles are the aligned 64 KiB fragments
    const bool ranged = host_out && pflags == 0 && complete && c.opt.host_pipeline && nfrag > (u32)c.opt.pipe_chunk_frags;
    int ri = 0;
    if (tvalid) {
        rc = decode_launch(c, d_in, n, hdr, d_out, claimed, idx, st, 0, tvalid, ranged ? host_out : nullptr, &ri, 0, ost, tf);
        if (rc != SNAPPY_B200_OK) return rc;
    }
    rc = decode_finish(c, st, ranged);
    if (rc > 0) return rc;
    if (rc == 0 && complete) {
        if (ranged && host_copied) *host_copied = true;
        c.last_path = 1;
        return SNAPPY_B200_OK;
    }
    c.last_path = 2;
    // some tiles were rejected, or the index ends early: the bounded serial walk decides
    if (tvalid < nfrag) CU(cudaMemsetAsync(tf + tvalid, 1, nfrag - tvalid, st));
    if (!complete) CU(cudaMemsetAsync(tf + nfrag - 1, 1, 1, st));  // the walk must see the end of the stream (length check)
    DecodeResult* res = (DecodeResult*)c.result.p;
    k_decode_serial_tiles<<<1, 32, 0, st>>>(d_in, (u64)n, idx, ost, nfrag, tf, d_out, (u64)claimed, res);
    c.last_launches[1] += 1;
    CU(cudaGetLastError());
    DecodeResult* h = (DecodeResult*)((u8*)c.pinned + 128);
    CU(cudaMemcpyAsync(h, res, sizeof(DecodeResult), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    if (host_copied) *host_copied = false;  // ranges that went down early may hold bytes of rejected tiles
    return h->status;
}

int uncompress_device_locked(Context& c, const u8* d_in, size_t n, u8* d_out, size_t out_cap,
                             size_t* out_len, const u64* d_index, cudaStream_t st, u8* host_out = nullptr,
                             bool* host_copied = nullptr) {
    c.last_launches[1] = 0;
    // the varint header decides the output size (src/Snappy.jl:47)
    u8* hb = (u8*)c.pinned + 256;
    const size_t hn = n < 5 ? n : 5;
    if (hn) {
        CU(cudaMemcpyAsync(hb, d_in, hn, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    u32 claimed = 0;
    size_t hdr = 0;
    int rc = parse_varint(hb, hn, &claimed, &hdr);
    if (rc != SNAPPY_B200_OK) return rc;
    if (out_cap < claimed) return SNAPPY_B200_BUFFER_TOO_SMALL;
    *out_len = claimed;
    if (c.opt.decode_variant != 1) {
        if (d_index) {  // a wrong index cannot change the result: any rejected fragment sends us to the parse
            c.last_path = 0;
            rc = decode_indexed_locked(c, d_in, n, hdr, d_out, claimed, d_index, st, host_out, host_copied);
            if (rc >= 0) return rc;
            if (host_copied) *host_copied = false;
        }
        rc = decode_parsed_locked(c, d_in, n, hdr, d_out, claimed, st, host_out, host_copied);
        if (rc >= 0) return rc;
    }
    c.last_path = 3;
    return decode_exact_locked(c, d_in, n, hdr, d_out, claimed, st);
}

// ---- validation (snappy_b200_validate_*): uncompress_device_locked's chain, status only --------------------------
// The same paths in the same order with the same verdicts, but no output buffer: the device memory is the parse's
// (O(n / parse chunk)) plus the tile index (O(claimed / 64 KiB)), never O(claimed).

// status-only whole-stream walk (path 3)
int validate_exact_locked(Context& c, const u8* d_in, size_t n, size_t hdr, u32 claimed, cudaStream_t st) {
    DecodeResult* res = (DecodeResult*)c.result.p;
    k_validate_serial<<<1, 32, 0, st>>>(d_in, (u64)n, (u64)hdr, (u64)claimed, res);
    c.last_launches[1] += 1;
    CU(cudaGetLastError());
    DecodeResult* h = (DecodeResult*)((u8*)c.pinned + 128);
    CU(cudaMemcpyAsync(h, res, sizeof(DecodeResult), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return h->status;
}

// path 0: every fragment of the side index is clean -> OK; -1 when some fragment is not (caller: the parse)
int validate_indexed_locked(Context& c, const u8* d_in, size_t n, size_t hdr, u32 claimed, const u64* d_index,
                            cudaStream_t st) {
    const u32 nfrag = frag_count(claimed);
    if (nfrag == 0) return -1;
    CU(cudaMemsetAsync(c.result.p, 0, sizeof(DecodeResult), st));
    if (c.opt.timing) CU(cudaEventRecord(c.ev[2], st));
    const u32 grid = (nfrag + kDecodeWarpsPerCta - 1) / kDecodeWarpsPerCta;
    k_validate_fragments<<<grid, kDecodeWarpsPerCta * 32, 0, st>>>(d_in, d_index, nfrag, (u64)hdr, (u64)n,
                                                                    (u64)claimed, (DecodeResult*)c.result.p);
    c.last_launches[1] += 1;
    return decode_finish(c, st, false);
}

// decode_parsed_locked without the decode.  The parse's first failing element and its length check decide every
// stream whose chain it followed to the end (path 1): a complete, error-free parse whose lengths add up means the
// reference accepts the stream, because its three element checks depend on the element header and the output position
// only (k_build_index).  A parse that lost the chain hands over to the status-only walk from the last tile start it
// reached (path 2).  -1: nothing usable came out of the parse (caller: whole-stream walk).
int validate_parsed_locked(Context& c, const u8* d_in, size_t n, size_t hdr, u32 claimed, cudaStream_t st) {
    const u32 nfrag = frag_count(claimed);
    if (nfrag == 0 || n <= hdr) return -1;
    CU(c.index.ensure(((size_t)nfrag + 1) * 8));
    CU(c.index_out.ensure(((size_t)nfrag + 1) * 8));
    CU(c.tile_flags.ensure((size_t)nfrag + 64));
    u64* idx = (u64*)c.index.p;
    u64* ost = (u64*)c.index_out.p;
    u8* tf = (u8*)c.tile_flags.p;
    CU(cudaMemsetAsync(idx, 0xff, ((size_t)nfrag + 1) * 8, st));
    CU(cudaMemsetAsync(ost, 0xff, ((size_t)nfrag + 1) * 8, st));
    u64* hseed = (u64*)((u8*)c.pinned + 3072);  // tile 0 starts behind the header whatever the parse finds
    hseed[0] = hdr;
    hseed[1] = 0;
    hseed[2] = claimed;
    CU(cudaMemcpyAsync(idx, hseed, 8, cudaMemcpyHostToDevice, st));
    CU(cudaMemcpyAsync(ost, hseed + 1, 8, cudaMemcpyHostToDevice, st));
    u64 ex = 0, total = 0, pflags = 0, first_err = ~0ull;
    int rc = build_index_segment(c, d_in, n, hdr, n, 0, nfrag, st, &ex, &total, ost, &pflags, (u64)claimed, &first_err);
    if (rc != 0) return rc;
    c.last_path = 1;
    if (first_err != ~0ull) return (int)(first_err & 7);
    if (!(pflags & (PF_ANOMALY | PF_BROKEN)))
        return total == claimed ? SNAPPY_B200_OK : SNAPPY_B200_INVALID_INPUT;  // src/Snappy.jl:50
    // the chain broke: tiles [0, tvalid) have both ends in the index; the walk starts at the last entry the parse wrote
    // and runs to the end of the stream (the length check) or to the first failing element
    CU(cudaMemcpyAsync(ost + nfrag, hseed + 2, 8, cudaMemcpyHostToDevice, st));
    u32* d_first = (u32*)((u8*)c.result.p + 128);
    u32* h_first = (u32*)((u8*)c.pinned + 3104);
    *h_first = nfrag + 1;
    CU(cudaMemcpyAsync(d_first, h_first, 4, cudaMemcpyHostToDevice, st));
    k_first_missing<<<(nfrag + 1 + 255) / 256, 256, 0, st>>>(idx, nfrag, (u64)n, d_first);
    CU(cudaMemcpyAsync(h_first, d_first, 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    const u32 first = *h_first;
    u32 tvalid = first == 0 ? 0u : (first > nfrag ? nfrag : first - 1);
    if (first <= nfrag && first > 0 && tvalid > 0) tvalid = first - 1;
    c.last_path = 2;
    CU(cudaMemsetAsync(tf, 0, (size_t)nfrag + 64, st));
    if (tvalid < nfrag) CU(cudaMemsetAsync(tf + tvalid, 1, nfrag - tvalid, st));
    CU(cudaMemsetAsync(tf + nfrag - 1, 1, 1, st));  // the walk must see the end of the stream (length check)
    CU(cudaMemsetAsync(c.result.p, 0, sizeof(DecodeResult), st));
    DecodeResult* res = (DecodeResult*)c.result.p;
    k_validate_serial_tiles<<<1, 32, 0, st>>>(d_in, (u64)n, idx, ost, nfrag, tf, (u64)claimed, res);
    c.last_launches[1] += 2;
    CU(cudaGetLastError());
    DecodeResult* h = (DecodeResult*)((u8*)c.pinned + 128);
    CU(cudaMemcpyAsync(h, res, sizeof(DecodeResult), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    return h->status;
}

// uncompress_device_locked, step for step, without an output: the status uncompress returns when out_cap is unlimited
int validate_device_locked(Context& c, const u8* d_in, size_t n, const u64* d_index, size_t* claimed_out,
                           cudaStream_t st) {
    c.last_launches[1] = 0;
    u8* hb = (u8*)c.pinned + 256;
    const size_t hn = n < 5 ? n : 5;
    if (hn) {
        CU(cudaMemcpyAsync(hb, d_in, hn, cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
    }
    u32 claimed = 0;
    size_t hdr = 0;
    int rc = parse_varint(hb, hn, &claimed, &hdr);
    if (rc != SNAPPY_B200_OK) return rc;
    if (claimed_out) *claimed_out = claimed;
    if (c.opt.decode_variant != 1) {
        if (d_index) {  // as in uncompress: a wrong index only costs the fragment pass
            c.last_path = 0;
            rc = validate_indexed_locked(c, d_in, n, hdr, claimed, d_index, st);
            if (rc >= 0) return rc;
        }
        rc = validate_parsed_locked(c, d_in, n, hdr, claimed, st);
        if (rc >= 0) return rc;
    }
    c.last_path = 3;
    return validate_exact_locked(c, d_in, n, hdr, claimed, st);
}

// Takes a lane of the addressed device for the duration of a call: resolves the device, makes it current (the
// caller's current device is restored on exit), picks a free lane or creates one.
struct Locked {
    std::unique_lock<std::mutex> lk;
    Context* c = nullptr;
    int rc = SNAPPY_B200_OK;
    int prev_device = -1;
    Locked() {
        parse_env_options();
        int d = -1;
        rc = resolve_device(&d);
        if (rc != SNAPPY_B200_OK) return;
        cudaGetDevice(&prev_device);
        cudaError_t e = cudaSetDevice(d);
        if (e != cudaSuccess) {
            rc = fail_cuda(e, "cudaSetDevice");
            return;
        }
        DeviceSlot& slot = g_dev[d];
        {
            std::unique_lock<std::mutex> sl(slot.mu);
            for (int i = 0; i < slot.nlanes && !c; i++) {
                std::unique_lock<std::mutex> t(slot.lanes[i]->mu, std::try_to_lock);
                if (t.owns_lock()) {
                    lk = std::move(t);
                    c = slot.lanes[i];
                }
            }
            if (!c && slot.nlanes < kMaxLanes) {
                Context* n = new Context();
                n->lane = slot.nlanes;
                lk = std::unique_lock<std::mutex>(n->mu);
                rc = ctx_init(*n, d, slot);
                if (rc != SNAPPY_B200_OK) {
                    lk.unlock();
                    lk = std::unique_lock<std::mutex>();
                    delete n;
                    return;
                }
                slot.lanes[slot.nlanes++] = n;
                c = n;
            }
        }
        if (!c) {  // every lane is busy: wait for one (spread the waiters over the lanes)
            static std::atomic<unsigned> turn{0};
            Context* w = g_dev[d].lanes[turn.fetch_add(1) % kMaxLanes];
            lk = std::unique_lock<std::mutex>(w->mu);
            c = w;
        }
        tl_last = c;
    }
    ~Locked() {
        if (lk.owns_lock()) lk.unlock();
        if (prev_device >= 0) cudaSetDevice(prev_device);
    }
};

}  // namespace

// ------------------------------------------------------------------------------------------
extern "C" {

const char* snappy_b200_status_string(int status) {
    switch (status) {
        case SNAPPY_B200_OK: return "OK";
        case SNAPPY_B200_INPUT_TOO_LARGE: return "Input too large.";
        case SNAPPY_B200_INVALID_INPUT: return "Invalid input.";
        case SNAPPY_B200_CORRUPT_COPY_OFFSET: return "Invalid input: corrupt copy offset";
        case SNAPPY_B200_CORRUPT_COPY_LENGTH: return "Invalid input: corrupt copy length";
        case SNAPPY_B200_CORRUPT_LITERAL: return "Invalid input: corrupt literal";
        case SNAPPY_B200_BAD_VARINT: return "Could not decode varint32.";
        case SNAPPY_B200_BUFFER_TOO_SMALL: return "output buffer too small";
        case SNAPPY_B200_CUDA_ERROR: return "CUDA error";
        case SNAPPY_B200_NO_DEVICE: return "no usable sm_100 CUDA device";
        case SNAPPY_B200_BAD_ARGUMENT: return "bad argument";
        default: return "unknown status";
    }
}

const char* snappy_b200_last_error(void) { return g_last_error.c_str(); }

int snappy_b200_init(int device) {
    // device >= 0: bind the calling thread to that device; < 0: unbind (current CUDA device / $SNAPPY_B200_DEVICE)
    if (device >= 0) {
        int count = 0;
        cudaError_t e = cudaGetDeviceCount(&count);
        if (e != cudaSuccess || count == 0) {
            g_last_error = std::string("no CUDA device: ") + cudaGetErrorString(e);
            return SNAPPY_B200_NO_DEVICE;
        }
        if (device >= count || device >= kMaxDevices) {
            char buf[96];
            snprintf(buf, sizeof buf, "device %d does not exist (%d CUDA devices)", device, count);
            g_last_error = buf;
            return SNAPPY_B200_BAD_ARGUMENT;
        }
    }
    tl_device = device < 0 ? -1 : device;
    Locked L;  // creates the first lane of the device (checks that it is an sm_100 part)
    return L.rc;
}

void snappy_b200_shutdown(void) {
    // releases every lane of every device; callers must not be inside another entry point
    int prev = -1;
    cudaGetDevice(&prev);
    for (int d = 0; d < kMaxDevices; d++) {
        DeviceSlot& slot = g_dev[d];
        std::unique_lock<std::mutex> sl(slot.mu);
        if (!slot.nlanes) continue;
        cudaSetDevice(d);
        for (int i = 0; i < slot.nlanes; i++) {
            {
                std::unique_lock<std::mutex> lk(slot.lanes[i]->mu);
                ctx_destroy(*slot.lanes[i]);
            }
            if (tl_last == slot.lanes[i]) tl_last = nullptr;
            delete slot.lanes[i];
            slot.lanes[i] = nullptr;
        }
        slot.nlanes = 0;
        slot.once = false;
    }
    if (prev >= 0) cudaSetDevice(prev);
}

size_t snappy_b200_max_compressed_length(size_t n) { return 32 + n + n / 6; }  // src/Snappy.jl:80-82

int snappy_b200_encode_header(uint32_t value, uint8_t out[5]) { return encode_varint(value, out); }

int snappy_b200_parse_header(const uint8_t* in, size_t n, uint32_t* value, size_t* header_len) {
    if (!in && n) return SNAPPY_B200_BAD_ARGUMENT;
    return parse_varint(in, n, value, header_len);
}

int snappy_b200_uncompressed_length(const uint8_t* in, size_t n, size_t* result) {
    u32 v = 0;
    size_t hdr = 0;
    int rc = parse_varint(in, n, &v, &hdr);
    if (rc == SNAPPY_B200_OK) *result = v;
    return rc;
}

// src/internal.jl:344-387 on the host (tests call Snappy.find_match_length directly)
size_t snappy_b200_find_match_length(const uint8_t* a, size_t i1, size_t i2, size_t limit) {
    size_t matched = 0;
    while (i2 + 8 <= limit) {
        u64 x, y;
        memcpy(&x, a + i1 + matched, 8);
        memcpy(&y, a + i2, 8);
        if (x != y) return matched + (size_t)(__builtin_ctzll(x ^ y) >> 3);
        i2 += 8;
        matched += 8;
    }
    while (i2 < limit && a[i1 + matched] == a[i2]) {
        i2++;
        matched++;
    }
    return matched;
}

int snappy_b200_compress_device(const uint8_t* d_in, size_t n, uint8_t* d_out, size_t out_cap,
                                size_t* out_len, uint64_t* d_frag_index, void* stream) {
    if (!out_len || (!d_in && n) || !d_out) return SNAPPY_B200_BAD_ARGUMENT;
    if (n > 0xffffffffull) return SNAPPY_B200_INPUT_TOO_LARGE;  // src/Snappy.jl:21 (before any device work)
    Locked L;
    if (L.rc != SNAPPY_B200_OK) return L.rc;
    return compress_device_locked(*L.c, d_in, n, d_out, out_cap, out_len, (u64*)d_frag_index,
                                  (cudaStream_t)stream);
}

int snappy_b200_uncompress_device(const uint8_t* d_in, size_t n, uint8_t* d_out, size_t out_cap,
                                  size_t* out_len, const uint64_t* d_frag_index, void* stream) {
    if (!out_len || (!d_in && n)) return SNAPPY_B200_BAD_ARGUMENT;
    Locked L;
    if (L.rc != SNAPPY_B200_OK) return L.rc;
    return uncompress_device_locked(*L.c, d_in, n, d_out, out_cap, out_len, (const u64*)d_frag_index,
                                    (cudaStream_t)stream);
}

int snappy_b200_validate_device(const uint8_t* d_in, size_t n, const uint64_t* d_frag_index, size_t* uncompressed_len,
                                void* stream) {
    if (!d_in && n) return SNAPPY_B200_BAD_ARGUMENT;
    Locked L;
    if (L.rc != SNAPPY_B200_OK) return L.rc;
    return validate_device_locked(*L.c, d_in, n, (const u64*)d_frag_index, uncompressed_len, (cudaStream_t)stream);
}

extern "C++" {
namespace {

// ---- pageable host buffers (what the reference API hands over: src/Snappy.jl:25,48 allocate plain Vector{UInt8}) ----
// A cudaMemcpyAsync from pageable memory is a synchronous, single-threaded staging copy inside the driver (~5 GB/s
// measured through this library's streamed paths: 236 ms per GiB round trip against 49 ms from pinned buffers).  So
// the streamed paths bounce pageable buffers through a small ring of pinned slots themselves:
//   up   : every piece is [host function: parallel memcpy user -> slot][copy slot -> device], enqueued UP FRONT on
//          two alternating streams (the memcpy of piece k+1 overlaps the DMA of piece k); being ordinary stream work
//          it keeps the rule of the streamed compress path that everything a persistent kernel waits for is queued
//          before that kernel;
//   down : [copy device -> slot] a few pieces ahead, then parallel memcpy slot -> user on the calling thread.
// One block of a big copy with non-temporal stores: the destination is either a pinned slot the DMA engine reads next
// or the caller's result buffer, neither is read by this core soon, and a cached store would first fetch the line it
// overwrites (a third of the copy's memory traffic).
#if defined(__x86_64__)
}  // namespace
}  // extern "C++"
#include <immintrin.h>
extern "C++" {
namespace {
__attribute__((target("avx2"))) void stream_copy_avx2(u8* d, const u8* s, size_t n) {
    while (n && (reinterpret_cast<uintptr_t>(d) & 31)) {
        *d++ = *s++;
        n--;
    }
    for (; n >= 128; n -= 128, s += 128, d += 128) {
        const __m256i a = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(s));
        const __m256i b = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(s + 32));
        const __m256i c = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(s + 64));
        const __m256i e = _mm256_loadu_si256(reinterpret_cast<const __m256i*>(s + 96));
        _mm256_stream_si256(reinterpret_cast<__m256i*>(d), a);
        _mm256_stream_si256(reinterpret_cast<__m256i*>(d + 32), b);
        _mm256_stream_si256(reinterpret_cast<__m256i*>(d + 64), c);
        _mm256_stream_si256(reinterpret_cast<__m256i*>(d + 96), e);
    }
    if (n) memcpy(d, s, n);
    _mm_sfence();
}
inline void block_copy(u8* d, const u8* s, size_t n) {
    static const bool avx2 = __builtin_cpu_supports("avx2") && !getenv("SNAPPY_B200_NO_STREAM_COPY");
    if (avx2) stream_copy_avx2(d, s, n);
    else memcpy(d, s, n);
}
#else
inline void block_copy(u8* d, const u8* s, size_t n) { memcpy(d, s, n); }
#endif

class CopyPool {  // a few persistent threads that split one memcpy among themselves (and the caller)
   public:
    static CopyPool& get() {
        // never destroyed: its threads sleep on the condition variable until the process ends (destroying a
        // condition variable that has waiters blocks, which would hang the process at exit)
        static CopyPool* p = new CopyPool();
        return *p;
    }
    void copy(void* dst, const void* src, size_t n) {
        if (n < (4u << 20) || th_.empty()) {
            memcpy(dst, src, n);
            return;
        }
        std::unique_lock<std::mutex> one(job_mu_);  // one job at a time: the memory system is the limit anyway
        {
            std::unique_lock<std::mutex> lk(mu_);
            dst_ = (u8*)dst;
            src_ = (const u8*)src;
            n_ = n;
            next_.store(0);
            pending_ = (int)th_.size();
            gen_++;
        }
        cv_.notify_all();
        work();
        std::unique_lock<std::mutex> lk(mu_);
        done_cv_.wait(lk, [&] { return pending_ == 0; });
    }

   private:
    static constexpr size_t kBlock = 1u << 20;
    CopyPool() {
        unsigned hw = std::thread::hardware_concurrency();
        int t = hw >= 16 ? 7 : (hw >= 8 ? 3 : (hw >= 4 ? 1 : 0));
        if (const char* e = getenv("SNAPPY_B200_COPY_THREADS")) t = atoi(e) - 1;
        for (int i = 0; i < t; i++) th_.emplace_back([this] { loop(); });
        for (auto& x : th_) x.detach();  // they sleep on the condition variable for the life of the process
    }
    void work() {
        for (;;) {
            const size_t o = next_.fetch_add(kBlock);
            if (o >= n_) break;
            block_copy(dst_ + o, src_ + o, n_ - o < kBlock ? n_ - o : kBlock);
        }
    }
    void loop() {
        unsigned long seen = 0;
        for (;;) {
            {
                std::unique_lock<std::mutex> lk(mu_);
                cv_.wait(lk, [&] { return gen_ != seen; });
                seen = gen_;
            }
            work();
            std::unique_lock<std::mutex> lk(mu_);
            if (--pending_ == 0) done_cv_.notify_all();
        }
    }
    std::vector<std::thread> th_;
    std::mutex mu_, job_mu_;
    std::condition_variable cv_, done_cv_;
    u8* dst_ = nullptr;
    const u8* src_ = nullptr;
    size_t n_ = 0;
    std::atomic<size_t> next_{0};
    int pending_ = 0;
    unsigned long gen_ = 0;
};

constexpr size_t kBounceSlot = 16u << 20;  // bytes per pinned slot
constexpr int kBounceUp = 4, kBounceDown = 4;

struct Bounce {  // per lane, created on the first pageable call
    u8* pin = nullptr;  // (kBounceUp + kBounceDown) slots
    cudaStream_t s_up[2] = {nullptr, nullptr};
    cudaEvent_t ev_up[2] = {nullptr, nullptr};
    cudaEvent_t ev_down[kBounceDown] = {};
};

bool is_pageable(const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return true;
    }
    return a.type == cudaMemoryTypeUnregistered;
}

struct UpJob {
    void* dst;
    const void* src;
    size_t n;
};
void CUDART_CB up_job_fn(void* p) {
    UpJob* j = (UpJob*)p;
    CopyPool::get().copy(j->dst, j->src, j->n);
}

int bounce_init(Context& c) {
    if (c.bounce) return SNAPPY_B200_OK;
    Bounce* b = new Bounce();
    cudaError_t e = cudaMallocHost((void**)&b->pin, (size_t)(kBounceUp + kBounceDown) * kBounceSlot);
    if (e != cudaSuccess) {
        delete b;
        return fail_cuda(e, "cudaMallocHost (bounce slots)");
    }
    c.bounce = b;
    for (int i = 0; i < 2; i++) {
        CU(cudaStreamCreateWithFlags(&b->s_up[i], cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&b->ev_up[i], cudaEventDisableTiming));
    }
    for (int i = 0; i < kBounceDown; i++) CU(cudaEventCreateWithFlags(&b->ev_down[i], cudaEventDisableTiming));
    return SNAPPY_B200_OK;
}

void bounce_destroy(Context& c) {
    Bounce* b = c.bounce;
    if (!b) return;
    for (int i = 0; i < 2; i++) {
        if (b->s_up[i]) cudaStreamDestroy(b->s_up[i]);
        if (b->ev_up[i]) cudaEventDestroy(b->ev_up[i]);
    }
    for (int i = 0; i < kBounceDown; i++)
        if (b->ev_down[i]) cudaEventDestroy(b->ev_down[i]);
    if (b->pin) cudaFreeHost(b->pin);
    delete b;
    c.bounce = nullptr;
}

// Host -> device.  Pinned source: one copy on c.s_h2d.  Pageable source: pieces through the pinned slots, all
// enqueued now (see above).  after(stream) is where the caller queues what must follow everything put so far
// (a ready count, an event): it first makes `stream` wait for the other upload stream.
struct Uploader {
    Context& c;
    bool pageable;
    std::vector<UpJob> jobs;  // reserved up front: the host functions hold pointers into it
    int piece = 0;
    cudaStream_t last = nullptr;
    Uploader(Context& ctx, bool pg, size_t total_bytes, int extra) : c(ctx), pageable(pg) {
        if (pageable) jobs.reserve(total_bytes / kBounceSlot + (size_t)extra + 8);
        last = c.s_h2d;
    }
    ~Uploader() {  // the host functions read `jobs`: nothing of ours may be pending when it goes away
        if (pageable && piece > 0 && c.bounce)
            for (cudaStream_t s : c.bounce->s_up)
                if (s) cudaStreamSynchronize(s);
    }
    int begin(cudaEvent_t after_this) {  // the upload streams start behind `after_this` (recorded by the caller)
        if (!pageable) return SNAPPY_B200_OK;
        for (int i = 0; i < 2; i++) CU(cudaStreamWaitEvent(c.bounce->s_up[i], after_this, 0));
        return SNAPPY_B200_OK;
    }
    int put(u8* d_dst, const u8* h_src, size_t len) {
        if (!pageable) {
            if (len) CU(cudaMemcpyAsync(d_dst, h_src, len, cudaMemcpyHostToDevice, c.s_h2d));
            last = c.s_h2d;
            return SNAPPY_B200_OK;
        }
        Bounce& b = *c.bounce;
        for (size_t o = 0; o < len; o += kBounceSlot) {
            const size_t l = len - o < kBounceSlot ? len - o : kBounceSlot;
            const int par = piece & 1;
            u8* slot = b.pin + (size_t)(piece % kBounceUp) * kBounceSlot;
            if (jobs.size() == jobs.capacity()) return fail_cuda(cudaErrorInvalidValue, "upload: piece list full");
            jobs.push_back(UpJob{slot, h_src + o, l});
            CU(cudaLaunchHostFunc(b.s_up[par], up_job_fn, &jobs.back()));
            CU(cudaMemcpyAsync(d_dst + o, slot, l, cudaMemcpyHostToDevice, b.s_up[par]));
            CU(cudaEventRecord(b.ev_up[par], b.s_up[par]));
            last = b.s_up[par];
            piece++;
        }
        return SNAPPY_B200_OK;
    }
    int after(cudaStream_t* st) {
        *st = last;
        if (pageable && piece > 0) {
            Bounce& b = *c.bounce;
            const int par = last == b.s_up[0] ? 0 : 1;
            CU(cudaStreamWaitEvent(last, b.ev_up[par ^ 1], 0));
        }
        return SNAPPY_B200_OK;
    }
    int mark() {  // what the caller queued behind after() is now the latest thing on that stream
        if (pageable && piece > 0) {
            Bounce& b = *c.bounce;
            const int par = last == b.s_up[0] ? 0 : 1;
            CU(cudaEventRecord(b.ev_up[par], last));
        }
        return SNAPPY_B200_OK;
    }
    int sync() {
        if (pageable)
            for (int i = 0; i < 2; i++) CU(cudaStreamSynchronize(c.bounce->s_up[i]));
        return SNAPPY_B200_OK;
    }
};

// Device -> host for data that is ready on the device (the caller waited for it).
struct Downloader {
    Context& c;
    bool pageable;
    struct Piece {
        u8* h_dst;
        size_t len;
        int slot;
    };
    Piece q[kBounceDown];
    int head = 0, count = 0, next_slot = 0;
    Downloader(Context& ctx, bool pg) : c(ctx), pageable(pg) {}
    int drain_one() {
        Bounce& b = *c.bounce;
        const Piece p = q[head];
        head = (head + 1) % kBounceDown;
        count--;
        CU(cudaEventSynchronize(b.ev_down[p.slot]));
        CopyPool::get().copy(p.h_dst, b.pin + (size_t)(kBounceUp + p.slot) * kBounceSlot, p.len);
        return SNAPPY_B200_OK;
    }
    int push(u8* h_dst, const u8* d_src, size_t len) {
        if (!pageable) {
            if (len) CU(cudaMemcpyAsync(h_dst, d_src, len, cudaMemcpyDeviceToHost, c.s_d2h));
            return SNAPPY_B200_OK;
        }
        Bounce& b = *c.bounce;
        for (size_t o = 0; o < len; o += kBounceSlot) {
            const size_t l = len - o < kBounceSlot ? len - o : kBounceSlot;
            if (count == kBounceDown) {
                int rc = drain_one();
                if (rc != SNAPPY_B200_OK) return rc;
            }
            const int slot = next_slot;
            next_slot = (next_slot + 1) % kBounceDown;
            CU(cudaMemcpyAsync(b.pin + (size_t)(kBounceUp + slot) * kBounceSlot, d_src + o, l, cudaMemcpyDeviceToHost, c.s_d2h));
            CU(cudaEventRecord(b.ev_down[slot], c.s_d2h));
            q[(head + count) % kBounceDown] = Piece{h_dst + o, l, slot};
            count++;
        }
        return SNAPPY_B200_OK;
    }
    int finish() {
        while (pageable && count) {
            int rc = drain_one();
            if (rc != SNAPPY_B200_OK) return rc;
        }
        return SNAPPY_B200_OK;
    }
};

}  // namespace
}  // extern "C++"

// The streamed host paths enqueue copies from / into the CALLER's buffers on several streams.  Whatever way such a
// function returns, nothing may still be in flight: an early error return drains the pipeline first.
struct PipeGuard {
    Context& c;
    bool drained = false;
    ~PipeGuard() {
        if (drained) return;
        for (cudaStream_t st : {c.s_h2d, c.s_comp, c.side, c.s_pack, c.s_d2h})
            if (st) cudaStreamSynchronize(st);
        if (c.bounce)
            for (cudaStream_t st : c.bounce->s_up)
                if (st) cudaStreamSynchronize(st);
    }
};

// Host-buffer compress, streamed (SURVEY.md 8(f)1): ONE launch of the persistent compress kernels
// covers the whole input.  The input goes up in chunks on a copy stream, each followed by a 4-byte
// copy that raises the device-side `ready` count the kernels wait on before they touch a fragment;
// finished fragments are counted per output chunk, and a small scan kernel per chunk waits for its
// count, after which the chunk is compacted behind the stream so far and its bytes go down on a
// third stream while the rest still compresses.  Only the running stream length (8 bytes per chunk)
// is read by the host.
int compress_host_streamed(Context& c, const u8* in, size_t n, u8* out, size_t* out_len) {
    PipeGuard guard{c};
    const size_t cf = 1024;  // fragments per chunk (64 MiB up, ~30 MB down)
    const size_t need = snappy_b200_max_compressed_length(n);
    const u32 nfrag = (u32)((n + kBlockSize - 1) / kBlockSize);
    const int nchunks = (int)((nfrag + cf - 1) / cf);
    CU(c.stage_in.ensure(n + 16));
    CU(c.stage_out.ensure(need + 16));
    CU(c.scratch.ensure((size_t)nfrag * kSlotStride));
    CU(c.frag_sizes.ensure((size_t)nfrag * sizeof(u32)));
    CU(c.frag_offsets.ensure(((size_t)nfrag + 1) * sizeof(u64) + 8));
    CU(c.flags.ensure(64 + (size_t)kMaxPipeChunks * 4));
    CU(c.tail.ensure(kTailSlot));
    u8* d_in = (u8*)c.stage_in.p;
    u8* d_out = (u8*)c.stage_out.p;
    u8* scratch = (u8*)c.scratch.p;
    u32* sizes = (u32*)c.frag_sizes.p;
    u64* offs = (u64*)c.frag_offsets.p;
    u64* running = offs + nfrag + 1;            // device: bytes in the stream so far
    u32* d_ready = (u32*)c.flags.p;             // device: fragments resident
    u32* d_done = (u32*)((u8*)c.flags.p + 64);  // device: fragments finished, per chunk
    u64* h_tot = (u64*)((u8*)c.pinned + 2048);  // host: stream length after each chunk
    u32* h_ready = (u32*)((u8*)c.pinned + 2048 + kMaxPipeChunks * 8);
    const u32 shift = table_shift(n);
    u8* hdr = (u8*)c.pinned + 64;
    const int k = encode_varint((u32)n, hdr);   // src/Snappy.jl:26
    u64* h_k = (u64*)((u8*)c.pinned + 96);
    *h_k = (u64)k;
    // plain (pageable) caller buffers go through the pinned bounce slots, pinned ones straight
    const bool pg_in = c.opt.pin_host && is_pageable(in), pg_out = c.opt.pin_host && is_pageable(out);
    if (pg_in || pg_out) {
        int rb = bounce_init(c);
        if (rb != SNAPPY_B200_OK) return rb;
    }
    Uploader up(c, pg_in, n, nchunks);
    Downloader down(c, pg_out);
    CU(cudaMemsetAsync(c.flags.p, 0, 64 + (size_t)nchunks * 4, c.s_comp));
    CU(cudaMemcpyAsync(d_out, hdr, (size_t)k, cudaMemcpyHostToDevice, c.s_comp));
    CU(cudaMemcpyAsync(running, h_k, 8, cudaMemcpyHostToDevice, c.s_comp));
    CU(cudaEventRecord(c.ev_in[0], c.s_comp));
    // The copies are enqueued BEFORE the kernels that wait for them: streams can share a hardware queue
    // (CUDA_DEVICE_MAX_CONNECTIONS), and a copy queued behind a kernel that waits for it would never run.
    // input: chunk, then the count of resident fragments
    CU(cudaStreamWaitEvent(c.s_h2d, c.ev_in[0], 0));
    {   // padded copy of the last fragment, straight from the host buffer and first of all: nothing on this
        // stream may need an SM (a device-to-device copy or a memset can be a kernel) once the persistent
        // kernels sit on every SM waiting for the counts below
        const u64 tail_start = (u64)(nfrag - 1) * kBlockSize;
        const size_t tail_len = n - tail_start;
        CU(cudaMemcpyAsync(c.tail.p, in + tail_start, tail_len, cudaMemcpyHostToDevice, c.s_h2d));
        CU(cudaMemcpyAsync((u8*)c.tail.p + tail_len, c.pinned_zero, kTailPad, cudaMemcpyHostToDevice, c.s_h2d));
        CU(cudaEventRecord(c.ev_in[1], c.s_h2d));
    }
    {
        int ru = up.begin(c.ev_in[1]);  // behind the tail copy (which is behind the setup on s_comp)
        if (ru != SNAPPY_B200_OK) return ru;
    }
    for (int i = 0; i < nchunks; i++) {
        const size_t off = (size_t)i * cf * kBlockSize;
        const size_t len = (n - off < cf * kBlockSize) ? (n - off) : cf * kBlockSize;
        int ru = up.put(d_in + off, in + off, len);
        if (ru != SNAPPY_B200_OK) return ru;
        h_ready[i] = (i == nchunks - 1) ? nfrag : (u32)((size_t)(i + 1) * cf);
        cudaStream_t us = nullptr;
        ru = up.after(&us);  // the count follows every byte put so far, and the counts follow each other
        if (ru != SNAPPY_B200_OK) return ru;
        CU(cudaMemcpyAsync(d_ready, h_ready + i, 4, cudaMemcpyHostToDevice, us));
        ru = up.mark();
        if (ru != SNAPPY_B200_OK) return ru;
    }
    // the persistent kernels
    int launches = 0;
    Gate gate;
    gate.ready = d_ready;
    gate.done = d_done;
    gate.div = (u32)cf;
    if (c.opt.timing) CU(cudaEventRecord(c.ev[0], c.s_comp));
    int rc = launch_chain_kernels(c, d_in, n, shift, scratch, sizes, c.s_comp, &launches, nullptr, 0, 0, &gate);
    if (rc != SNAPPY_B200_OK) return rc;
    if (c.opt.timing) {
        CU(cudaEventRecord(c.ev[1], c.s_comp));
        c.ev_pending[0] = true;
    }
    // output: per chunk wait + scan, compaction, stream length
    CU(cudaStreamWaitEvent(c.s_pack, c.ev_in[0], 0));
    for (int i = 0; i < nchunks; i++) {
        const size_t f0 = (size_t)i * cf;
        const u32 nf = (u32)((nfrag - f0 < cf) ? (nfrag - f0) : cf);
        k_scan_chunk<<<1, 256, 0, c.s_pack>>>(sizes + f0, nf, offs + f0, running, d_done + i, nf, h_tot + i);
        k_compact<<<nf, 256, 0, c.s_pack>>>(scratch + f0 * kSlotStride, sizes + f0, offs + f0, d_out);
        launches += 2;
        CU(cudaEventRecord(c.ev_done[i], c.s_pack));
    }
    CU(cudaGetLastError());
    u64 prev = 0;
    for (int i = 0; i < nchunks; i++) {
        CU(cudaEventSynchronize(c.ev_done[i]));
        const u64 end = ((volatile u64*)h_tot)[i];
        int rd = down.push(out + prev, d_out + prev, (size_t)(end - prev));
        if (rd != SNAPPY_B200_OK) return rd;
        prev = end;
    }
    {
        int rd = down.finish();
        if (rd != SNAPPY_B200_OK) return rd;
    }
    CU(cudaStreamSynchronize(c.s_d2h));
    CU(cudaStreamSynchronize(c.s_comp));
    CU(cudaStreamSynchronize(c.s_h2d));
    {
        int ru = up.sync();
        if (ru != SNAPPY_B200_OK) return ru;
    }
    harvest_timing(c, 0);
    c.last_launches[0] = launches;
    *out_len = (size_t)prev;
    guard.drained = true;
    return SNAPPY_B200_OK;
}

// Host-buffer compress, pipelined (SURVEY.md 8(f)1): the input goes up in chunks of
// kPipeChunkFrags fragments on a copy stream, each chunk is compressed + compacted behind the
// previous one's bytes as soon as it has landed, and its bytes go back down on a third stream
// while the next chunk compresses.  Only the chunk totals (8 bytes each) are read by the host.
int compress_host_pipelined(Context& c, const u8* in, size_t n, u8* out, size_t* out_len) {
    PipeGuard guard{c};
    const size_t kPipeChunkFrags = (size_t)c.opt.pipe_chunk_frags;
    const size_t need = snappy_b200_max_compressed_length(n);
    const u32 nfrag = (u32)((n + kBlockSize - 1) / kBlockSize);
    const int nchunks = (int)((nfrag + kPipeChunkFrags - 1) / kPipeChunkFrags);
    CU(c.stage_in.ensure(n + 16));
    CU(c.stage_out.ensure(need + 16));
    CU(c.scratch.ensure((size_t)nfrag * kSlotStride));
    CU(c.frag_sizes.ensure((size_t)nfrag * sizeof(u32)));
    CU(c.frag_offsets.ensure(((size_t)nfrag + 1) * sizeof(u64) + 8));
    u8* d_in = (u8*)c.stage_in.p;
    u8* d_out = (u8*)c.stage_out.p;
    u8* scratch = (u8*)c.scratch.p;
    u32* sizes = (u32*)c.frag_sizes.p;
    u64* offs = (u64*)c.frag_offsets.p;
    u64* running = offs + nfrag + 1;           // device: bytes in the stream so far
    u64* h_tot = (u64*)((u8*)c.pinned + 2048);  // host: stream length after each chunk
    const u32 shift = table_shift(n);
    u8* hdr = (u8*)c.pinned + 64;
    const int k = encode_varint((u32)n, hdr);   // src/Snappy.jl:26
    u64* h_k = (u64*)((u8*)c.pinned + 96);
    *h_k = (u64)k;
    CU(cudaMemcpyAsync(d_out, hdr, (size_t)k, cudaMemcpyHostToDevice, c.s_comp));
    CU(cudaMemcpyAsync(running, h_k, 8, cudaMemcpyHostToDevice, c.s_comp));
    int launches = 0;
    for (int i = 0; i < nchunks; i++) {
        const size_t off = (size_t)i * kPipeChunkFrags * kBlockSize;
        const size_t len = (n - off < kPipeChunkFrags * kBlockSize) ? (n - off) : kPipeChunkFrags * kBlockSize;
        CU(cudaMemcpyAsync(d_in + off, in + off, len, cudaMemcpyHostToDevice, c.s_h2d));
        CU(cudaEventRecord(c.ev_in[i], c.s_h2d));
    }
    for (int i = 0; i < nchunks; i++) {
        const size_t f0 = (size_t)i * kPipeChunkFrags;
        const size_t off = f0 * kBlockSize;
        const size_t len = (n - off < kPipeChunkFrags * kBlockSize) ? (n - off) : kPipeChunkFrags * kBlockSize;
        const u32 nf = (u32)((len + kBlockSize - 1) / kBlockSize);
        CU(cudaStreamWaitEvent(c.s_comp, c.ev_in[i], 0));
        int rc = launch_chain_kernels(c, d_in + off, len, shift, scratch + f0 * kSlotStride, sizes + f0,
                                      c.s_comp, &launches);
        if (rc != SNAPPY_B200_OK) return rc;
        k_scan_sizes<<<1, 1024, 0, c.s_comp>>>(sizes + f0, nf, 0, offs + f0, running);
        k_compact<<<nf, 256, 0, c.s_comp>>>(scratch + f0 * kSlotStride, sizes + f0, offs + f0, d_out);
        launches += 2;
        CU(cudaMemcpyAsync(h_tot + i, running, 8, cudaMemcpyDeviceToHost, c.s_comp));
        CU(cudaEventRecord(c.ev_done[i], c.s_comp));
    }
    CU(cudaGetLastError());
    u64 prev = 0;
    for (int i = 0; i < nchunks; i++) {
        CU(cudaEventSynchronize(c.ev_done[i]));
        const u64 end = ((volatile u64*)h_tot)[i];
        CU(cudaMemcpyAsync(out + prev, d_out + prev, (size_t)(end - prev), cudaMemcpyDeviceToHost, c.s_d2h));
        prev = end;
    }
    CU(cudaStreamSynchronize(c.s_d2h));
    c.last_launches[0] = launches;
    *out_len = (size_t)prev;
    return SNAPPY_B200_OK;
}

int snappy_b200_compress(const uint8_t* in, size_t n, uint8_t* out, size_t* out_len) {
    if (!out_len || (!in && n) || !out) return SNAPPY_B200_BAD_ARGUMENT;
    if (n > 0xffffffffull) return SNAPPY_B200_INPUT_TOO_LARGE;  // src/Snappy.jl:21
    const size_t need = snappy_b200_max_compressed_length(n);
    if (*out_len < need) return SNAPPY_B200_BUFFER_TOO_SMALL;
    Locked L;
    if (L.rc != SNAPPY_B200_OK) return L.rc;
    Context& c = *L.c;
    if (c.opt.compress_variant == 0 && c.opt.host_pipeline == 1 && c.opt.window && !c.opt.wide &&
        n > (size_t)2048 * kBlockSize)
        return compress_host_streamed(c, in, n, out, out_len);
    if (c.opt.compress_variant == 0 && c.opt.host_pipeline && n > (size_t)c.opt.pipe_chunk_frags * kBlockSize)
        return compress_host_pipelined(c, in, n, out, out_len);
    CU(c.stage_in.ensure(n + 16));
    CU(c.stage_out.ensure(need + 16));
    cudaStream_t st = c.s_comp;
    if (n) CU(cudaMemcpyAsync(c.stage_in.p, in, n, cudaMemcpyHostToDevice, st));
    size_t clen = 0;
    int rc = compress_device_locked(c, (const u8*)c.stage_in.p, n, (u8*)c.stage_out.p, need, &clen,
                                    nullptr, st);
    if (rc != SNAPPY_B200_OK) return rc;
    CU(cudaMemcpyAsync(out, c.stage_out.p, clen, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    *out_len = clen;
    return SNAPPY_B200_OK;
}

// Host-buffer uncompress, streamed (SURVEY.md 8(f)1+2): the stream goes up in 16 chunks; it is parsed
// in 4 segments, each as soon as its bytes (and one chunk of slack for the elements that run past
// its end) have landed; the fragments a segment completes are decoded and sent down while the next
// segment is still on its way up.  Returns -1 when the stream needs the whole-stream paths (not
// fragment-clean, anomalies): the caller then runs them on the resident copy.
int uncompress_host_streamed(Context& c, const u8* in, size_t n, size_t hdr, u32 claimed, u8* out) {
    PipeGuard guard{c};
    const int kChunks = 16;
    const int kSegs = (c.opt.uncompress_segments == 2 || c.opt.uncompress_segments == 8) ? c.opt.uncompress_segments : 4;
    const u32 nfrag = frag_count(claimed);
    cudaStream_t st = c.s_comp;
    u8* d_in = (u8*)c.stage_in.p;
    u8* d_out = (u8*)c.stage_out.p;
    CU(c.index.ensure(((size_t)nfrag + 1) * 8));
    CU(cudaMemsetAsync(c.index.p, 0xff, ((size_t)nfrag + 1) * 8, st));
    CU(cudaMemsetAsync(c.result.p, 0, sizeof(DecodeResult), st));
    if (c.opt.timing) CU(cudaEventRecord(c.ev[2], st));
    size_t cb[kChunks + 1];
    const size_t csz = ((n + kChunks - 1) / kChunks + 4095) & ~(size_t)4095;
    for (int i = 0; i <= kChunks; i++) cb[i] = ((size_t)i * csz < n) ? (size_t)i * csz : n;
    const bool pg_in = c.opt.pin_host && is_pageable(in), pg_out = c.opt.pin_host && is_pageable(out);
    if (pg_in || pg_out) {
        int rb = bounce_init(c);
        if (rb != SNAPPY_B200_OK) return rb;
    }
    Uploader up(c, pg_in, n, kChunks);
    Downloader down(c, pg_out);
    std::vector<Context::DownRange> ranges;
    struct DeferGuard {
        Context& c;
        ~DeferGuard() { c.defer_down = nullptr; }
    } defer_guard{c};
    if (pg_out) c.defer_down = &ranges;
    size_t drained = 0;
    auto drain_ranges = [&](size_t upto) -> int {  // finished output ranges -> the caller's pageable buffer
        for (; drained < upto && drained < ranges.size(); drained++) {
            CU(cudaEventSynchronize(c.ev_done[ranges[drained].ev]));
            int rd = down.push(out + ranges[drained].off, d_out + ranges[drained].off, ranges[drained].len);
            if (rd != SNAPPY_B200_OK) return rd;
        }
        return SNAPPY_B200_OK;
    };
    for (int i = 0; i < kChunks; i++) {
        if (cb[i + 1] > cb[i]) {
            int ru = up.put(d_in + cb[i], in + cb[i], cb[i + 1] - cb[i]);
            if (ru != SNAPPY_B200_OK) return ru;
        }
        cudaStream_t us = nullptr;
        int ru = up.after(&us);
        if (ru != SNAPPY_B200_OK) return ru;
        CU(cudaEventRecord(c.ev_in[i], us));
    }
    const bool dbg = getenv("SNAPPY_B200_DEBUG") != nullptr;
    const auto t0 = std::chrono::steady_clock::now();
    auto ms = [&]() { return std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count(); };
    u64 entry = hdr, out_base = 0;
    u64* h_exit = (u64*)((u8*)c.pinned + 1536);  // one slot per segment (read by async copies)
    u32 f_done = 0;
    int ri = 0, rc = 0;
    for (int j = 0; j < kSegs && rc == 0; j++) {
        const int last_chunk = (j + 1) * (kChunks / kSegs) - 1;            // the segment ends with this chunk
        const int need_chunk = last_chunk + 1 < kChunks ? last_chunk + 1 : kChunks - 1;  // + slack
        const size_t E = cb[last_chunk + 1];
        CU(cudaStreamWaitEvent(st, c.ev_in[need_chunk], 0));
        if (E <= entry) {  // a long literal swallowed the segment
            if (j == kSegs - 1) rc = -1;
            continue;
        }
        u64 ex = 0, produced = 0;
        if (dbg) fprintf(stderr, "[snappy_b200] t=%.2f ms: segment %d parse enqueue\n", ms(), j);
        rc = build_index_segment(c, d_in, n, (size_t)entry, E, out_base, nfrag, st, &ex, &produced);
        if (dbg) fprintf(stderr, "[snappy_b200] t=%.2f ms: segment %d parsed rc=%d\n", ms(), j, rc);
        if (rc != 0) break;
        out_base += produced;
        entry = ex;
        if (out_base > claimed) {
            rc = -1;
            break;
        }
        u32 f_hi = (j == kSegs - 1) ? nfrag : (u32)(out_base / kBlockSize);
        if (j < kSegs - 1 && f_hi > f_done && out_base % kBlockSize == 0) {
            // the boundary element is the next segment's first: its position is this segment's exit
            h_exit[j] = ex;
            CU(cudaMemcpyAsync((u64*)c.index.p + f_hi, h_exit + j, 8, cudaMemcpyHostToDevice, st));
        }
        if (f_hi > f_done) {
            // the decoder runs on its own stream, next to the parse of the next segment: one launch per
            // segment (a launch costs one fragment's latency, ~2.6 ms, however few fragments it has)
            CU(cudaEventRecord(c.ev_fork, st));
            CU(cudaStreamWaitEvent(c.s_pack, c.ev_fork, 0));
            int r2 = decode_launch(c, d_in, n, hdr, d_out, claimed, (const u64*)c.index.p, c.s_pack, f_done, f_hi, out,
                                   &ri, f_hi - f_done);
            if (r2 != SNAPPY_B200_OK) return r2;
            f_done = f_hi;
            if (pg_out && ranges.size() > 1) {  // the range before this one has had a segment's time to finish
                r2 = drain_ranges(ranges.size() - 1);
                if (r2 != SNAPPY_B200_OK) return r2;
            }
        }
    }
    if (rc > 0) return rc;
    if (rc == 0 && out_base != claimed) rc = -1;
    if (pg_out && rc == 0) {
        int r2 = drain_ranges(ranges.size());
        if (r2 == SNAPPY_B200_OK) r2 = down.finish();
        if (r2 != SNAPPY_B200_OK) return r2;
    }
    if (dbg) {
        CU(cudaStreamSynchronize(st));
        CU(cudaStreamSynchronize(c.s_pack));
        fprintf(stderr, "[snappy_b200] t=%.2f ms: decode done\n", ms());
    }
    const int rf = decode_finish(c, st, true);
    if (dbg) fprintf(stderr, "[snappy_b200] t=%.2f ms: copies done\n", ms());
    CU(cudaStreamSynchronize(c.s_h2d));
    {
        int ru = up.sync();
        if (ru != SNAPPY_B200_OK) return ru;
    }
    if (rf > 0) return rf;
    return (rc == 0 && rf == 0) ? SNAPPY_B200_OK : -1;
}

int snappy_b200_uncompress(const uint8_t* in, size_t n, uint8_t* out, size_t* out_len) {
    if (!out_len || (!in && n)) return SNAPPY_B200_BAD_ARGUMENT;
    u32 claimed = 0;
    size_t hdr = 0;
    int rc = parse_varint(in, n, &claimed, &hdr);  // src/Snappy.jl:47
    if (rc != SNAPPY_B200_OK) return rc;
    if (*out_len < claimed) return SNAPPY_B200_BUFFER_TOO_SMALL;
    Locked L;
    if (L.rc != SNAPPY_B200_OK) return L.rc;
    Context& c = *L.c;
    CU(c.stage_in.ensure(n + 16));
    CU(c.stage_out.ensure((size_t)claimed + 16));
    cudaStream_t st = c.s_comp;
    size_t olen = 0;
    bool copied = false;
    bool resident = false;
    if (c.opt.host_pipeline == 1 && c.opt.decode_variant != 1 && n > ((size_t)64 << 20) && claimed > 0) {
        c.last_launches[1] = 0;
        rc = uncompress_host_streamed(c, in, n, hdr, claimed, out);
        if (rc == SNAPPY_B200_OK) {
            *out_len = claimed;
            return SNAPPY_B200_OK;
        }
        if (rc > 0) return rc;
        resident = true;  // the whole-stream paths decide (the stream is on the device by now)
    }
    if (!resident) CU(cudaMemcpyAsync(c.stage_in.p, in, n, cudaMemcpyHostToDevice, st));
    rc = uncompress_device_locked(c, (const u8*)c.stage_in.p, n, (u8*)c.stage_out.p, (size_t)claimed,
                                  &olen, nullptr, st, out, &copied);
    if (rc != SNAPPY_B200_OK) return rc;
    if (olen && !copied) CU(cudaMemcpyAsync(out, c.stage_out.p, olen, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    *out_len = olen;
    return SNAPPY_B200_OK;
}

// Host-buffer validation: the stream goes up as the host uncompress sends it (pinned: one copy; pageable: through the
// bounce slots), then the device chain judges it.  No output buffer on either side.
int snappy_b200_validate_compressed_buffer(const uint8_t* in, size_t n) {
    if (!in && n) return SNAPPY_B200_BAD_ARGUMENT;
    u32 claimed = 0;
    size_t hdr = 0;
    int rc = parse_varint(in, n, &claimed, &hdr);  // src/Snappy.jl:47
    if (rc != SNAPPY_B200_OK) return rc;
    Locked L;
    if (L.rc != SNAPPY_B200_OK) return L.rc;
    Context& c = *L.c;
    CU(c.stage_in.ensure(n + 16));
    const bool pg_in = c.opt.pin_host && is_pageable(in);
    if (pg_in) {
        int rb = bounce_init(c);
        if (rb != SNAPPY_B200_OK) return rb;
    }
    {
        PipeGuard guard{c};
        Uploader up(c, pg_in, n, 0);
        int ru = up.put((u8*)c.stage_in.p, in, n);
        if (ru == SNAPPY_B200_OK) ru = up.sync();
        if (ru != SNAPPY_B200_OK) return ru;
        CU(cudaStreamSynchronize(c.s_h2d));
        guard.drained = true;
    }
    size_t claimed_len = 0;
    return validate_device_locked(c, (const u8*)c.stage_in.p, n, nullptr, &claimed_len, c.s_comp);
}

int snappy_b200_compress_shard_device(const uint8_t* d_shard, size_t shard_len, uint64_t total_len,
                                      uint8_t* d_out, size_t out_cap, size_t* out_len,
                                      uint32_t* d_frag_sizes, void* stream) {
    if (!out_len || (!d_shard && shard_len) || !d_out) return SNAPPY_B200_BAD_ARGUMENT;
    if (total_len > 0xffffffffull) return SNAPPY_B200_INPUT_TOO_LARGE;
    if (shard_len > total_len) return SNAPPY_B200_BAD_ARGUMENT;
    if (out_cap < snappy_b200_max_compressed_length(shard_len)) return SNAPPY_B200_BUFFER_TOO_SMALL;
    Locked L;
    if (L.rc != SNAPPY_B200_OK) return L.rc;
    u64 total = 0;
    int rc = compress_shard_locked(*L.c, d_shard, shard_len, total_len, d_out, 0, &total, nullptr,
                                   d_frag_sizes, (cudaStream_t)stream);
    if (rc == SNAPPY_B200_OK) *out_len = (size_t)total;
    return rc;
}

int snappy_b200_uncompress_shard_device(const uint8_t* d_in, const uint64_t* d_frag_offsets,
                                        size_t nfrag, uint8_t* d_out, size_t out_len, void* stream) {
    if (!d_in || !d_frag_offsets || (!d_out && out_len)) return SNAPPY_B200_BAD_ARGUMENT;
    if (nfrag != (out_len + kBlockSize - 1) / kBlockSize) return SNAPPY_B200_BAD_ARGUMENT;
    if (nfrag == 0) return SNAPPY_B200_OK;
    Locked L;
    if (L.rc != SNAPPY_B200_OK) return L.rc;
    Context& c = *L.c;
    cudaStream_t st = (cudaStream_t)stream;
    c.last_launches[1] = 0;
    // the shard's own first/last offsets bound its element bytes
    u64* h = (u64*)((u8*)c.pinned + 512);
    CU(cudaMemcpyAsync(h, d_frag_offsets, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaMemcpyAsync(h + 1, d_frag_offsets + nfrag, 8, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    DecodeResult* res = (DecodeResult*)c.result.p;
    CU(cudaMemsetAsync(res, 0, sizeof(DecodeResult), st));
    if (c.opt.timing) CU(cudaEventRecord(c.ev[2], st));
    const u32 grid = ((u32)nfrag + kDecodeWarpsPerCta - 1) / kDecodeWarpsPerCta;
    k_decode_fragments<8><<<grid, kDecodeWarpsPerCta * 32, 0, st>>>(d_in, d_frag_offsets, (u32)nfrag, 0u,
                                                                 (u32)nfrag, h[0], h[1], d_out, (u64)out_len, res);
    if (c.opt.timing) {
        CU(cudaEventRecord(c.ev[3], st));
        c.ev_pending[1] = true;
    }
    c.last_launches[1] = 1;
    CU(cudaGetLastError());
    DecodeResult* hr = (DecodeResult*)((u8*)c.pinned + 128);
    CU(cudaMemcpyAsync(hr, res, sizeof(DecodeResult), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    harvest_timing(c, 1);
    // a shard has no stream-order context for exact error attribution
    return hr->fallback ? SNAPPY_B200_INVALID_INPUT : SNAPPY_B200_OK;
}

int snappy_b200_compress_shards_device(const uint8_t* const* d_shards, const size_t* shard_lens,
                                       const uint64_t* total_lens, size_t count, uint8_t* const* d_outs,
                                       const size_t* out_caps, size_t* out_lens,
                                       uint32_t* const* d_frag_sizes, void* stream) {
    if (count == 0) return SNAPPY_B200_OK;
    if (!d_shards || !shard_lens || !total_lens || !d_outs || !out_caps || !out_lens || count > 4096)
        return SNAPPY_B200_BAD_ARGUMENT;
    std::vector<ShardDesc> descs;
    std::vector<size_t> owner;  // descs[i] describes shard owner[i] (empty shards have no desc)
    u64 nfrag_total = 0;
    for (size_t k = 0; k < count; k++) {
        out_lens[k] = 0;
        if (total_lens[k] > 0xffffffffull) return SNAPPY_B200_INPUT_TOO_LARGE;
        if (shard_lens[k] > total_lens[k] || (!d_shards[k] && shard_lens[k]) || !d_outs[k])
            return SNAPPY_B200_BAD_ARGUMENT;
        if (out_caps[k] < snappy_b200_max_compressed_length(shard_lens[k])) return SNAPPY_B200_BUFFER_TOO_SMALL;
        const u32 nf = (u32)((shard_lens[k] + kBlockSize - 1) / kBlockSize);
        if (nf == 0) continue;
        ShardDesc d;
        d.ptr = d_shards[k];
        d.tail = nullptr;
        d.len = shard_lens[k];
        d.frag_begin = (u32)nfrag_total;
        d.nfrag = nf;
        d.shift = table_shift(total_lens[k]);
        d.pad_ = 0;
        descs.push_back(d);
        owner.push_back(k);
        nfrag_total += nf;
    }
    if (descs.empty()) return SNAPPY_B200_OK;
    if (nfrag_total > 0x7fffffffull) return SNAPPY_B200_BAD_ARGUMENT;
    Locked L;
    if (L.rc != SNAPPY_B200_OK) return L.rc;
    Context& c = *L.c;
    cudaStream_t st = (cudaStream_t)stream;
    const u32 nd = (u32)descs.size();
    CU(c.tail.ensure(kTailSlot * nd));
    CU(c.scratch.ensure((size_t)nfrag_total * kSlotStride));
    CU(c.frag_sizes.ensure((size_t)nfrag_total * sizeof(u32)));
    CU(c.frag_offsets.ensure(((size_t)nfrag_total + nd + 1) * sizeof(u64)));
    CU(c.descs.ensure(sizeof(ShardDesc) * nd));
    for (u32 i = 0; i < nd; i++) {
        descs[i].tail = (const u8*)c.tail.p + (size_t)i * kTailSlot;
        int rc = stage_tail(c, descs[i].ptr, (size_t)descs[i].len, i, st);
        if (rc != SNAPPY_B200_OK) return rc;
    }
    CU(cudaMemcpyAsync(c.descs.p, descs.data(), sizeof(ShardDesc) * nd, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));  // descs.data() is pageable host memory
    u8* scratch = (u8*)c.scratch.p;
    u32* sizes = (u32*)c.frag_sizes.p;
    u64* offs = (u64*)c.frag_offsets.p;
    int launches = 0;
    if (c.opt.timing) CU(cudaEventRecord(c.ev[0], st));
    int rc = launch_chain_kernels(c, nullptr, 0, 0, scratch, sizes, st, &launches, (const ShardDesc*)c.descs.p,
                                  nd, (u32)nfrag_total);
    if (rc != SNAPPY_B200_OK) return rc;
    if (c.opt.timing) {
        CU(cudaEventRecord(c.ev[1], st));
        c.ev_pending[0] = true;
    }
    u64* h = (u64*)((u8*)c.pinned + kPinnedShardLens);  // count <= 4096 checked on entry
    for (u32 i = 0; i < nd; i++) {
        const u32 fb = descs[i].frag_begin, nf = descs[i].nfrag;
        u64* o = offs + fb + i;  // nf + 1 entries per shard
        k_scan_sizes<<<1, 1024, 0, st>>>(sizes + fb, nf, 0, o);
        k_compact<<<nf, 256, 0, st>>>(scratch + (size_t)fb * kSlotStride, sizes + fb, o, d_outs[owner[i]]);
        launches += 2;
        CU(cudaMemcpyAsync(h + i, o + nf, 8, cudaMemcpyDeviceToHost, st));
        if (d_frag_sizes && d_frag_sizes[owner[i]])
            CU(cudaMemcpyAsync(d_frag_sizes[owner[i]], sizes + fb, (size_t)nf * 4, cudaMemcpyDeviceToDevice, st));
    }
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(st));
    harvest_timing(c, 0);
    c.last_launches[0] = launches;
    for (u32 i = 0; i < nd; i++) out_lens[owner[i]] = (size_t)h[i];
    return SNAPPY_B200_OK;
}

int snappy_b200_uncompress_shards_device(const uint8_t* const* d_ins, const uint64_t* const* d_frag_offsets,
                                         const size_t* out_lens, size_t count, uint8_t* const* d_outs,
                                         void* stream) {
    if (count == 0) return SNAPPY_B200_OK;
    if (!d_ins || !d_frag_offsets || !out_lens || !d_outs || count > 4096) return SNAPPY_B200_BAD_ARGUMENT;
    std::vector<DecodeDesc> descs;
    u64 nfrag_total = 0;
    for (size_t k = 0; k < count; k++) {
        const u32 nf = (u32)((out_lens[k] + kBlockSize - 1) / kBlockSize);
        if (nf == 0) continue;
        if (!d_ins[k] || !d_frag_offsets[k] || !d_outs[k]) return SNAPPY_B200_BAD_ARGUMENT;
        DecodeDesc d;
        d.in = d_ins[k];
        d.frag_off = d_frag_offsets[k];
        d.out = d_outs[k];
        d.out_len = out_lens[k];
        d.frag_begin = (u32)nfrag_total;
        d.nfrag = nf;
        d.flag = nullptr;
        descs.push_back(d);
        nfrag_total += nf;
    }
    if (descs.empty()) return SNAPPY_B200_OK;
    if (nfrag_total > 0x7fffffffull) return SNAPPY_B200_BAD_ARGUMENT;
    Locked L;
    if (L.rc != SNAPPY_B200_OK) return L.rc;
    Context& c = *L.c;
    cudaStream_t st = (cudaStream_t)stream;
    const u32 nd = (u32)descs.size();
    CU(c.descs.ensure(sizeof(DecodeDesc) * nd));
    CU(cudaMemcpyAsync(c.descs.p, descs.data(), sizeof(DecodeDesc) * nd, cudaMemcpyHostToDevice, st));
    CU(cudaStreamSynchronize(st));
    DecodeResult* res = (DecodeResult*)c.result.p;
    CU(cudaMemsetAsync(res, 0, sizeof(DecodeResult), st));
    if (c.opt.timing) CU(cudaEventRecord(c.ev[2], st));
    const u32 grid = ((u32)nfrag_total + kDecodeWarpsPerCta - 1) / kDecodeWarpsPerCta;
    k_decode_fragments<12><<<grid, kDecodeWarpsPerCta * 32, 0, st>>>(nullptr, nullptr, 0u, 0u, (u32)nfrag_total, 0, 0,
                                                                     nullptr, 0, res, (const DecodeDesc*)c.descs.p, nd);
    if (c.opt.timing) {
        CU(cudaEventRecord(c.ev[3], st));
        c.ev_pending[1] = true;
    }
    c.last_launches[1] = 1;
    CU(cudaGetLastError());
    DecodeResult* hr = (DecodeResult*)((u8*)c.pinned + 128);
    CU(cudaMemcpyAsync(hr, res, sizeof(DecodeResult), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    harvest_timing(c, 1);
    return hr->fallback ? SNAPPY_B200_INVALID_INPUT : SNAPPY_B200_OK;
}

int snappy_b200_compress_batched_device(const uint8_t* d_in, const uint64_t* d_in_offsets,
                                        const uint32_t* d_in_sizes, size_t count, uint8_t* d_out,
                                        const uint64_t* d_out_offsets, uint32_t* d_out_sizes,
                                        void* stream) {
    if (count == 0) return SNAPPY_B200_OK;
    if (!d_in || !d_in_offsets || !d_in_sizes || !d_out || !d_out_offsets || !d_out_sizes)
        return SNAPPY_B200_BAD_ARGUMENT;
    if (count > 0x7fffffffull) return SNAPPY_B200_BAD_ARGUMENT;
    Locked L;
    if (L.rc != SNAPPY_B200_OK) return L.rc;
    Context& c = *L.c;
    cudaStream_t st = (cudaStream_t)stream;
    // the largest page decides the shared-memory footprint (fragment buffer + table)
    u32* d_max = (u32*)c.result.p;
    CU(cudaMemsetAsync(d_max, 0, sizeof(DecodeResult), st));
    k_max_u32<<<(unsigned)((count + 1023) / 1024 < 1024 ? (count + 1023) / 1024 : 1024), 256, 0, st>>>(
        d_in_sizes, (u32)count, d_max);
    u32* h = (u32*)((u8*)c.pinned + 640);
    CU(cudaMemcpyAsync(h, d_max, 4, cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));
    const u32 max_size = h[0];
    u32 frag_cap = max_size < kBlockSize ? ((max_size + 15) & ~15u) : kBlockSize;
    if (frag_cap < 16) frag_cap = 16;
    const u32 rules = (u32)c.opt.rules;
    u32 entries = 256;
    while (entries < (rules == 2 ? 2u : 1u) * kMaxTableEntries && entries < max_size) entries <<= 1;
    const size_t smem = (size_t)frag_cap + kFragPad + (size_t)entries * 2 + 16;
    if (c.opt.timing) CU(cudaEventRecord(c.ev[0], st));
    if (c.opt.pages_window && max_size <= kPageWindowMax) {
        // small pages: the window round, table and whole page in shared memory, persistent warps (K1bw)
        u32 ring = 1024;
        while (ring < max_size) ring <<= 1;
        const size_t per_warp = (size_t)entries * 2 + ring + kRingMirror;
        u32 warps = (u32)((226 * 1024) / per_warp);
        if (warps > 16) warps = 16;
        u32 ctas = (u32)((count + warps - 1) / warps);
        if (ctas > (u32)c.sm_count) ctas = (u32)c.sm_count;
        u32* counter = (u32*)((u8*)c.result.p + 64);
        CU(cudaMemsetAsync(counter, 0, 4, st));
        if (rules)
            k_compress_pages_window<true><<<ctas, warps * 32, warps * per_warp, st>>>(
                d_in, d_in_offsets, d_in_sizes, (u32)count, d_out, d_out_offsets, d_out_sizes, ring, entries, counter, rules);
        else
            k_compress_pages_window<false><<<ctas, warps * 32, warps * per_warp, st>>>(
                d_in, d_in_offsets, d_in_sizes, (u32)count, d_out, d_out_offsets, d_out_sizes, ring, entries, counter);
    } else if (rules)
        k_compress_pages<true><<<(unsigned)count, 32, smem, st>>>(d_in, d_in_offsets, d_in_sizes, d_out, d_out_offsets,
                                                                  d_out_sizes, frag_cap, entries, rules);
    else
        k_compress_pages<false><<<(unsigned)count, 32, smem, st>>>(d_in, d_in_offsets, d_in_sizes, d_out,
                                                                   d_out_offsets, d_out_sizes, frag_cap, entries);
    if (c.opt.timing) {
        CU(cudaEventRecord(c.ev[1], st));
        c.ev_pending[0] = true;
    }
    c.last_launches[0] = 2;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(st));
    harvest_timing(c, 0);
    return SNAPPY_B200_OK;
}

int snappy_b200_uncompress_batched_device(const uint8_t* d_in, const uint64_t* d_in_offsets,
                                          const uint32_t* d_in_sizes, size_t count, uint8_t* d_out,
                                          const uint64_t* d_out_offsets, const uint32_t* d_out_caps,
                                          uint32_t* d_out_sizes, int32_t* d_statuses, void* stream) {
    if (count == 0) return SNAPPY_B200_OK;
    if (!d_in || !d_in_offsets || !d_in_sizes || !d_out || !d_out_offsets || !d_out_caps ||
        !d_out_sizes || !d_statuses)
        return SNAPPY_B200_BAD_ARGUMENT;
    if (count > 0x7fffffffull) return SNAPPY_B200_BAD_ARGUMENT;
    Locked L;
    if (L.rc != SNAPPY_B200_OK) return L.rc;
    Context& c = *L.c;
    cudaStream_t st = (cudaStream_t)stream;
    if (c.opt.timing) CU(cudaEventRecord(c.ev[2], st));
    const unsigned grid = (unsigned)((count + kDecodeWarpsPerCta - 1) / kDecodeWarpsPerCta);
    k_decode_pages<<<grid, kDecodeWarpsPerCta * 32, 0, st>>>(d_in, d_in_offsets, d_in_sizes, (u32)count,
                                                             d_out, d_out_offsets, d_out_caps,
                                                             d_out_sizes, d_statuses);
    if (c.opt.timing) {
        CU(cudaEventRecord(c.ev[3], st));
        c.ev_pending[1] = true;
    }
    c.last_launches[1] = 1;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(st));
    harvest_timing(c, 1);
    return SNAPPY_B200_OK;
}

int snappy_b200_validate_batched_device(const uint8_t* d_in, const uint64_t* d_in_offsets, const uint32_t* d_in_sizes,
                                        size_t count, uint32_t* d_claimed, int32_t* d_statuses, void* stream) {
    if (count == 0) return SNAPPY_B200_OK;
    if (!d_in || !d_in_offsets || !d_in_sizes || !d_claimed || !d_statuses) return SNAPPY_B200_BAD_ARGUMENT;
    if (count > 0x7fffffffull) return SNAPPY_B200_BAD_ARGUMENT;
    Locked L;
    if (L.rc != SNAPPY_B200_OK) return L.rc;
    Context& c = *L.c;
    cudaStream_t st = (cudaStream_t)stream;
    if (c.opt.timing) CU(cudaEventRecord(c.ev[2], st));
    const unsigned grid = (unsigned)((count + kDecodeWarpsPerCta - 1) / kDecodeWarpsPerCta);
    k_validate_pages<<<grid, kDecodeWarpsPerCta * 32, 0, st>>>(d_in, d_in_offsets, d_in_sizes, (u32)count, d_claimed,
                                                               d_statuses);
    if (c.opt.timing) {
        CU(cudaEventRecord(c.ev[3], st));
        c.ev_pending[1] = true;
    }
    c.last_launches[1] = 1;
    CU(cudaGetLastError());
    CU(cudaStreamSynchronize(st));
    harvest_timing(c, 1);
    return SNAPPY_B200_OK;
}

float snappy_b200_last_kernel_ms(int which) {
    Context* c = tl_last;  // the lane this thread's last call ran on
    return (c && (which == 0 || which == 1)) ? c->last_ms[which] : 0.f;
}

// ---- side-index sidecar (host only) ---------------------------------------------------------
static const char kIdxMagic[8] = {'S', 'B', '2', 'I', 'D', 'X', '1', 0};

static u32 fnv1a(const u8* p, size_t n) {
    u32 h = 2166136261u;
    for (size_t i = 0; i < n; i++) h = (h ^ p[i]) * 16777619u;
    return h;
}

size_t snappy_b200_index_pack_bound(size_t nfrag) { return 8 + 4 + 4 + 8 + 8 + (nfrag + 1) * 10 + 4; }

int snappy_b200_index_pack(const uint64_t* index, size_t nfrag, uint64_t uncompressed_len, uint8_t* out,
                           size_t* out_len) {
    if (!index || !out || !out_len || nfrag > 0xffffffffull) return SNAPPY_B200_BAD_ARGUMENT;
    if (*out_len < snappy_b200_index_pack_bound(nfrag)) return SNAPPY_B200_BUFFER_TOO_SMALL;
    u8* p = out;
    memcpy(p, kIdxMagic, 8);
    p += 8;
    const u32 nf = (u32)nfrag, zero = 0;
    memcpy(p, &nf, 4);
    memcpy(p + 4, &zero, 4);
    memcpy(p + 8, &uncompressed_len, 8);
    memcpy(p + 16, &index[nfrag], 8);
    p += 24;
    u64 prev = 0;
    for (size_t i = 0; i <= nfrag; i++) {
        if (index[i] < prev) return SNAPPY_B200_BAD_ARGUMENT;  // offsets never decrease
        u64 d = index[i] - prev;
        prev = index[i];
        while (d >= 0x80) {
            *p++ = (u8)(d | 0x80);
            d >>= 7;
        }
        *p++ = (u8)d;
    }
    const u32 h = fnv1a(out, (size_t)(p - out));
    memcpy(p, &h, 4);
    p += 4;
    *out_len = (size_t)(p - out);
    return SNAPPY_B200_OK;
}

int snappy_b200_index_unpack(const uint8_t* in, size_t n, uint64_t* index, size_t* nfrag,
                             uint64_t* uncompressed_len, uint64_t* stream_len) {
    if (!in || !nfrag) return SNAPPY_B200_BAD_ARGUMENT;
    if (n < 8 + 24 + 1 + 4 || memcmp(in, kIdxMagic, 8) != 0) return SNAPPY_B200_INVALID_INPUT;
    u32 nf, h;
    u64 ulen, slen;
    memcpy(&nf, in + 8, 4);
    memcpy(&ulen, in + 16, 8);
    memcpy(&slen, in + 24, 8);
    memcpy(&h, in + n - 4, 4);
    if (fnv1a(in, n - 4) != h) return SNAPPY_B200_INVALID_INPUT;
    if ((u64)nf != (ulen + kBlockSize - 1) / kBlockSize) return SNAPPY_B200_INVALID_INPUT;
    if (index && *nfrag < nf) return SNAPPY_B200_BUFFER_TOO_SMALL;
    const u8* p = in + 32;
    const u8* end = in + n - 4;
    u64 cur = 0;
    for (u64 i = 0; i <= nf; i++) {
        u64 d = 0;
        int shift = 0;
        for (;;) {
            if (p >= end || shift > 63) return SNAPPY_B200_INVALID_INPUT;
            const u8 b = *p++;
            d |= (u64)(b & 0x7f) << shift;
            shift += 7;
            if (!(b & 0x80)) break;
        }
        cur += d;
        if (index) index[i] = cur;
    }
    if (p != end || cur != slen) return SNAPPY_B200_INVALID_INPUT;
    *nfrag = nf;
    if (uncompressed_len) *uncompressed_len = ulen;
    if (stream_len) *stream_len = slen;
    return SNAPPY_B200_OK;
}

int snappy_b200_last_launch_count(int which) {
    Context* c = tl_last;
    return (c && (which == 0 || which == 1)) ? c->last_launches[which] : 0;
}


// option `trace`: begin / end of every fragment of this thread's last compress call (2 x u64 per fragment, see
// k_compress_window); returns the number of fragments copied
size_t snappy_b200_debug_trace(uint64_t* out, size_t max_frags) {
    Context* c = tl_last;
    if (!c || !out || !c->trace.p) return 0;
    std::unique_lock<std::mutex> lk(c->mu);
    int prev = -1;
    cudaGetDevice(&prev);
    cudaSetDevice(c->device);
    const size_t n = c->trace_frags < max_frags ? c->trace_frags : max_frags;
    cudaMemcpy(out, c->trace.p, n * 16, cudaMemcpyDeviceToHost);
    if (prev >= 0) cudaSetDevice(prev);
    return n;
}

int snappy_b200_get_option(const char* name) {
    if (!name) return -1;
    parse_env_options();
    std::unique_lock<std::mutex> lk(g_opt_mu);
    const Options& o = g_opt;
    if (!strcmp(name, "last_decode_path")) return tl_last ? tl_last->last_path : -1;
    if (!strcmp(name, "experiments")) {
#ifdef SB200_EXPERIMENTS
        return 1;
#else
        return 0;
#endif
    }
    const struct { const char* n; int v; } tab[] = {
        {"rules", o.rules}, {"smem_chains", o.smem_chains}, {"l2_chains", o.l2_chains},
        {"l2_chains_big", o.l2_chains_big}, {"l2_ctas", o.l2_ctas}, {"l2_reserve", o.l2_reserve},
        {"ring_smem", o.ring_smem}, {"ring_l2", o.ring_l2}, {"decode_variant", o.decode_variant},
        {"decode_occupancy", o.decode_occupancy}, {"pipe_chunk_frags", o.pipe_chunk_frags},
        {"parse_chunk_log2", o.parse_chunk_log2}, {"uncompress_segments", o.uncompress_segments},
        {"host_pipeline", o.host_pipeline}, {"timing", o.timing}, {"l2_persist", o.l2_persist},
        {"overlap_compact", o.overlap_compact}, {"window", o.window}, {"wide", o.wide}, {"slowcont", o.slowcont},
        {"compress_variant", o.compress_variant}, {"lpt", o.lpt}, {"pin_host", o.pin_host}, {"clean_cuts", o.clean_cuts}, {"trace", o.trace},
        {"profile_range", o.profile_range}, {"pages_window", o.pages_window}, {"mixed", o.mixed}, {"l2_first", o.l2_first}, {"two", o.two},
    };
    for (const auto& e : tab)
        if (!strcmp(name, e.n)) return e.v;
    return -1;
}

void snappy_b200_set_option(const char* name, int value) {
    parse_env_options();
    std::unique_lock<std::mutex> lk(g_opt_mu);
    apply_option(name, value);
}

}  // extern "C"

// ---- multi-GPU communicator (SURVEY.md 8(e)) ----------------------------------------------------------
#include "multi_host.inc"
