// libcropsr_b200: CROPSR Cas9 gRNA candidate scan + Rule-Set-1 score on B200 (sm_100a).
//
// This file is the host side: handles, HBM layout of a genome shard, launches and the C ABI
// (include/cropsr_b200.h).  The kernels live in scan.cuh (pack, scan + score, counts,
// rescore) and rs1.cuh (Rule-Set-1 arithmetic); all of it is HBM-bound integer / fp64
// work -- no tensor cores on this path.
//
// Reference semantics implemented: /root/reference/CROPSR.py:413-434 (scan, bounds,
// windows, transforms) and :285-313 (rs1_score); see DESIGN.md.

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <stdarg.h>
#include <string.h>
#include <stdlib.h>
#include <algorithm>
#include <atomic>
#include <mutex>
#include <new>
#include <type_traits>
#include <utility>
#include <vector>

#include "../../include/cropsr_b200.h"

#ifndef CRP_CTAS_PER_SM
#define CRP_CTAS_PER_SM 4
#endif
#include "scan.cuh"
#include "primers.cuh"
#include "extras.cuh"
#include "offtarget.cuh"

#define CRP_ABI_VERSION 11

static constexpr size_t kScanSmemFixed = (size_t)kStages * kRecBytes + 2 * (size_t)kListCap * sizeof(uint16_t);

// ------------------------------------------------------------------ errors
static thread_local char g_err[512] = "";
static int fail(int code, const char *fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof g_err, fmt, ap);
    va_end(ap);
    return code;
}
#define CUDA_TRY(expr)                                                                      \
    do {                                                                                    \
        cudaError_t e_ = (expr);                                                            \
        if (e_ != cudaSuccess)                                                              \
            return fail(CRP_ERR_CUDA, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(e_), \
                        __FILE__, __LINE__);                                                \
    } while (0)

// ------------------------------------------------------------------ context
struct Context {
    bool ready = false;
    int device = -1;
    int sm_count = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t lanes[3] = {nullptr, nullptr, nullptr};   // crp_scan_segments pipeline
    cudaStream_t lane_out = nullptr;                       // its device-to-host row copies
    std::atomic<uint64_t> launches{0};
    double *d_tables = nullptr;        // RS1 lane tables in device memory
    unsigned int *d_fault = nullptr;   // CRP_CHECKED builds: first violated kernel invariant
};
static Context g_ctx;

// counters behind crp_perf_report
struct Perf {
    std::atomic<uint64_t> commits{0}, scans{0}, sharded_scans{0}, fused_exchanges{0}, capacity_reruns{0};
    std::atomic<uint64_t> positions{0}, candidates{0}, h2d_bytes{0}, d2h_bytes{0}, cache_hits{0}, cache_misses{0};
    double ms_h2d = 0, ms_pack = 0, ms_scan = 0, ms_kernel = 0;     // sums over finished commits / scans
};
static Perf g_perf;

// ------------------------------------------------------------------ host objects
struct Segment {
    uint32_t token_id;
    const uint8_t *token;
    uint64_t token_len, begin, end;
    uint64_t stage_begin, stage_end;   // token positions copied to the device
    uint32_t first_tile, n_tiles;
    // FASTA record ingested on the device (crp_genome_add_fasta_record): token == NULL
    const uint8_t *raw = nullptr;      // first sequence byte of the record, as in the file
    uint64_t raw_bytes = 0;
    uint32_t width = 0, last = 0;
    uint64_t ascii_off = 0;            // token position stage_begin in the ASCII buffer kept on the device
};

struct crp_genome {
    std::vector<Segment> segs;
    cudaStream_t st = nullptr;         // every operation on this genome and its results is ordered on this stream
    cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};   // commit timing: start, H2D done, pack done
    bool committed = false;
    uint64_t n_positions = 0;          // owned positions
    uint4 *records = nullptr;          // n_tiles tile records (scan.cuh)
    unsigned char *pam = nullptr;      // n_tiles PAM records (count phase of the scan: tiles at the ends of a token)
    TileHdr *hdr = nullptr;            // n_tiles tile headers (count phase of the scan: descriptor + chunk counts)
    uint32_t n_tiles = 0;
    uint32_t *d_seg_first = nullptr, *d_seg_count = nullptr;
    float ms_h2d = 0.f, ms_pack = 0.f;
    uint8_t *d_ascii = nullptr;                // ASCII tokens, kept after the pack only for device-ingested FASTA records
    bool fasta = false;
    unsigned int *h_bad = nullptr;             // pinned: non-zero after the commit if a FASTA record was not plain
};

struct crp_result {
    const crp_genome *g = nullptr;
    cudaStream_t st = nullptr;
    cudaEvent_t ev[3] = {nullptr, nullptr, nullptr};   // scan start, scan (+ all-gather) end, counts on the host
    cudaEvent_t ev_kernel = nullptr;           // sharded scans: between the kernel and the all-gather
    unsigned long long *h_counts = nullptr;    // pinned, [2*stride]: counts land here when the scan has run
    uint32_t stride = 0;                       // count slots per strand: n_seg, or the `slots` of a sharded scan
    unsigned long long *d_gather = nullptr;    // sharded scans: [world][2*stride] counts of every rank (NCCL all-gather)
    unsigned long long *h_gather = nullptr;    // pinned copy
    bool fused = false;                        // counts exchanged by the kernel itself (peer stores), not by NCCL
    uint32_t epoch = 0;
    unsigned int *h_xchg_error = nullptr;      // pinned
    float ms_kernel = 0.f;
    int guide_len = 0;
    uint32_t flags = 0;
    uint64_t capacity = 0;
    uint64_t n_plus = 0, n_minus = 0;
    bool scored = false;
    uint32_t *pos[2] = {nullptr, nullptr};
    unsigned long long *packed[2] = {nullptr, nullptr};
    double *x[2] = {nullptr, nullptr};
    unsigned char *state = nullptr;            // warp_pref | cta_tot | segment counts | tickets, one allocation
    size_t state_bytes = 0, zero_offset = 0;   // segment counts and tickets start at zero_offset
    unsigned long long *d_counts = nullptr;    // [2*stride], inside state
    std::vector<uint64_t> seg_plus, seg_minus;
    float ms_scan = 0.f;                       // every launch of this scan, a capacity rerun included
    uint32_t n_launches = 0;
};

// CRP_TRACE=1: host-side wall time of every stage of the big calls, on stderr
#include <chrono>
struct Trace {
    const char *what;
    bool on;
    std::chrono::steady_clock::time_point t0;
    explicit Trace(const char *w) : what(w), on(getenv("CRP_TRACE") != nullptr), t0(std::chrono::steady_clock::now()) {}
    void lap(const char *stage) {
        if (!on) return;
        const auto t1 = std::chrono::steady_clock::now();
        fprintf(stderr, "[crp] %s: %s %.3f ms\n", what, stage, std::chrono::duration<double, std::milli>(t1 - t0).count());
        t0 = t1;
    }
};

static int need_ctx() {
    if (!g_ctx.ready) return fail(CRP_ERR_STATE, "crp_init has not been called");
    return 0;
}

// Device memory comes from a block cache of this library: cudaMalloc / cudaFree cost 10-70 ms per
// call on a 180 GB part and the driver's stream-ordered pool grows for milliseconds whenever the
// set of live sizes changes, while a genome commit and a scan allocate ~1 GB between them.  A freed
// block keeps an event recorded on the stream that used it last; whoever gets the block next makes
// its stream wait for that event, so reuse across streams is ordered without any host wait.
// Blocks are handed out best-fit within 1/8 of slack and only returned to the driver by crp_shutdown.
struct DevBlock {
    void *ptr;
    size_t bytes;
    cudaEvent_t ev;
};
static std::vector<DevBlock> g_dev_free;                       // idle blocks
static std::vector<DevBlock> g_dev_live;                       // blocks handed out
static std::mutex g_mem_mu;                                    // guards both block lists and the pinned list
template <typename T>
static cudaError_t dev_alloc(T **ptr, size_t bytes, cudaStream_t st) {
    std::lock_guard<std::mutex> lock(g_mem_mu);
    const size_t want = (bytes ? bytes : 16) + 255 & ~(size_t)255;
    // best fit among the idle blocks whose last user has FINISHED: a block that is still in use on another
    // stream would chain this stream behind that one (the copy-in of pipeline group k + 1 behind the pack
    // kernel of group k: a bubble on the copy engine per group); such a block is only taken when nothing
    // else fits and the driver has no memory left (below)
    size_t best = g_dev_free.size(), busy = g_dev_free.size();
    for (size_t i = 0; i < g_dev_free.size(); ++i) {
        const size_t b = g_dev_free[i].bytes;
        if (b < want || b - want > want / 8 + 4096) continue;
        if (cudaEventQuery(g_dev_free[i].ev) == cudaSuccess) {
            best = i;                                          // first fit: one query per allocation in the steady state
            break;
        } else {
            cudaGetLastError();                                // cudaErrorNotReady is not an error here
            if (busy == g_dev_free.size() || b < g_dev_free[busy].bytes) busy = i;
        }
    }
    DevBlock blk;
    if (best < g_dev_free.size()) {
        blk = g_dev_free[best];
        g_dev_free.erase(g_dev_free.begin() + best);
        g_perf.cache_hits++;
    } else if (cudaMalloc(&blk.ptr, want) == cudaSuccess) {
        g_perf.cache_misses++;
        blk.bytes = want;
        if (cudaError_t e = cudaEventCreateWithFlags(&blk.ev, cudaEventDisableTiming)) {
            cudaFree(blk.ptr);
            return e;
        }
    } else if (busy < g_dev_free.size()) {
        cudaGetLastError();
        blk = g_dev_free[busy];
        g_dev_free.erase(g_dev_free.begin() + busy);
        if (cudaError_t e = cudaStreamWaitEvent(st, blk.ev, 0)) return e;
    } else {
        cudaGetLastError();
        blk.bytes = want;
        if (cudaMalloc(&blk.ptr, want) != cudaSuccess) {        // out of memory: give the idle blocks back first
            cudaGetLastError();
            cudaDeviceSynchronize();
            for (DevBlock &b : g_dev_free) {
                cudaFree(b.ptr);
                cudaEventDestroy(b.ev);
            }
            g_dev_free.clear();
            if (cudaError_t e = cudaMalloc(&blk.ptr, want)) return e;
        }
        if (cudaError_t e = cudaEventCreateWithFlags(&blk.ev, cudaEventDisableTiming)) {
            cudaFree(blk.ptr);
            return e;
        }
    }
    g_dev_live.push_back(blk);
    *ptr = reinterpret_cast<T *>(blk.ptr);
    return cudaSuccess;
}
static void dev_free(void *ptr, cudaStream_t st) {
    if (!ptr) return;
    std::lock_guard<std::mutex> lock(g_mem_mu);
    for (size_t i = g_dev_live.size(); i-- > 0;)
        if (g_dev_live[i].ptr == ptr) {
            DevBlock blk = g_dev_live[i];
            g_dev_live.erase(g_dev_live.begin() + i);
            cudaEventRecord(blk.ev, st);
            g_dev_free.push_back(blk);
            return;
        }
}
static void dev_cache_release() {
    std::lock_guard<std::mutex> lock(g_mem_mu);
    for (DevBlock &b : g_dev_free) {
        cudaFree(b.ptr);
        cudaEventDestroy(b.ev);
    }
    g_dev_free.clear();
}

// Small pinned host blocks (the per-scan counts) are recycled: cudaHostAlloc takes ~0.1 ms.
static std::vector<std::pair<size_t, void *>> g_pinned_free;
static void *pinned_get(size_t bytes) {
    std::lock_guard<std::mutex> lock(g_mem_mu);
    for (size_t i = 0; i < g_pinned_free.size(); ++i)
        if (g_pinned_free[i].first >= bytes) {
            void *p = g_pinned_free[i].second;
            g_pinned_free.erase(g_pinned_free.begin() + i);
            return p;
        }
    const size_t want = bytes < 4096 ? 4096 : bytes;
    void *p = nullptr;
    if (cudaHostAlloc(&p, want + sizeof(size_t) * 2, cudaHostAllocMapped) != cudaSuccess) return nullptr;   // kernels may store into it
    *reinterpret_cast<size_t *>(p) = want;
    return reinterpret_cast<char *>(p) + sizeof(size_t) * 2;
}
static void pinned_put(void *p) {
    if (!p) return;
    std::lock_guard<std::mutex> lock(g_mem_mu);
    const size_t cap = *reinterpret_cast<size_t *>(reinterpret_cast<char *>(p) - sizeof(size_t) * 2);
    g_pinned_free.emplace_back(cap, p);
}


// ------------------------------------------------------------------ NCCL (one process per GPU)
// The library talks to NCCL through dlopen: a single-GPU run needs no NCCL at all, and inside a
// process that already carries one (PyTorch's bundled copy) the same copy is used.
#include <dlfcn.h>
#include <nccl.h>
struct Comm {
    void *dl = nullptr;
    ncclComm_t comm = nullptr;
    int rank = 0, world = 1;
    ncclResult_t (*GetUniqueId)(ncclUniqueId *) = nullptr;
    ncclResult_t (*CommInitRank)(ncclComm_t *, int, ncclUniqueId, int) = nullptr;
    ncclResult_t (*CommDestroy)(ncclComm_t) = nullptr;
    ncclResult_t (*AllGather)(const void *, void *, size_t, ncclDataType_t, ncclComm_t, cudaStream_t) = nullptr;
    ncclResult_t (*AllReduce)(const void *, void *, size_t, ncclDataType_t, ncclRedOp_t, ncclComm_t, cudaStream_t) = nullptr;
    const char *(*GetErrorString)(ncclResult_t) = nullptr;
    unsigned long long *d_scratch = nullptr;   // barrier payload
    // Fused exchange of the per-segment counts (scan.cuh): every rank owns one buffer
    //   gather [2 parities][world][2 * kXchgSlots] u64 | flags [2 parities][kMaxPeers] u32 | error u32
    // that its peers map through CUDA IPC and write with plain stores over NVLink.
    unsigned char *xchg = nullptr;             // this rank's buffer
    unsigned char *peer[kMaxPeers] = {};       // every rank's buffer as mapped here (peer[rank] == xchg)
    bool fused = false;                        // all peers mapped: crp_scan_score_sharded may use the fused exchange
    int mode = 0;                              // 0 = fused when possible, 1 = always the NCCL all-gather
    uint32_t epoch = 0;                        // sharded scans so far (the same on every rank: the call is collective)
    char why_not_fused[160] = "";
};
static Comm g_comm;
static constexpr uint32_t kXchgSlots = 32768;                       // segments per rank the fused exchange has room for
static size_t xchg_gather_bytes() { return (size_t)2 * kMaxPeers * 2 * kXchgSlots * sizeof(unsigned long long); }
static size_t xchg_bytes() { return xchg_gather_bytes() + 2 * kMaxPeers * sizeof(unsigned int) + 64; }
static unsigned long long *xchg_gather(unsigned char *base, uint32_t parity, uint32_t world, uint32_t stride) {
    (void)world;
    (void)stride;
    return reinterpret_cast<unsigned long long *>(base) + (size_t)parity * kMaxPeers * 2 * kXchgSlots;
}
static unsigned int *xchg_flags(unsigned char *base, uint32_t parity) {
    return reinterpret_cast<unsigned int *>(base + xchg_gather_bytes()) + (size_t)parity * kMaxPeers;
}
static unsigned int *xchg_error(unsigned char *base) {
    return reinterpret_cast<unsigned int *>(base + xchg_gather_bytes()) + 2 * kMaxPeers;
}

static int comm_load() {
    if (g_comm.dl) return 0;
    const char *names[] = {getenv("CRP_NCCL_LIB"), "libnccl.so.2", "libnccl.so"};
    for (const char *n : names) {
        if (!n) continue;
        if ((g_comm.dl = dlopen(n, RTLD_NOW | RTLD_GLOBAL))) break;
    }
    if (!g_comm.dl) return fail(CRP_ERR_STATE, "libnccl.so.2 not found: %s", dlerror());
#define CRP_NCCL_SYM(field, name)                                                         \
    if (!(*(void **)(&g_comm.field) = dlsym(g_comm.dl, name))) {                          \
        dlclose(g_comm.dl);                                                               \
        g_comm.dl = nullptr;                                                              \
        return fail(CRP_ERR_STATE, "NCCL symbol %s missing", name);                       \
    }
    CRP_NCCL_SYM(GetUniqueId, "ncclGetUniqueId")
    CRP_NCCL_SYM(CommInitRank, "ncclCommInitRank")
    CRP_NCCL_SYM(CommDestroy, "ncclCommDestroy")
    CRP_NCCL_SYM(AllGather, "ncclAllGather")
    CRP_NCCL_SYM(AllReduce, "ncclAllReduce")
    CRP_NCCL_SYM(GetErrorString, "ncclGetErrorString")
#undef CRP_NCCL_SYM
    return 0;
}
#define NCCL_TRY(expr)                                                                                \
    do {                                                                                              \
        ncclResult_t e_ = (expr);                                                                     \
        if (e_ != ncclSuccess) return fail(CRP_ERR_CUDA, "%s failed: %s", #expr, g_comm.GetErrorString(e_)); \
    } while (0)

static int comm_allgather_u64(const unsigned long long *send, unsigned long long *recv, size_t count, cudaStream_t st) {
    if (!g_comm.comm) return fail(CRP_ERR_STATE, "crp_comm_init has not been called");
    NCCL_TRY(g_comm.AllGather(send, recv, count, ncclUint64, g_comm.comm, st));
    return 0;
}

// ------------------------------------------------------------------ C ABI
extern "C" {

int crp_result_free(crp_result *r);
int crp_comm_shutdown(void);


int crp_abi_version(void) { return CRP_ABI_VERSION; }

int crp_tile_size(void) { return kTile; }

/* 1 if this build carries the kernel's self-checks (make checked, -DCRP_CHECKED) */
int crp_checked_build(void) {
#ifdef CRP_CHECKED
    return 1;
#else
    return 0;
#endif
}

const char *crp_last_error(void) { return g_err; }

/* debug hook of tools/phase_timeline.py: device buffer of 8 x u64 per CTA, or NULL */
int crp_debug_set_times(void *dev_ptr) {
    unsigned long long *p = (unsigned long long *)dev_ptr;
    CUDA_TRY(cudaMemcpyToSymbol(g_dbg_times, &p, sizeof p));
    return 0;
}

int crp_device_count(int *count) {
    if (!count) return fail(CRP_ERR_ARG, "count is NULL");
    CUDA_TRY(cudaGetDeviceCount(count));
    return 0;
}

int crp_init(int device) {
    if (g_ctx.ready) {
        if (g_ctx.device == device) return 0;
        return fail(CRP_ERR_STATE, "already initialised on device %d", g_ctx.device);
    }
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if (prop.major != 10)
        return fail(CRP_ERR_CUDA, "device %d is sm_%d%d; this library is built for sm_100a only", device,
                    prop.major, prop.minor);
    CUDA_TRY(cudaStreamCreateWithFlags(&g_ctx.stream, cudaStreamNonBlocking));
    {
        std::vector<double> tab;
        char msg[128];
        if (build_rs1_tables(tab, msg, sizeof msg)) return fail(CRP_ERR_STATE, "%s", msg);
        CUDA_TRY(cudaMalloc(&g_ctx.d_tables, tab.size() * sizeof(double)));
        CUDA_TRY(cudaMemcpy(g_ctx.d_tables, tab.data(), tab.size() * sizeof(double), cudaMemcpyHostToDevice));
    }
#ifdef CRP_CHECKED
    CUDA_TRY(cudaMalloc(&g_ctx.d_fault, sizeof(unsigned int)));
    CUDA_TRY(cudaMemset(g_ctx.d_fault, 0, sizeof(unsigned int)));
#endif
    g_ctx.device = device;
    g_ctx.sm_count = prop.multiProcessorCount;
    g_ctx.launches = 0;
    g_ctx.ready = true;
    return 0;
}

int crp_shutdown(void) {
    if (!g_ctx.ready) return 0;
    crp_comm_shutdown();
    cudaStreamSynchronize(g_ctx.stream);
    cudaDeviceSynchronize();
    dev_cache_release();
    {
        std::lock_guard<std::mutex> lock(g_mem_mu);
        for (auto &pf : g_pinned_free) cudaFreeHost(reinterpret_cast<char *>(pf.second) - sizeof(size_t) * 2);
        g_pinned_free.clear();
    }
    cudaStreamDestroy(g_ctx.stream);
    for (cudaStream_t l : g_ctx.lanes)
        if (l) cudaStreamDestroy(l);
    if (g_ctx.lane_out) cudaStreamDestroy(g_ctx.lane_out);
    cudaFree(g_ctx.d_tables);
    if (g_ctx.d_fault) cudaFree(g_ctx.d_fault);
    g_ctx.d_fault = nullptr;
    g_ctx.ready = false;
    g_ctx.device = -1;
    g_ctx.stream = nullptr;
    for (cudaStream_t &l : g_ctx.lanes) l = nullptr;
    g_ctx.lane_out = nullptr;
    g_ctx.d_tables = nullptr;
    g_ctx.launches = 0;
    return 0;
}

/* JSON object with the library's counters since crp_init (SURVEY.md section 5: perf report) */
int crp_perf_report(char *buf, uint64_t capacity, uint64_t *needed) {
    char tmp[1536];
    size_t live = 0, idle = 0, live_bytes = 0, idle_bytes = 0;
    {
        std::lock_guard<std::mutex> lock(g_mem_mu);
        live = g_dev_live.size();
        idle = g_dev_free.size();
        for (const DevBlock &b : g_dev_live) live_bytes += b.bytes;
        for (const DevBlock &b : g_dev_free) idle_bytes += b.bytes;
    }
    const int n = snprintf(
        tmp, sizeof tmp,
        "{\"abi\": %d, \"checked_build\": %d, \"device\": %d, \"sm_count\": %d, \"kernel_launches\": %llu, "
        "\"commits\": %llu, \"scans\": %llu, \"sharded_scans\": %llu, \"fused_exchanges\": %llu, \"capacity_reruns\": %llu, "
        "\"positions_packed\": %llu, \"candidates\": %llu, \"h2d_token_bytes\": %llu, \"d2h_row_bytes\": %llu, "
        "\"ms_h2d\": %.4f, \"ms_pack\": %.4f, \"ms_scan\": %.4f, \"ms_scan_kernels\": %.4f, "
        "\"comm\": {\"rank\": %d, \"world\": %d, \"fused_exchange\": %s}, "
        "\"block_cache\": {\"live_blocks\": %zu, \"live_bytes\": %zu, \"idle_blocks\": %zu, \"idle_bytes\": %zu, \"hits\": %llu, \"misses\": %llu}}",
        CRP_ABI_VERSION, crp_checked_build(), g_ctx.device, g_ctx.sm_count, (unsigned long long)g_ctx.launches.load(),
        (unsigned long long)g_perf.commits.load(), (unsigned long long)g_perf.scans.load(),
        (unsigned long long)g_perf.sharded_scans.load(), (unsigned long long)g_perf.fused_exchanges.load(),
        (unsigned long long)g_perf.capacity_reruns.load(), (unsigned long long)g_perf.positions.load(),
        (unsigned long long)g_perf.candidates.load(), (unsigned long long)g_perf.h2d_bytes.load(),
        (unsigned long long)g_perf.d2h_bytes.load(), g_perf.ms_h2d, g_perf.ms_pack, g_perf.ms_scan, g_perf.ms_kernel,
        g_comm.comm ? g_comm.rank : 0, g_comm.comm ? g_comm.world : 1, g_comm.comm && g_comm.fused && g_comm.mode == 0 ? "true" : "false",
        live, live_bytes, idle, idle_bytes, (unsigned long long)g_perf.cache_hits.load(), (unsigned long long)g_perf.cache_misses.load());
    if (needed) *needed = (uint64_t)n + 1;
    if (!buf || capacity < (uint64_t)n + 1) return fail(CRP_ERR_RANGE, "perf report needs %d bytes", n + 1);
    memcpy(buf, tmp, (size_t)n + 1);
    return 0;
}

int crp_launch_count(uint64_t *n) {
    if (!n) return fail(CRP_ERR_ARG, "n is NULL");
    *n = g_ctx.launches;
    return 0;
}

int crp_comm_unique_id(uint8_t *id) {
    if (!id) return fail(CRP_ERR_ARG, "id is NULL");
    if (int rc = comm_load()) return rc;
    ncclUniqueId u;
    NCCL_TRY(g_comm.GetUniqueId(&u));
    static_assert(sizeof u == CRP_COMM_ID_BYTES, "ncclUniqueId size");
    memcpy(id, &u, sizeof u);
    return 0;
}

int crp_comm_init(int rank, int world, const uint8_t *id) {
    if (int rc = need_ctx()) return rc;
    if (!id || world < 1 || rank < 0 || rank >= world) return fail(CRP_ERR_ARG, "bad rank %d / world %d", rank, world);
    if (g_comm.comm) return fail(CRP_ERR_STATE, "communicator already initialised (rank %d of %d)", g_comm.rank, g_comm.world);
    if (int rc = comm_load()) return rc;
    ncclUniqueId u;
    memcpy(&u, id, sizeof u);
    CUDA_TRY(cudaSetDevice(g_ctx.device));
    NCCL_TRY(g_comm.CommInitRank(&g_comm.comm, world, u, rank));
    g_comm.rank = rank;
    g_comm.world = world;
    CUDA_TRY(cudaMalloc(&g_comm.d_scratch, 2 * sizeof(unsigned long long)));
    CUDA_TRY(cudaMemset(g_comm.d_scratch, 0, 2 * sizeof(unsigned long long)));
    g_comm.epoch = 0;
    g_comm.mode = 0;
    if (const char *e = getenv("CRP_COMM_EXCHANGE")) g_comm.mode = !strcmp(e, "nccl") ? 1 : 0;
    // ---- fused exchange: map every rank's buffer into this process (CUDA IPC, peer access over NVLink).
    // Anything that does not work here leaves the NCCL all-gather as the exchange; the decision is
    // made together (an all-reduce of the per-rank verdicts), so that all ranks run the same protocol.
    g_comm.fused = false;
    g_comm.why_not_fused[0] = 0;
    bool ok = world <= kMaxPeers;
    if (!ok) snprintf(g_comm.why_not_fused, sizeof g_comm.why_not_fused, "world %d > %d", world, kMaxPeers);
    cudaIpcMemHandle_t mine;
    memset(&mine, 0, sizeof mine);
    if (ok) {
        if (cudaMalloc(&g_comm.xchg, xchg_bytes()) != cudaSuccess || cudaMemset(g_comm.xchg, 0, xchg_bytes()) != cudaSuccess ||
            cudaIpcGetMemHandle(&mine, g_comm.xchg) != cudaSuccess) {
            snprintf(g_comm.why_not_fused, sizeof g_comm.why_not_fused, "exchange buffer / IPC handle: %s",
                     cudaGetErrorString(cudaGetLastError()));
            ok = false;
        }
    }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
    std::vector<uint64_t> handles((size_t)world * 8);
    {
        unsigned long long *d = nullptr;
        CUDA_TRY(cudaMalloc(&d, ((size_t)world + 1) * 64));
        CUDA_TRY(cudaMemcpy(d, &mine, 64, cudaMemcpyHostToDevice));
        NCCL_TRY(g_comm.AllGather(d, d + 8, 8, ncclUint64, g_comm.comm, g_ctx.stream));
        CUDA_TRY(cudaStreamSynchronize(g_ctx.stream));
        CUDA_TRY(cudaMemcpy(handles.data(), d + 8, (size_t)world * 64, cudaMemcpyDeviceToHost));
        cudaFree(d);
    }
    for (int q = 0; q < world && ok; ++q) {
        if (q == rank) {
            g_comm.peer[q] = g_comm.xchg;
            continue;
        }
        cudaIpcMemHandle_t h;
        memcpy(&h, &handles[(size_t)q * 8], 64);
        void *ptr = nullptr;
        if (cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess) != cudaSuccess) {
            snprintf(g_comm.why_not_fused, sizeof g_comm.why_not_fused, "cudaIpcOpenMemHandle(rank %d): %s", q,
                     cudaGetErrorString(cudaGetLastError()));
            ok = false;
        } else {
            g_comm.peer[q] = static_cast<unsigned char *>(ptr);
        }
    }
    {   // unanimous?
        unsigned long long v = ok ? 0ull : 1ull;
        CUDA_TRY(cudaMemcpy(g_comm.d_scratch, &v, sizeof v, cudaMemcpyHostToDevice));
        NCCL_TRY(g_comm.AllReduce(g_comm.d_scratch, g_comm.d_scratch + 1, 1, ncclUint64, ncclSum, g_comm.comm, g_ctx.stream));
        CUDA_TRY(cudaStreamSynchronize(g_ctx.stream));
        CUDA_TRY(cudaMemcpy(&v, g_comm.d_scratch + 1, sizeof v, cudaMemcpyDeviceToHost));
        CUDA_TRY(cudaMemset(g_comm.d_scratch, 0, 2 * sizeof(unsigned long long)));
        if (v && ok) snprintf(g_comm.why_not_fused, sizeof g_comm.why_not_fused, "%llu other rank(s) could not map the buffers", v);
        g_comm.fused = v == 0;
    }
    return 0;
}

/* 0: the kernel exchanges the counts itself when every rank could map its peers' buffers (default);
 * 1: always the NCCL all-gather behind the kernel.  Collective in effect: set it on every rank. */
int crp_comm_set_exchange(int mode) {
    if (mode != 0 && mode != 1) return fail(CRP_ERR_ARG, "mode must be 0 (fused) or 1 (nccl)");
    g_comm.mode = mode;
    return 0;
}

/* *fused = 1 if sharded scans of this communicator exchange their counts inside the kernel;
 * otherwise why (a static string) says what prevented it. */
int crp_comm_exchange_info(int *fused, const char **why) {
    if (fused) *fused = g_comm.comm && g_comm.fused && g_comm.mode == 0 ? 1 : 0;
    if (why) *why = g_comm.mode == 1 ? "NCCL exchange selected" : g_comm.why_not_fused;
    return 0;
}

int crp_comm_info(int *rank, int *world) {
    if (rank) *rank = g_comm.comm ? g_comm.rank : 0;
    if (world) *world = g_comm.comm ? g_comm.world : 1;
    return 0;
}

/* all ranks' streams have drained and every rank has arrived (all-reduce of one word + sync) */
int crp_comm_barrier(void) {
    if (int rc = need_ctx()) return rc;
    CUDA_TRY(cudaDeviceSynchronize());
    if (!g_comm.comm) return 0;
    NCCL_TRY(g_comm.AllReduce(g_comm.d_scratch, g_comm.d_scratch + 1, 1, ncclUint64, ncclSum, g_comm.comm, g_ctx.stream));
    CUDA_TRY(cudaStreamSynchronize(g_ctx.stream));
    return 0;
}

/* element-wise maximum of n doubles over all ranks (timings: the slowest rank sets the step) */
int crp_comm_max_f64(double *v, uint32_t n) {
    if (int rc = need_ctx()) return rc;
    if (!v && n) return fail(CRP_ERR_ARG, "v is NULL");
    if (!g_comm.comm || n == 0) return 0;
    double *d = nullptr;
    CUDA_TRY(dev_alloc(&d, n * sizeof(double), g_ctx.stream));
    CUDA_TRY(cudaMemcpyAsync(d, v, n * sizeof(double), cudaMemcpyHostToDevice, g_ctx.stream));
    NCCL_TRY(g_comm.AllReduce(d, d, n, ncclDouble, ncclMax, g_comm.comm, g_ctx.stream));
    CUDA_TRY(cudaMemcpyAsync(v, d, n * sizeof(double), cudaMemcpyDeviceToHost, g_ctx.stream));
    CUDA_TRY(cudaStreamSynchronize(g_ctx.stream));
    dev_free(d, g_ctx.stream);
    return 0;
}

int crp_comm_sum_f64(double *v, uint32_t n) {
    if (int rc = need_ctx()) return rc;
    if (!v && n) return fail(CRP_ERR_ARG, "v is NULL");
    if (!g_comm.comm || n == 0) return 0;
    double *d = nullptr;
    CUDA_TRY(dev_alloc(&d, n * sizeof(double), g_ctx.stream));
    CUDA_TRY(cudaMemcpyAsync(d, v, n * sizeof(double), cudaMemcpyHostToDevice, g_ctx.stream));
    NCCL_TRY(g_comm.AllReduce(d, d, n, ncclDouble, ncclSum, g_comm.comm, g_ctx.stream));
    CUDA_TRY(cudaMemcpyAsync(v, d, n * sizeof(double), cudaMemcpyDeviceToHost, g_ctx.stream));
    CUDA_TRY(cudaStreamSynchronize(g_ctx.stream));
    dev_free(d, g_ctx.stream);
    return 0;
}

/* all-gather of n host words per rank: out[rank * n + i] (host in, host out; bootstrap-sized payloads) */
int crp_comm_allgather_u64(const uint64_t *in, uint32_t n, uint64_t *out) {
    if (int rc = need_ctx()) return rc;
    if (n && (!in || !out)) return fail(CRP_ERR_ARG, "NULL argument");
    if (n == 0) return 0;
    if (!g_comm.comm) {
        memcpy(out, in, n * sizeof(uint64_t));
        return 0;
    }
    unsigned long long *d = nullptr;
    const size_t w = (size_t)g_comm.world;
    CUDA_TRY(dev_alloc(&d, (w + 1) * n * sizeof(uint64_t), g_ctx.stream));
    CUDA_TRY(cudaMemcpyAsync(d, in, n * sizeof(uint64_t), cudaMemcpyHostToDevice, g_ctx.stream));
    if (int rc = comm_allgather_u64(d, d + n, n, g_ctx.stream)) {
        dev_free(d, g_ctx.stream);
        return rc;
    }
    CUDA_TRY(cudaMemcpyAsync(out, d + n, w * n * sizeof(uint64_t), cudaMemcpyDeviceToHost, g_ctx.stream));
    CUDA_TRY(cudaStreamSynchronize(g_ctx.stream));
    dev_free(d, g_ctx.stream);
    return 0;
}

/* Link probe: h2d_bytes host->device and d2h_bytes device->host, both pinned, both directions at
 * once on two streams, `reps` times; *ms = mean wall time of one round.  What a step that moves
 * exactly these bytes could reach if the kernels were free. */
int crp_link_probe(uint64_t h2d_bytes, uint64_t d2h_bytes, uint32_t reps, float *ms) {
    if (int rc = need_ctx()) return rc;
    if (!ms || !reps) return fail(CRP_ERR_ARG, "bad argument");
    void *h_in = nullptr, *h_out = nullptr;
    unsigned char *d_in = nullptr, *d_out = nullptr;
    cudaStream_t s2 = nullptr;
    int rc = 0;
    do {
        if (cudaHostAlloc(&h_in, h2d_bytes + 16, cudaHostAllocDefault) != cudaSuccess ||
            cudaHostAlloc(&h_out, d2h_bytes + 16, cudaHostAllocDefault) != cudaSuccess) {
            rc = fail(CRP_ERR_NOMEM, "cudaHostAlloc of the probe buffers failed");
            break;
        }
        memset(h_in, 1, h2d_bytes + 16);
        memset(h_out, 1, d2h_bytes + 16);
        if (dev_alloc(&d_in, h2d_bytes + 16, g_ctx.stream) != cudaSuccess || dev_alloc(&d_out, d2h_bytes + 16, g_ctx.stream) != cudaSuccess ||
            cudaStreamCreateWithFlags(&s2, cudaStreamNonBlocking) != cudaSuccess) {
            rc = fail(CRP_ERR_NOMEM, "device buffers of the link probe failed");
            break;
        }
        cudaStreamSynchronize(g_ctx.stream);
        double total = 0.0;
        for (uint32_t i = 0; i <= reps; ++i) {            // round 0 warms up
            const auto t0 = std::chrono::steady_clock::now();
            cudaMemcpyAsync(d_in, h_in, h2d_bytes, cudaMemcpyHostToDevice, g_ctx.stream);
            cudaMemcpyAsync(h_out, d_out, d2h_bytes, cudaMemcpyDeviceToHost, s2);
            cudaStreamSynchronize(g_ctx.stream);
            cudaStreamSynchronize(s2);
            if (i) total += std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now() - t0).count();
        }
        if (cudaGetLastError() != cudaSuccess) rc = fail(CRP_ERR_CUDA, "link probe copies failed");
        *ms = (float)(total / reps);
    } while (0);
    if (s2) cudaStreamDestroy(s2);
    dev_free(d_in, g_ctx.stream);
    dev_free(d_out, g_ctx.stream);
    if (h_in) cudaFreeHost(h_in);
    if (h_out) cudaFreeHost(h_out);
    return rc;
}

int crp_comm_shutdown(void) {
    if (g_comm.comm) {
        cudaDeviceSynchronize();
        // nobody unmaps while a peer may still be storing: everyone meets first (the call is collective)
        g_comm.AllReduce(g_comm.d_scratch, g_comm.d_scratch + 1, 1, ncclUint64, ncclSum, g_comm.comm, g_ctx.stream);
        cudaStreamSynchronize(g_ctx.stream);
        for (int q = 0; q < g_comm.world && q < kMaxPeers; ++q)
            if (g_comm.peer[q] && q != g_comm.rank) cudaIpcCloseMemHandle(g_comm.peer[q]);
        for (auto &pp : g_comm.peer) pp = nullptr;
        if (g_comm.xchg) cudaFree(g_comm.xchg);
        g_comm.xchg = nullptr;
        g_comm.fused = false;
        g_comm.CommDestroy(g_comm.comm);
        cudaFree(g_comm.d_scratch);
        g_comm.comm = nullptr;
        g_comm.d_scratch = nullptr;
        g_comm.rank = 0;
        g_comm.world = 1;
    }
    return 0;
}

/* Evict the L2 cache (benchmarks: between timed scans): a memset larger than L2, on the library stream. */
int crp_flush_l2(void) {
    if (int rc = need_ctx()) return rc;
    unsigned char *buf = nullptr;                    // from the block cache: allocated once, reused by every call
    const size_t bytes = 512ull << 20;
    CUDA_TRY(dev_alloc(&buf, bytes, g_ctx.stream));
    cudaError_t e = cudaMemsetAsync(buf, 0, bytes, g_ctx.stream);
    dev_free(buf, g_ctx.stream);
    CUDA_TRY(e);
    CUDA_TRY(cudaStreamSynchronize(g_ctx.stream));
    return 0;
}

int crp_device_synchronize(void) {
    if (int rc = need_ctx()) return rc;
    CUDA_TRY(cudaDeviceSynchronize());
    return 0;
}

int crp_host_alloc(void **ptr, uint64_t bytes) {
    if (!ptr) return fail(CRP_ERR_ARG, "ptr is NULL");
    if (int rc = need_ctx()) return rc;
    CUDA_TRY(cudaHostAlloc(ptr, bytes ? bytes : 1, cudaHostAllocDefault));
    return 0;
}

int crp_host_free(void *ptr) {
    if (ptr) CUDA_TRY(cudaFreeHost(ptr));
    return 0;
}

static cudaStream_t stream_of(const crp_genome *g) { return g->st ? g->st : g_ctx.stream; }

int crp_genome_new(crp_genome **g) {
    if (!g) return fail(CRP_ERR_ARG, "g is NULL");
    if (int rc = need_ctx()) return rc;
    *g = new (std::nothrow) crp_genome();
    if (!*g) return fail(CRP_ERR_NOMEM, "out of host memory");
    return 0;
}

int crp_genome_add_segment(crp_genome *g, uint32_t token_id, const uint8_t *token_ascii,
                           uint64_t token_len, uint64_t seg_begin, uint64_t seg_end) {
    if (!g) return fail(CRP_ERR_ARG, "g is NULL");
    if (g->committed) return fail(CRP_ERR_STATE, "genome already committed");
    if (!token_ascii && token_len) return fail(CRP_ERR_ARG, "token_ascii is NULL");
    if (seg_begin > seg_end || seg_end > token_len)
        return fail(CRP_ERR_ARG, "segment [%llu,%llu) outside token of length %llu",
                    (unsigned long long)seg_begin, (unsigned long long)seg_end, (unsigned long long)token_len);
    if (seg_begin % kAlign) return fail(CRP_ERR_ARG, "seg_begin must be a multiple of %u", kAlign);
    if (token_len >= (1ull << 31) - (1ull << 15))
        return fail(CRP_ERR_RANGE, "token of %llu positions exceeds the 31-bit position range",
                    (unsigned long long)token_len);
    Segment s{};
    s.token_id = token_id;
    s.token = token_ascii;
    s.token_len = token_len;
    s.begin = seg_begin;
    s.end = seg_end;
    g->segs.push_back(s);
    return 0;
}

int crp_genome_add_fasta_record(crp_genome *g, uint32_t token_id, const uint8_t *seq_bytes, uint64_t n_bytes,
                                uint32_t line_width, int last_record) {
    if (!g) return fail(CRP_ERR_ARG, "g is NULL");
    if (g->committed) return fail(CRP_ERR_STATE, "genome already committed");
    if (!seq_bytes || !n_bytes || !line_width) return fail(CRP_ERR_FORMAT, "empty FASTA record");
    // bytes = bases + one line end per full line, the last one optional
    const uint64_t body = seq_bytes[n_bytes - 1] == '\n' ? n_bytes - 1 : n_bytes;
    const uint64_t k = body / ((uint64_t)line_width + 1), r = body % ((uint64_t)line_width + 1);
    if (r == 0) return fail(CRP_ERR_FORMAT, "FASTA record is not made of %u-base lines", line_width);
    const uint64_t n_bases = k * line_width + r, token_len = n_bases + 4;
    if (token_len >= (1ull << 31) - (1ull << 15))
        return fail(CRP_ERR_RANGE, "token of %llu positions exceeds the 31-bit position range",
                    (unsigned long long)token_len);
    Segment s{};
    s.token_id = token_id;
    s.token = nullptr;
    s.token_len = token_len;
    s.begin = 0;
    s.end = token_len;
    s.raw = seq_bytes;
    s.raw_bytes = n_bytes;
    s.width = line_width;
    s.last = last_record ? 1u : 0u;
    g->segs.push_back(s);
    g->fasta = true;
    return 0;
}

int crp_genome_token_length(const crp_genome *g, uint32_t segment, uint64_t *token_len) {
    if (!g || !token_len) return fail(CRP_ERR_ARG, "NULL argument");
    if (segment >= g->segs.size()) return fail(CRP_ERR_ARG, "segment %u out of range", segment);
    *token_len = g->segs[segment].token_len;
    return 0;
}

int crp_genome_fetch_token(const crp_genome *g, uint32_t segment, uint8_t *dst, uint64_t capacity) {
    if (!g || !dst) return fail(CRP_ERR_ARG, "NULL argument");
    if (int rc = need_ctx()) return rc;
    if (!g->committed || !g->d_ascii) return fail(CRP_ERR_STATE, "the genome keeps no tokens on the device");
    if (segment >= g->segs.size()) return fail(CRP_ERR_ARG, "segment %u out of range", segment);
    const Segment &s = g->segs[segment];
    if (!s.raw) return fail(CRP_ERR_STATE, "segment %u was not ingested from FASTA bytes", segment);
    if (capacity < s.token_len) return fail(CRP_ERR_RANGE, "token needs %llu bytes", (unsigned long long)s.token_len);
    cudaStream_t st = g->st ? g->st : g_ctx.stream;
    CUDA_TRY(cudaMemcpyAsync(dst, g->d_ascii + s.ascii_off, s.token_len, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return 0;
}

int crp_genome_release_tokens(crp_genome *g) {
    if (!g) return fail(CRP_ERR_ARG, "g is NULL");
    dev_free(g->d_ascii, g->st ? g->st : g_ctx.stream);
    g->d_ascii = nullptr;
    return 0;
}

int crp_genome_num_segments(const crp_genome *g, uint32_t *n) {
    if (!g || !n) return fail(CRP_ERR_ARG, "NULL argument");
    *n = (uint32_t)g->segs.size();
    return 0;
}

int crp_genome_num_positions(const crp_genome *g, uint64_t *n) {
    if (!g || !n) return fail(CRP_ERR_ARG, "NULL argument");
    *n = g->n_positions;
    return 0;
}

// Enqueue the whole ingest of a genome on its stream: H2D of the token bytes the segments need,
// the pack kernel, release of the staging buffer.  Nothing here waits for the device.
static int commit_enqueue(crp_genome *g) {
    cudaStream_t st = stream_of(g);
    // ---- layout: every segment owns whole tile records; the bytes it needs (its positions
    // plus 32 of context each side) go to an ASCII staging buffer, 16-byte aligned per segment
    const bool one = g->segs.size() == 1;      // single segment: descriptors by arithmetic, no uploads
    std::vector<PackDesc> descs;
    std::vector<uint64_t> seg_ascii;
    std::vector<uint32_t> seg_first, seg_count;
    uint64_t ascii_bytes = 0, n_tiles = 0;
    g->n_positions = 0;
    for (size_t si = 0; si < g->segs.size(); ++si) {
        Segment &s = g->segs[si];
        s.stage_begin = s.begin >= 32 ? s.begin - 32 : 0;
        s.stage_end = s.end + 32 < s.token_len ? s.end + 32 : s.token_len;
        seg_ascii.push_back(ascii_bytes);
        s.first_tile = (uint32_t)n_tiles;
        s.n_tiles = (uint32_t)((s.end - s.begin + kTile - 1) / kTile);
        n_tiles += s.n_tiles;
        if (n_tiles >= (1ull << 31)) return fail(CRP_ERR_RANGE, "shard has too many tiles");
        for (uint32_t j = 0; j < (one ? (s.n_tiles ? 1u : 0u) : s.n_tiles); ++j) {
            const uint64_t t = s.begin + (uint64_t)j * kTile;
            PackDesc pd;
            pd.ascii_off = ascii_bytes;
            pd.stage_begin = (uint32_t)s.stage_begin;
            pd.stage_end = (uint32_t)s.stage_end;
            pd.td.t_start = (uint32_t)t;
            pd.td.L = (uint32_t)s.token_len;
            pd.td.n = (uint32_t)((s.end - t) < (uint64_t)kTile ? (s.end - t) : (uint64_t)kTile);
            pd.td.segment = (uint32_t)si;
            descs.push_back(pd);
        }
        seg_first.push_back(s.first_tile);
        seg_count.push_back(s.n_tiles);
        g->n_positions += s.end - s.begin;
        ascii_bytes += (s.stage_end - s.stage_begin + 15) / 16 * 16;
    }
    if (g->n_positions >= (1ull << 32))
        return fail(CRP_ERR_RANGE, "shard of %llu positions exceeds the 32-bit candidate count range",
                    (unsigned long long)g->n_positions);
    g->n_tiles = (uint32_t)n_tiles;
    g_perf.commits++;
    g_perf.positions += g->n_positions;
    g_perf.h2d_bytes += ascii_bytes;

    uint8_t *d_ascii = nullptr;
    PackDesc *d_descs = nullptr;
    const size_t rec_bytes = (size_t)g->n_tiles * kRecBytes;
    if (dev_alloc(&d_ascii, ascii_bytes + 64, st) != cudaSuccess ||
        (!one && dev_alloc(&d_descs, (descs.size() + 1) * sizeof(PackDesc), st) != cudaSuccess) ||
        dev_alloc(&g->records, rec_bytes + 16, st) != cudaSuccess ||
        dev_alloc(&g->pam, (size_t)g->n_tiles * kPamBytes + 16, st) != cudaSuccess ||
        dev_alloc(&g->hdr, ((size_t)g->n_tiles + 1) * sizeof(TileHdr), st) != cudaSuccess) {
        cudaGetLastError();
        dev_free(d_ascii, st);
        dev_free(d_descs, st);
        return fail(CRP_ERR_NOMEM, "cudaMalloc of %llu record bytes + %llu staging bytes failed",
                    (unsigned long long)rec_bytes, (unsigned long long)ascii_bytes);
    }
    for (int i = 0; i < 3; ++i)
        if (!g->ev[i]) CUDA_TRY(cudaEventCreate(&g->ev[i]));
    CUDA_TRY(cudaEventRecord(g->ev[0], st));
    uint8_t *d_raw = nullptr;
    FastaRec *d_recs = nullptr;
    unsigned int *d_bad = nullptr;
    std::vector<FastaRec> frecs;
    uint64_t raw_total = 0, strip_items = 0;
    for (size_t si = 0; si < g->segs.size(); ++si) {
        Segment &s = g->segs[si];
        s.ascii_off = seg_ascii[si];
        if (!s.raw) continue;
        FastaRec fr{};
        fr.raw_off = raw_total;
        fr.ascii_off = seg_ascii[si];
        fr.first_item = strip_items;
        fr.n_bases = (uint32_t)(s.token_len - 4);
        fr.width = s.width;
        fr.last = s.last;
        frecs.push_back(fr);
        raw_total += (s.raw_bytes + 15) / 16 * 16;
        strip_items += (s.token_len + 15) / 16;
    }
    if (!frecs.empty()) {
        if (dev_alloc(&d_raw, raw_total + 64, st) != cudaSuccess ||
            dev_alloc(&d_recs, frecs.size() * sizeof(FastaRec), st) != cudaSuccess ||
            dev_alloc(&d_bad, sizeof(unsigned int), st) != cudaSuccess) {
            cudaGetLastError();
            return fail(CRP_ERR_NOMEM, "cudaMalloc of %llu FASTA bytes failed", (unsigned long long)raw_total);
        }
        CUDA_TRY(cudaMemsetAsync(d_bad, 0, sizeof(unsigned int), st));
    }
    for (size_t si = 0, fi = 0; si < g->segs.size(); ++si) {
        const Segment &s = g->segs[si];
        if (s.raw) {
            CUDA_TRY(cudaMemcpyAsync(d_raw + frecs[fi++].raw_off, s.raw, s.raw_bytes, cudaMemcpyHostToDevice, st));
        } else if (s.stage_end > s.stage_begin && s.n_tiles) {
            CUDA_TRY(cudaMemcpyAsync(d_ascii + seg_ascii[si], s.token + s.stage_begin, s.stage_end - s.stage_begin,
                                     cudaMemcpyHostToDevice, st));
        }
    }
    if (!frecs.empty()) {
        CUDA_TRY(cudaMemcpyAsync(d_recs, frecs.data(), frecs.size() * sizeof(FastaRec), cudaMemcpyHostToDevice, st));
        const uint64_t want = (strip_items + 255) / 256, cap = (uint64_t)g_ctx.sm_count * 16;
        k_fasta_strip<<<(unsigned)(want < cap ? want : cap), 256, 0, st>>>(d_raw, d_recs, (uint32_t)frecs.size(),
                                                                           strip_items, d_ascii, d_bad);
        g_ctx.launches++;
        CUDA_TRY(cudaGetLastError());
        if (!g->h_bad) g->h_bad = static_cast<unsigned int *>(pinned_get(sizeof(unsigned int)));
        if (!g->h_bad) return fail(CRP_ERR_NOMEM, "cudaHostAlloc failed");
        *g->h_bad = 0;
        CUDA_TRY(cudaMemcpyAsync(g->h_bad, d_bad, sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
        dev_free(d_raw, st);
        dev_free(d_recs, st);
        dev_free(d_bad, st);
    }
    if (!one && !descs.empty())
        CUDA_TRY(cudaMemcpyAsync(d_descs, descs.data(), descs.size() * sizeof(PackDesc), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaEventRecord(g->ev[1], st));
    const uint64_t n_items = (uint64_t)g->n_tiles * kPackItems;
    if (n_items) {
        PackDesc first = descs[0];
        if (one) first.td.n = (uint32_t)(g->segs[0].end - g->segs[0].begin);     // positions of the whole segment
        const uint64_t want = (n_items + 255) / 256, cap = (uint64_t)g_ctx.sm_count * 16;
        CUDA_TRY(cudaMemsetAsync(g->hdr, 0, (size_t)g->n_tiles * sizeof(TileHdr), st));      // chunk counts are accumulated
        k_pack<<<(unsigned)(want < cap ? want : cap), 256, 0, st>>>(d_ascii, d_descs, first, n_items, g->records, g->pam, g->hdr);
        g_ctx.launches++;
        CUDA_TRY(cudaGetLastError());
    }
    CUDA_TRY(cudaEventRecord(g->ev[2], st));
    if (!one && !g->segs.empty()) {
        const size_t nb = g->segs.size() * sizeof(uint32_t);
        CUDA_TRY(dev_alloc(&g->d_seg_first, nb, st));
        CUDA_TRY(dev_alloc(&g->d_seg_count, nb, st));
        CUDA_TRY(cudaMemcpyAsync(g->d_seg_first, seg_first.data(), nb, cudaMemcpyHostToDevice, st));
        CUDA_TRY(cudaMemcpyAsync(g->d_seg_count, seg_count.data(), nb, cudaMemcpyHostToDevice, st));
    }
    if (g->fasta) g->d_ascii = d_ascii;   // kept: the host fetches the tokens it formats rows from
    else dev_free(d_ascii, st);           // stream ordered: after the pack kernel
    dev_free(d_descs, st);
    g->committed = true;
    return 0;
}

int crp_genome_commit(crp_genome *g) {
    if (!g) return fail(CRP_ERR_ARG, "g is NULL");
    if (int rc = need_ctx()) return rc;
    if (g->committed) return fail(CRP_ERR_STATE, "genome already committed");
    Trace tr("commit");
    if (int rc = commit_enqueue(g)) return rc;
    tr.lap("enqueue");
    CUDA_TRY(cudaStreamSynchronize(stream_of(g)));
    tr.lap("sync");
    CUDA_TRY(cudaEventElapsedTime(&g->ms_h2d, g->ev[0], g->ev[1]));
    CUDA_TRY(cudaEventElapsedTime(&g->ms_pack, g->ev[1], g->ev[2]));
    g_perf.ms_h2d += g->ms_h2d;
    g_perf.ms_pack += g->ms_pack;
    for (Segment &s : g->segs) s.token = nullptr;   // host tokens may be released now
    if (g->h_bad && *g->h_bad)
        return fail(CRP_ERR_FORMAT, "a FASTA record is not plain fixed-width text; use the host ingest for this file");
    return 0;
}

int crp_genome_timing(const crp_genome *g, float *ms_h2d, float *ms_pack) {
    if (!g) return fail(CRP_ERR_ARG, "g is NULL");
    if (ms_h2d) *ms_h2d = g->ms_h2d;
    if (ms_pack) *ms_pack = g->ms_pack;
    return 0;
}

int crp_genome_free(crp_genome *g) {
    if (!g) return 0;
    cudaStream_t st = stream_of(g);
    dev_free(g->records, st);
    dev_free(g->pam, st);
    dev_free(g->hdr, st);
    dev_free(g->d_ascii, st);
    pinned_put(g->h_bad);
    dev_free(g->d_seg_first, st);
    dev_free(g->d_seg_count, st);
    for (cudaEvent_t e : g->ev)
        if (e) cudaEventDestroy(e);
    delete g;
    return 0;
}

static void free_streams(crp_result *r) {
    for (int s = 0; s < 2; ++s) {
        dev_free(r->pos[s], r->st);
        dev_free(r->packed[s], r->st);
        dev_free(r->x[s], r->st);
        r->pos[s] = nullptr;
        r->packed[s] = nullptr;
        r->x[s] = nullptr;
    }
}

static int alloc_streams(crp_result *r, uint64_t cap, bool scored) {
    r->capacity = cap;
    const uint64_t n = cap ? cap : 1;
    for (int s = 0; s < 2; ++s) {
        if (dev_alloc(&r->pos[s], n * sizeof(uint32_t), r->st) != cudaSuccess) goto oom;
        if (scored) {
            if (dev_alloc(&r->packed[s], n * sizeof(unsigned long long), r->st) != cudaSuccess) goto oom;
            if (dev_alloc(&r->x[s], n * sizeof(double), r->st) != cudaSuccess) goto oom;
        }
    }
    return 0;
oom:
    cudaGetLastError();
    free_streams(r);
    return fail(CRP_ERR_NOMEM, "cudaMalloc of candidate streams (%llu entries per strand) failed",
                (unsigned long long)cap);
}

// Launch geometry of the cooperative scan kernel for a genome of n_tiles tiles.
struct ScanPlan {
    const void *fn;
    unsigned grid, threads;
    size_t smem;
};

static int plan_scan(const crp_genome *g, bool scored, ScanPlan *p) {
    p->threads = kThreads;
    p->fn = scored ? (const void *)k_scan_score<true> : (const void *)k_scan_score<false>;
    const unsigned grid_max = (unsigned)g_ctx.sm_count * CRP_CTAS_PER_SM;
    p->smem = kScanSmemFixed + (size_t)grid_max * sizeof(unsigned long long);
    static_assert(kScanSmemFixed >= (size_t)kHdrBatch * sizeof(TileHdr), "the count phase stages its tile headers in the emit phase's tile slots");
    static int per_sm_cache[2] = {0, 0};       // occupancy of the two instantiations, queried once
    int &per_sm = per_sm_cache[scored ? 1 : 0];
    if (per_sm == 0) {
        CUDA_TRY(cudaFuncSetAttribute(p->fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)p->smem));
        CUDA_TRY(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, p->fn, kThreads, p->smem));
        if (per_sm < 1) return fail(CRP_ERR_CUDA, "scan kernel does not fit on an SM");
        if (per_sm > CRP_CTAS_PER_SM) per_sm = CRP_CTAS_PER_SM;
    }
    // persistent grid, every CTA resident (grid barrier between the count and emit phases)
    uint64_t grid = (uint64_t)g_ctx.sm_count * per_sm;
    if (const char *e = getenv("CRP_SCAN_GRID")) {       // tests: few CTAs give long count ranges on small inputs
        const long v = atol(e);
        if (v > 0 && (uint64_t)v < grid) grid = (uint64_t)v;
    }
    if (grid > g->n_tiles) grid = g->n_tiles;
    if (grid < 1) grid = 1;
    p->grid = (unsigned)grid;
    return 0;
}

static int launch_scan(const crp_genome *g, crp_result *r, const ScanPlan &p) {
    cudaStream_t st = r->st;
    ScanArgs a;
    a.records = g->records;
    a.pam = g->pam;
    a.hdr = g->hdr;
    a.n_tiles = g->n_tiles;
    a.static_eighths = 4;
    if (const char *e = getenv("CRP_STATIC_EIGHTHS")) a.static_eighths = (uint32_t)atoi(e) > 8 ? 8 : (uint32_t)atoi(e);
    a.guide_len = r->guide_len;
    a.flags = r->flags;
    a.tables = g_ctx.d_tables;
    a.capacity = r->capacity < 0xFFFFFFFFull ? r->capacity : 0xFFFFFFFFull;   // rows are 32-bit in the kernel (counts are packed 32 | 32)
    a.pos_plus = r->pos[0];
    a.pos_minus = r->pos[1];
    a.packed_plus = r->packed[0];
    a.packed_minus = r->packed[1];
    a.x_plus = r->x[0];
    a.x_minus = r->x[1];
    const uint32_t n_seg = (uint32_t)g->segs.size();
    unsigned long long *s64 = reinterpret_cast<unsigned long long *>(r->state);
    a.warp_pref = s64;
    a.cta_tot = s64 + (size_t)g->n_tiles * kPrefWords;
    a.seg_counts = r->d_counts;
    a.tickets = reinterpret_cast<unsigned int *>(r->d_counts + 2 * (size_t)r->stride);
    a.n_seg = n_seg;
    a.seg_stride = r->stride;
    a.seg_first_tile = g->d_seg_first;      // NULL for a single-segment genome
    a.seg_tile_count = g->d_seg_count;
    a.seg_counts_host = r->h_counts;        // mapped pinned memory: the kernel stores the counts there itself
    a.fault = g_ctx.d_fault;
    a.world = 1;
    a.rank = 0;
    a.epoch = 0;
    a.xchg_error = nullptr;
    a.xchg_timeout_ns = 20ull * 1000 * 1000 * 1000;
    for (int q = 0; q < kMaxPeers; ++q) {
        a.peer_gather[q] = nullptr;
        a.peer_flags[q] = nullptr;
    }
    const unsigned long long *gathered = r->d_gather;       // where the blocks of all ranks end up
    if (r->fused) {
        // Fused exchange: the kernel stores this rank's counts into every rank's buffer right after its
        // count phase and leaves once all blocks are in its own -- no collective launch behind the kernel.
        a.world = (uint32_t)g_comm.world;
        a.rank = (uint32_t)g_comm.rank;
        a.epoch = r->epoch;
        a.xchg_error = xchg_error(g_comm.xchg);
        if (const char *e = getenv("CRP_XCHG_TIMEOUT_MS")) a.xchg_timeout_ns = strtoull(e, nullptr, 10) * 1000000ull;
        for (int q = 0; q < g_comm.world; ++q) {
            a.peer_gather[q] = xchg_gather(g_comm.peer[q], r->epoch & 1u, a.world, r->stride);
            a.peer_flags[q] = xchg_flags(g_comm.peer[q], r->epoch & 1u);
        }
        gathered = xchg_gather(g_comm.xchg, r->epoch & 1u, a.world, r->stride);
    }
    CUDA_TRY(cudaEventRecord(r->ev[0], st));
    if (g->n_tiles) {
        void *params[] = {(void *)&a};
        CUDA_TRY(cudaLaunchCooperativeKernel(p.fn, dim3(p.grid), dim3(p.threads), params, p.smem, st));
        g_ctx.launches++;
        CUDA_TRY(cudaGetLastError());
    } else if (r->fused) {
        k_exchange_empty<<<1, 256, 0, st>>>(a);
        g_ctx.launches++;
        CUDA_TRY(cudaGetLastError());
    } else if (r->stride) {
        CUDA_TRY(cudaMemsetAsync(r->d_counts, 0, 2 * (size_t)r->stride * sizeof(unsigned long long), st));
        memset(r->h_counts, 0, 2 * (size_t)r->stride * sizeof(unsigned long long));
    }
    if (r->ev_kernel) CUDA_TRY(cudaEventRecord(r->ev_kernel, st));
    if (r->d_gather && !r->fused) {
        // NCCL exchange: every rank's per-segment counts to every rank, right behind the kernel on the
        // same stream, so the CUDA events bracket kernel + collective
        if (int rc = comm_allgather_u64(r->d_counts, r->d_gather, 2 * (size_t)r->stride, st)) return rc;
    }
    CUDA_TRY(cudaEventRecord(r->ev[1], st));
    // (the per-segment counts are already in r->h_counts: the kernel stored them into mapped host memory)
    if (r->h_gather && gathered)
        CUDA_TRY(cudaMemcpyAsync(r->h_gather, gathered, (size_t)g_comm.world * 2 * r->stride * sizeof(unsigned long long),
                                 cudaMemcpyDeviceToHost, st));
    if (r->fused)
        CUDA_TRY(cudaMemcpyAsync(r->h_xchg_error, xchg_error(g_comm.xchg), sizeof(unsigned int), cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaEventRecord(r->ev[2], st));
    return 0;
}

// Allocate the result of a scan and enqueue the scan on the genome's stream (no waiting).
static int scan_enqueue(crp_genome *g, int guide_len, uint32_t flags, crp_result **res, uint32_t slots = 0) {
    crp_result *r = new (std::nothrow) crp_result();
    if (!r) return fail(CRP_ERR_NOMEM, "out of host memory");
    r->g = g;
    r->st = stream_of(g);
    r->guide_len = guide_len;
    r->flags = flags;
    r->scored = guide_len == 20 && !(flags & CRP_SCAN_NO_SCORE);
    const uint32_t n_seg = (uint32_t)g->segs.size();
    int rc = 0;
    auto bail = [&](int code) {
        crp_result_free(r);
        return code;
    };
    ScanPlan plan = {};
    if ((rc = plan_scan(g, r->scored, &plan))) return bail(rc);
    r->stride = slots ? slots : n_seg;
    r->zero_offset = ((size_t)g->n_tiles * kPrefWords + (size_t)plan.grid) * sizeof(unsigned long long);
    r->state_bytes = r->zero_offset + 2 * (size_t)r->stride * sizeof(unsigned long long) +
                     4 * sizeof(unsigned int);
    if (dev_alloc(&r->state, r->state_bytes, r->st) != cudaSuccess)
        return bail(fail(CRP_ERR_NOMEM, "cudaMalloc of scan state failed"));
    r->d_counts = reinterpret_cast<unsigned long long *>(r->state + r->zero_offset);
    r->h_counts = static_cast<unsigned long long *>(pinned_get((2 * (size_t)r->stride + 1) * sizeof(unsigned long long)));
    if (!r->h_counts) return bail(fail(CRP_ERR_NOMEM, "cudaHostAlloc of the counts failed"));
    if (slots) {
        const size_t gb = (size_t)g_comm.world * 2 * slots * sizeof(unsigned long long);
        r->fused = g_comm.fused && g_comm.mode == 0 && slots <= kXchgSlots;
        r->epoch = ++g_comm.epoch;
        if (r->fused) {
            r->h_xchg_error = static_cast<unsigned int *>(pinned_get(sizeof(unsigned int)));
            if (!r->h_xchg_error) return bail(fail(CRP_ERR_NOMEM, "cudaHostAlloc failed"));
            *r->h_xchg_error = 0;
        }
        if (dev_alloc(&r->d_gather, gb, r->st) != cudaSuccess)
            return bail(fail(CRP_ERR_NOMEM, "cudaMalloc of the gathered counts failed"));
        r->h_gather = static_cast<unsigned long long *>(pinned_get(gb));
        if (!r->h_gather) return bail(fail(CRP_ERR_NOMEM, "cudaHostAlloc of the gathered counts failed"));
        if (cudaEventCreate(&r->ev_kernel) != cudaSuccess) return bail(fail(CRP_ERR_CUDA, "cudaEventCreate failed"));
    }
    if (cudaEventCreate(&r->ev[0]) != cudaSuccess || cudaEventCreate(&r->ev[1]) != cudaSuccess ||
        cudaEventCreateWithFlags(&r->ev[2], cudaEventDisableTiming) != cudaSuccess)
        return bail(fail(CRP_ERR_CUDA, "cudaEventCreate failed"));
    // First guess of the per-strand capacity: 1/8 candidate per position (GC 70 %
    // upper-case sequence gives 0.1225); a second pass with the exact counts
    // follows if it was too small.
    if ((rc = alloc_streams(r, g->n_positions / 8 + 4096, r->scored))) return bail(rc);
    if ((rc = launch_scan(g, r, plan))) return bail(rc);
    *res = r;
    return 0;
}

// Wait for the scan, read the counts; run it again with exact capacity if the guess was short.
static int scan_finish(crp_genome *g, crp_result *r, cudaStream_t post = nullptr) {
    // post: the stream the caller will read the rows on (crp_scan_segments: its row-copy stream).  The
    // optional logistic pass goes there -- the genome's own stream may already hold the H2D, pack and
    // scan of later segments, and a pass queued behind them would hold this segment's rows back.
    const uint32_t n_seg = (uint32_t)g->segs.size();
    for (int attempt = 0; attempt < 2; ++attempt) {
        if (cudaError_t e = cudaEventSynchronize(r->ev[2]))   // not the stream: it may already hold later segments
            return fail(CRP_ERR_CUDA, "scan kernels failed: %s", cudaGetErrorString(e));
        r->n_plus = r->n_minus = 0;
        r->seg_plus.assign(n_seg, 0);
        r->seg_minus.assign(n_seg, 0);
        for (uint32_t s = 0; s < n_seg; ++s) {
            r->seg_plus[s] = r->h_counts[s];
            r->seg_minus[s] = r->h_counts[r->stride + s];
            r->n_plus += r->seg_plus[s];
            r->n_minus += r->seg_minus[s];
        }
        {
            float ms = 0.f;
            cudaEventElapsedTime(&ms, r->ev[0], r->ev[1]);
            r->ms_scan += ms;
            if (r->ev_kernel) cudaEventElapsedTime(&ms, r->ev[0], r->ev_kernel);
            r->ms_kernel += ms;
            r->n_launches++;
        }
#ifdef CRP_CHECKED
        {
            unsigned int fault = 0;
            cudaMemcpy(&fault, g_ctx.d_fault, sizeof fault, cudaMemcpyDeviceToHost);
            if (fault) {
                cudaMemset(g_ctx.d_fault, 0, sizeof fault);
                return fail(CRP_ERR_STATE, "checked build: kernel invariant %u violated (scan.cuh:%u)", fault & 0xFFu, fault >> 8);
            }
        }
#endif
        if (r->fused && *r->h_xchg_error)
            return fail(CRP_ERR_CUDA, "sharded scan: the counts of rank %u did not arrive (peer not scanning?)", *r->h_xchg_error - 1);
        const uint64_t need = r->n_plus > r->n_minus ? r->n_plus : r->n_minus;
        if (need <= r->capacity) break;
        if (attempt == 1) return fail(CRP_ERR_STATE, "candidate streams overflowed twice");
        // the rerun is local: the counts are already exchanged, the second launch only fills the streams
        r->fused = false;
        if (r->d_gather) {
            dev_free(r->d_gather, r->st);
            r->d_gather = nullptr;               // keeps h_gather of the first launch
        }
        free_streams(r);
        if (int rc = alloc_streams(r, need, r->scored)) return rc;
        ScanPlan plan = {};
        if (int rc = plan_scan(g, r->scored, &plan)) return rc;
        if (int rc = launch_scan(g, r, plan)) return rc;
    }
    g_perf.scans++;
    if (r->stride != (uint32_t)g->segs.size() || r->h_gather) g_perf.sharded_scans++;
    if (r->epoch && g_comm.fused && g_comm.mode == 0) g_perf.fused_exchanges++;
    g_perf.capacity_reruns += r->n_launches - 1;
    g_perf.candidates += r->n_plus + r->n_minus;
    g_perf.ms_scan += r->ms_scan;
    g_perf.ms_kernel += r->ms_kernel;
    if (r->scored && (r->flags & CRP_SCAN_LOGISTIC)) {
        const uint64_t n[2] = {r->n_plus, r->n_minus};
        for (int s = 0; s < 2; ++s)
            if (n[s]) {
                const uint64_t want = (n[s] + 255) / 256, cap = (uint64_t)g_ctx.sm_count * 16;
                k_logistic<<<(unsigned)(want < cap ? want : cap), 256, 0, post ? post : r->st>>>(r->x[s], n[s]);
                g_ctx.launches++;
            }
        CUDA_TRY(cudaGetLastError());
        // whoever reads the streams from yet another stream orders itself after this event
        CUDA_TRY(cudaEventRecord(r->ev[2], post ? post : r->st));
    }
    return 0;
}

int crp_scan_score(crp_genome *g, int guide_len, uint32_t flags, crp_result **res) {
    if (!g || !res) return fail(CRP_ERR_ARG, "NULL argument");
    if (int rc = need_ctx()) return rc;
    if (!g->committed) return fail(CRP_ERR_STATE, "genome not committed");
    if (guide_len < 1 || guide_len > 1000000) return fail(CRP_ERR_ARG, "guide_len %d out of range", guide_len);
    Trace tr("scan");
    crp_result *r = nullptr;
    if (int rc = scan_enqueue(g, guide_len, flags, &r)) return rc;
    tr.lap("enqueue");
    if (int rc = scan_finish(g, r)) {
        crp_result_free(r);
        return rc;
    }
    tr.lap("finish");
    *res = r;
    return 0;
}

int crp_scan_score_sharded(crp_genome *g, int guide_len, uint32_t flags, uint32_t slots, crp_result **res) {
    if (!g || !res) return fail(CRP_ERR_ARG, "NULL argument");
    if (int rc = need_ctx()) return rc;
    if (!g_comm.comm) return fail(CRP_ERR_STATE, "crp_comm_init has not been called");
    if (!g->committed) return fail(CRP_ERR_STATE, "genome not committed");
    if (guide_len < 1 || guide_len > 1000000) return fail(CRP_ERR_ARG, "guide_len %d out of range", guide_len);
    if (slots == 0 || slots < g->segs.size())
        return fail(CRP_ERR_ARG, "slots = %u is smaller than the %zu segments of this shard", slots, g->segs.size());
    crp_result *r = nullptr;
    if (int rc = scan_enqueue(g, guide_len, flags, &r, slots)) return rc;
    if (int rc = scan_finish(g, r)) {
        crp_result_free(r);
        return rc;
    }
    *res = r;
    return 0;
}

int crp_result_gathered_counts(const crp_result *res, uint64_t *counts) {
    if (!res || !counts) return fail(CRP_ERR_ARG, "NULL argument");
    if (!res->h_gather) return fail(CRP_ERR_STATE, "not the result of a sharded scan");
    memcpy(counts, res->h_gather, (size_t)g_comm.world * 2 * res->stride * sizeof(uint64_t));
    return 0;
}

static int rs1_rows(uint64_t n, const uint8_t *rows, const uint8_t *cls, double *score, int logistic);
int crp_rs1_score(uint64_t n, const uint8_t *rows, const uint8_t *cls, double *score) {
    return rs1_rows(n, rows, cls, score, 1);
}
int crp_rs1_preactivation(uint64_t n, const uint8_t *rows, const uint8_t *cls, double *x) {
    return rs1_rows(n, rows, cls, x, 0);
}
static int rs1_rows(uint64_t n, const uint8_t *rows, const uint8_t *cls, double *score, int logistic) {
    if (n && (!rows || !cls || !score)) return fail(CRP_ERR_ARG, "NULL argument");
    if (int rc = need_ctx()) return rc;
    if (!n) return 0;
    cudaStream_t st = g_ctx.stream;
    uint8_t *d_rows = nullptr;
    double *d_out = nullptr;
    if (dev_alloc(&d_rows, 31 * n, st) != cudaSuccess || dev_alloc(&d_out, n * sizeof(double), st) != cudaSuccess) {
        cudaGetLastError();
        dev_free(d_rows, st);
        return fail(CRP_ERR_NOMEM, "cudaMalloc for %llu rows failed", (unsigned long long)n);
    }
    CUDA_TRY(cudaMemcpyAsync(d_rows, rows, 30 * n, cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(d_rows + 30 * n, cls, n, cudaMemcpyHostToDevice, st));
    k_rs1_rows<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(d_rows, d_rows + 30 * n, n, d_out, logistic);
    g_ctx.launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(score, d_out, n * sizeof(double), cudaMemcpyDeviceToHost, st));
    dev_free(d_rows, st);
    dev_free(d_out, st);
    CUDA_TRY(cudaStreamSynchronize(st));
    return 0;
}

int crp_logistic(uint64_t n, const double *x, double *score) {
    if (n && (!x || !score)) return fail(CRP_ERR_ARG, "NULL argument");
    if (int rc = need_ctx()) return rc;
    if (!n) return 0;
    cudaStream_t st = g_ctx.stream;
    double *d = nullptr;
    if (dev_alloc(&d, n * sizeof(double), st) != cudaSuccess) {
        cudaGetLastError();
        return fail(CRP_ERR_NOMEM, "cudaMalloc of %llu doubles failed", (unsigned long long)n);
    }
    CUDA_TRY(cudaMemcpyAsync(d, x, n * sizeof(double), cudaMemcpyHostToDevice, st));
    const uint64_t want = (n + 255) / 256, cap = (uint64_t)g_ctx.sm_count * 16;
    k_logistic<<<(unsigned)(want < cap ? want : cap), 256, 0, st>>>(d, n);
    g_ctx.launches++;
    CUDA_TRY(cudaGetLastError());
    CUDA_TRY(cudaMemcpyAsync(score, d, n * sizeof(double), cudaMemcpyDeviceToHost, st));
    dev_free(d, st);
    CUDA_TRY(cudaStreamSynchronize(st));
    return 0;
}

int crp_result_totals(const crp_result *res, uint64_t *n_plus, uint64_t *n_minus) {
    if (!res) return fail(CRP_ERR_ARG, "res is NULL");
    if (n_plus) *n_plus = res->n_plus;
    if (n_minus) *n_minus = res->n_minus;
    return 0;
}

int crp_result_segment_counts(const crp_result *res, uint64_t *n_plus, uint64_t *n_minus) {
    if (!res) return fail(CRP_ERR_ARG, "res is NULL");
    for (size_t s = 0; s < res->seg_plus.size(); ++s) {
        if (n_plus) n_plus[s] = res->seg_plus[s];
        if (n_minus) n_minus[s] = res->seg_minus[s];
    }
    return 0;
}

int crp_result_device_counts(const crp_result *res, void **dev_ptr) {
    if (!res || !dev_ptr) return fail(CRP_ERR_ARG, "NULL argument");
    *dev_ptr = res->d_counts;
    return 0;
}

// D2H of rows [first, first + count) of one strand stream, enqueued on the result's stream
static int fetch_enqueue(const crp_result *res, int s, uint64_t first, uint64_t count, uint32_t *pos, uint64_t *packed,
                         double *x, cudaStream_t st = nullptr) {
    if (!st) st = res->st;
    g_perf.d2h_bytes += count * ((pos ? 4 : 0) + (packed ? 8 : 0) + (x ? 8 : 0));
    if (count) {
        if (pos) CUDA_TRY(cudaMemcpyAsync(pos, res->pos[s] + first, count * sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        if (packed)
            CUDA_TRY(cudaMemcpyAsync(packed, res->packed[s] + first, count * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        if (x) CUDA_TRY(cudaMemcpyAsync(x, res->x[s] + first, count * sizeof(double), cudaMemcpyDeviceToHost, st));
    }
    return 0;
}

int crp_result_fetch(const crp_result *res, char strand, uint64_t first, uint64_t count, uint32_t *pos,
                     uint64_t *packed, double *x) {
    if (!res) return fail(CRP_ERR_ARG, "res is NULL");
    if (int rc = need_ctx()) return rc;
    if (strand != '+' && strand != '-') return fail(CRP_ERR_ARG, "strand must be '+' or '-'");
    const int s = strand == '+' ? 0 : 1;
    const uint64_t total = s == 0 ? res->n_plus : res->n_minus;
    if (first > total || count > total - first)
        return fail(CRP_ERR_ARG, "range [%llu,+%llu) outside stream of %llu candidates", (unsigned long long)first,
                    (unsigned long long)count, (unsigned long long)total);
    if ((packed || x) && !res->scored && count)
        return fail(CRP_ERR_STATE, "this result carries positions only (guide_len != 20 or CRP_SCAN_NO_SCORE)");
    if (int rc = fetch_enqueue(res, s, first, count, pos, packed, x)) return rc;
    CUDA_TRY(cudaStreamSynchronize(res->st));
    return 0;
}

int crp_result_timing(const crp_result *res, float *ms_scan) {
    if (!res) return fail(CRP_ERR_ARG, "res is NULL");
    if (ms_scan) *ms_scan = res->ms_scan;
    return 0;
}

int crp_result_timing_detail(const crp_result *res, float *ms_kernels, float *ms_total, uint32_t *n_launches) {
    if (!res) return fail(CRP_ERR_ARG, "res is NULL");
    if (ms_kernels) *ms_kernels = res->ms_kernel;
    if (ms_total) *ms_total = res->ms_scan;
    if (n_launches) *n_launches = res->n_launches;
    return 0;
}

int crp_result_free(crp_result *r) {
    if (!r) return 0;
    free_streams(r);
    dev_free(r->state, r->st);
    dev_free(r->d_gather, r->st);
    pinned_put(r->h_counts);
    pinned_put(r->h_gather);
    pinned_put(r->h_xchg_error);
    if (r->ev_kernel) cudaEventDestroy(r->ev_kernel);
    for (cudaEvent_t e : r->ev)
        if (e) cudaEventDestroy(e);
    delete r;
    return 0;
}

// ------------------------------------------------------------------ pipelined whole-call path
// Segments in, candidate arrays out, host memory on both sides: segment k+1 is copied in and
// packed while segment k is scanned and segment k-1 is copied out (three streams, PCIe both
// ways at once).  Rows of a strand land in the caller's arena in segment order.
int crp_scan_segments(uint32_t n_segments, const crp_segment_desc *segments, int guide_len, uint32_t flags,
                      uint64_t capacity, uint32_t *pos_plus, uint64_t *packed_plus, double *x_plus,
                      uint32_t *pos_minus, uint64_t *packed_minus, double *x_minus, uint64_t *n_plus,
                      uint64_t *n_minus, float *ms_device) {
    if (int rc = need_ctx()) return rc;
    if (n_segments && (!segments || !n_plus || !n_minus)) return fail(CRP_ERR_ARG, "NULL argument");
    if (guide_len < 1 || guide_len > 1000000) return fail(CRP_ERR_ARG, "guide_len %d out of range", guide_len);
    const bool scored = guide_len == 20 && !(flags & CRP_SCAN_NO_SCORE);
    // every descriptor is checked before the first group is enqueued: a bad one in the middle of the
    // list must not leave the groups before it copied, packed and scanned (the rules of add_segment)
    for (uint32_t k = 0; k < n_segments; ++k) n_plus[k] = n_minus[k] = 0;
    for (uint32_t k = 0; k < n_segments; ++k) {
        const crp_segment_desc &sd = segments[k];
        if (!sd.token && sd.token_len) return fail(CRP_ERR_ARG, "segment %u: token is NULL", k);
        if (sd.begin > sd.end || sd.end > sd.token_len)
            return fail(CRP_ERR_ARG, "segment %u: [%llu,%llu) outside token of length %llu", k,
                        (unsigned long long)sd.begin, (unsigned long long)sd.end, (unsigned long long)sd.token_len);
        if (sd.begin % kAlign) return fail(CRP_ERR_ARG, "segment %u: begin must be a multiple of %u", k, kAlign);
        if (sd.token_len >= (1ull << 31) - (1ull << 15))
            return fail(CRP_ERR_ARG, "segment %u: token of %llu positions exceeds the 31-bit position range", k,
                        (unsigned long long)sd.token_len);
    }
    constexpr int kLanes = 3;
    if (!g_ctx.lanes[0])
        for (int i = 0; i < kLanes; ++i) CUDA_TRY(cudaStreamCreateWithFlags(&g_ctx.lanes[i], cudaStreamNonBlocking));
    Trace tr("scan_segments");
    // The unit of the pipeline is a GROUP of up to ~32 M positions: a longer segment is cut into pieces of
    // that size (tile-aligned: a 300 Mbp chromosome does not hold the scan back until all of it has
    // arrived), and consecutive small segments share one group -- one commit, one scan, one copy per
    // stream -- so a genome of 20,000 scaffolds costs a few hundred launches, not 20,000 commits and scans.
    // Measured on the 135 Mbp config (5 chromosomes of 21-34 Mbp): 32 M -> 3.29 ms, 16 M -> 3.73 ms,
    // 8 M -> 4.3 ms, 2 M -> 7.1 ms per call: every group costs two logistic launches and four row copies
    // on the copy-out stream (~25 us of engine latency), which finer groups multiply.
    uint64_t piece_bytes = 32ull << 20;
    if (const char *e = getenv("CRP_PIECE_POSITIONS")) {
        const unsigned long long v = strtoull(e, nullptr, 10);
        if (v >= (unsigned long long)kTile) piece_bytes = v / kTile * kTile;
    }
    struct Piece {
        uint32_t seg;              // index of the caller's segment
        uint64_t begin, end;
    };
    std::vector<Piece> pieces;
    for (uint32_t k = 0; k < n_segments; ++k) {
        const uint64_t end = segments[k].end;
        uint64_t b0 = segments[k].begin;
        if (end <= b0) {
            pieces.push_back(Piece{k, b0, end});
            continue;
        }
        while (b0 < end) {
            uint64_t e0 = b0 + piece_bytes;
            if (e0 + piece_bytes / 4 >= end) e0 = end;       // no crumb at the end
            pieces.push_back(Piece{k, b0, e0});
            b0 = e0;
        }
    }
    struct Group {
        uint32_t first, count;     // pieces
        uint64_t bytes;
    };
    std::vector<Group> groups;
    for (uint32_t k = 0; k < (uint32_t)pieces.size(); ++k) {
        const uint64_t nb = pieces[k].end > pieces[k].begin ? pieces[k].end - pieces[k].begin : 0;
        if (groups.empty() || groups.back().bytes + nb > piece_bytes + piece_bytes / 4 || groups.back().count >= 4096)
            groups.push_back(Group{k, 0, 0});
        groups.back().count++;
        groups.back().bytes += nb;
    }
    const uint32_t n_groups = (uint32_t)groups.size();
    std::vector<crp_genome *> gs(n_groups, nullptr);
    std::vector<crp_result *> rs(n_groups, nullptr);
    int rc = 0;
    uint64_t off[2] = {0, 0};
    float ms = 0.f;
    bool overflow = false;
    // Groups are enqueued AHEAD of the one whose counts the host waits for (its rows can only be
    // placed once the counts of every earlier group are known): up to kAheadBytes of tokens, at
    // least two groups, so that the host-to-device copy engine always has the next token queued.
    // The rows leave on a stream of their own: a lane may already hold later groups.
    constexpr uint64_t kAheadBytes = 512ull << 20;
    if (!g_ctx.lane_out) CUDA_TRY(cudaStreamCreateWithFlags(&g_ctx.lane_out, cudaStreamNonBlocking));
    auto finish = [&](uint32_t q) -> int {
        if (int e = scan_finish(gs[q], rs[q], g_ctx.lane_out)) return e;
        for (uint32_t j = 0; j < groups[q].count; ++j) {
            n_plus[pieces[groups[q].first + j].seg] += rs[q]->seg_plus[j];
            n_minus[pieces[groups[q].first + j].seg] += rs[q]->seg_minus[j];
        }
        ms += rs[q]->ms_scan;
        if (off[0] + rs[q]->n_plus > capacity || off[1] + rs[q]->n_minus > capacity) {
            overflow = true;        // keep counting so that the caller learns the capacity it needs
        } else {
            // the rows leave on lane_out: after everything scan_finish queued (the logistic pass)
            if (cudaError_t e = cudaStreamWaitEvent(g_ctx.lane_out, rs[q]->ev[2], 0))
                return fail(CRP_ERR_CUDA, "cudaStreamWaitEvent failed: %s", cudaGetErrorString(e));
            if (int e = fetch_enqueue(rs[q], 0, 0, rs[q]->n_plus, pos_plus ? pos_plus + off[0] : nullptr,
                                      scored && packed_plus ? packed_plus + off[0] : nullptr,
                                      scored && x_plus ? x_plus + off[0] : nullptr, g_ctx.lane_out)) return e;
            if (int e = fetch_enqueue(rs[q], 1, 0, rs[q]->n_minus, pos_minus ? pos_minus + off[1] : nullptr,
                                      scored && packed_minus ? packed_minus + off[1] : nullptr,
                                      scored && x_minus ? x_minus + off[1] : nullptr, g_ctx.lane_out)) return e;
        }
        off[0] += rs[q]->n_plus;
        off[1] += rs[q]->n_minus;
        return 0;
    };
    auto enqueue = [&](uint32_t q) -> int {
        if (int e = crp_genome_new(&gs[q])) return e;
        gs[q]->st = g_ctx.lanes[q % kLanes];
        for (uint32_t j = 0; j < groups[q].count; ++j) {
            const Piece &pc = pieces[groups[q].first + j];
            const crp_segment_desc &sd = segments[pc.seg];
            if (int e = crp_genome_add_segment(gs[q], sd.token_id, sd.token, sd.token_len, pc.begin, pc.end)) return e;
        }
        if (int e = commit_enqueue(gs[q])) return e;
        return scan_enqueue(gs[q], guide_len, flags, &rs[q]);
    };
    uint32_t next_enq = 0;
    uint64_t ahead = 0;
    for (uint32_t q = 0; q < n_groups && !rc; ++q) {
        while (!rc && next_enq < n_groups && (next_enq < q + 2 || ahead + groups[next_enq].bytes <= kAheadBytes)) {
            rc = enqueue(next_enq);
            ahead += groups[next_enq].bytes;
            ++next_enq;
        }
        tr.lap("enqueue");
        if (!rc) rc = finish(q);
        ahead -= groups[q].bytes;
        tr.lap("finish");
    }
    for (int i = 0; i < kLanes; ++i) cudaStreamSynchronize(g_ctx.lanes[i]);
    cudaStreamSynchronize(g_ctx.lane_out);
    tr.lap("drain");
    for (uint32_t q = 0; q < n_groups; ++q) {
        crp_result_free(rs[q]);
        crp_genome_free(gs[q]);
    }
    tr.lap("free");
    if (ms_device) *ms_device = ms;
    if (rc) return rc;
    if (overflow)
        return fail(CRP_ERR_RANGE, "arena capacity %llu rows per strand is too small: need %llu / %llu",
                    (unsigned long long)capacity, (unsigned long long)off[0], (unsigned long long)off[1]);
    return 0;
}

// rows of one segment inside a strand stream
static int segment_rows(const crp_result *res, uint32_t segment, char strand, uint64_t *first, uint64_t *count) {
    if (strand != '+' && strand != '-') return fail(CRP_ERR_ARG, "strand must be '+' or '-'");
    const std::vector<uint64_t> &c = strand == '+' ? res->seg_plus : res->seg_minus;
    if (segment >= c.size()) return fail(CRP_ERR_ARG, "segment %u out of range", segment);
    uint64_t f = 0;
    for (uint32_t s = 0; s < segment; ++s) f += c[s];
    *first = f;
    *count = c[segment];
    return 0;
}

int crp_result_extras(const crp_result *res, uint32_t segment, char strand, uint32_t flank, uint8_t *gc,
                      uint8_t *flags, uint8_t *run, uint32_t *cut, uint32_t *flank_lo, uint32_t *flank_hi) {
    if (!res) return fail(CRP_ERR_ARG, "res is NULL");
    if (int rc = need_ctx()) return rc;
    if (res->guide_len != 20) return fail(CRP_ERR_STATE, "extras are defined for guide_len 20 (30-base windows) only");
    uint64_t first = 0, n = 0;
    if (int rc = segment_rows(res, segment, strand, &first, &n)) return rc;
    if (n == 0) return 0;
    const crp_genome *g = res->g;
    const Segment &sg = g->segs[segment];
    cudaStream_t st = res->st;
    const int s = strand == '+' ? 0 : 1;
    uint8_t *d8 = nullptr;
    uint32_t *d32 = nullptr;
    CUDA_TRY(dev_alloc(&d8, 3 * n, st));
    if (dev_alloc(&d32, 3 * n * sizeof(uint32_t), st) != cudaSuccess) {
        dev_free(d8, st);
        return fail(CRP_ERR_NOMEM, "cudaMalloc failed");
    }
    ExtrasArgs a;
    a.records = g->records;
    a.pos = res->pos[s] + first;
    a.n = n;
    a.first_tile = sg.first_tile;
    a.seg_begin = (uint32_t)sg.begin;
    a.L = (uint32_t)sg.token_len;
    a.flank = flank;
    a.minus = s;
    a.gc = d8;
    a.flags = d8 + n;
    a.run = d8 + 2 * n;
    a.cut = d32;
    a.flank_lo = d32 + n;
    a.flank_hi = d32 + 2 * n;
    k_extras<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(a);
    g_ctx.launches++;
    int rc = 0;
    auto back = [&](void *dst, const void *src, size_t bytes) {
        if (dst && !rc && cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st) != cudaSuccess)
            rc = fail(CRP_ERR_CUDA, "D2H of extras failed");
    };
    back(gc, a.gc, n);
    back(flags, a.flags, n);
    back(run, a.run, n);
    back(cut, a.cut, n * 4);
    back(flank_lo, a.flank_lo, n * 4);
    back(flank_hi, a.flank_hi, n * 4);
    if (!rc && cudaStreamSynchronize(st) != cudaSuccess)
        rc = fail(CRP_ERR_CUDA, "extras kernel failed: %s", cudaGetErrorString(cudaGetLastError()));
    dev_free(d8, st);
    dev_free(d32, st);
    return rc;
}

/* The same for ALL segments of one strand stream in one call: one launch per segment queued back to
 * back, one copy per output array, one wait -- a genome of 20,000 scaffolds costs 20,000 launches, not
 * 120,000 host round trips. */
int crp_result_extras_strand(const crp_result *res, char strand, uint32_t flank, uint8_t *gc, uint8_t *flags,
                             uint8_t *run, uint32_t *cut, uint32_t *flank_lo, uint32_t *flank_hi) {
    if (!res) return fail(CRP_ERR_ARG, "res is NULL");
    if (int rc = need_ctx()) return rc;
    if (strand != '+' && strand != '-') return fail(CRP_ERR_ARG, "strand must be '+' or '-'");
    if (res->guide_len != 20) return fail(CRP_ERR_STATE, "extras are defined for guide_len 20 (30-base windows) only");
    const int s = strand == '+' ? 0 : 1;
    const uint64_t n = s == 0 ? res->n_plus : res->n_minus;
    if (n == 0) return 0;
    const crp_genome *g = res->g;
    const std::vector<uint64_t> &cnt = s == 0 ? res->seg_plus : res->seg_minus;
    cudaStream_t st = res->st;
    uint8_t *d8 = nullptr;
    uint32_t *d32 = nullptr;
    CUDA_TRY(dev_alloc(&d8, 3 * n, st));
    if (dev_alloc(&d32, 3 * n * sizeof(uint32_t), st) != cudaSuccess) {
        dev_free(d8, st);
        return fail(CRP_ERR_NOMEM, "cudaMalloc failed");
    }
    uint64_t first = 0;
    for (size_t sgi = 0; sgi < cnt.size(); ++sgi) {
        const uint64_t m = cnt[sgi];
        if (m) {
            const Segment &sg = g->segs[sgi];
            ExtrasArgs a;
            a.records = g->records;
            a.pos = res->pos[s] + first;
            a.n = m;
            a.first_tile = sg.first_tile;
            a.seg_begin = (uint32_t)sg.begin;
            a.L = (uint32_t)sg.token_len;
            a.flank = flank;
            a.minus = s;
            a.gc = d8 + first;
            a.flags = d8 + n + first;
            a.run = d8 + 2 * n + first;
            a.cut = d32 + first;
            a.flank_lo = d32 + n + first;
            a.flank_hi = d32 + 2 * n + first;
            k_extras<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(a);
            g_ctx.launches++;
        }
        first += m;
    }
    int rc = 0;
    auto back = [&](void *dst, const void *src, size_t bytes) {
        if (dst && !rc && cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st) != cudaSuccess)
            rc = fail(CRP_ERR_CUDA, "D2H of extras failed");
    };
    back(gc, d8, n);
    back(flags, d8 + n, n);
    back(run, d8 + 2 * n, n);
    back(cut, d32, n * 4);
    back(flank_lo, d32 + n, n * 4);
    back(flank_hi, d32 + 2 * n, n * 4);
    if (!rc && cudaStreamSynchronize(st) != cudaSuccess)
        rc = fail(CRP_ERR_CUDA, "extras kernels failed: %s", cudaGetErrorString(cudaGetLastError()));
    dev_free(d8, st);
    dev_free(d32, st);
    return rc;
}

/* Annotation of a whole strand stream: the intervals of segment s are [iv_offset[s], iv_offset[s + 1]) of
 * start / end (each segment's run sorted by start); feature[i] is an index into that segment's run, or -1. */
int crp_result_annotate_strand(const crp_result *res, char strand, const uint64_t *iv_offset, const uint32_t *start,
                               const uint32_t *end, int32_t *feature) {
    if (!res) return fail(CRP_ERR_ARG, "res is NULL");
    if (int rc = need_ctx()) return rc;
    if (strand != '+' && strand != '-') return fail(CRP_ERR_ARG, "strand must be '+' or '-'");
    const int s = strand == '+' ? 0 : 1;
    const uint64_t n = s == 0 ? res->n_plus : res->n_minus;
    if (n == 0) return 0;
    if (!feature || !iv_offset) return fail(CRP_ERR_ARG, "NULL argument");
    const std::vector<uint64_t> &cnt = s == 0 ? res->seg_plus : res->seg_minus;
    const uint64_t n_iv = iv_offset[cnt.size()];
    if (n_iv && (!start || !end)) return fail(CRP_ERR_ARG, "NULL interval arrays");
    std::vector<uint32_t> host(3 * (size_t)n_iv + 1);
    for (size_t sgi = 0; sgi < cnt.size(); ++sgi) {
        uint32_t running = 0;
        if (iv_offset[sgi + 1] < iv_offset[sgi]) return fail(CRP_ERR_ARG, "iv_offset must not decrease");
        for (uint64_t j = iv_offset[sgi]; j < iv_offset[sgi + 1]; ++j) {
            if (j > iv_offset[sgi] && start[j] < start[j - 1]) return fail(CRP_ERR_ARG, "intervals must be sorted by start");
            if (end[j] < start[j]) return fail(CRP_ERR_ARG, "interval %llu has end < start", (unsigned long long)j);
            running = end[j] > running ? end[j] : running;
            host[j] = start[j];
            host[n_iv + j] = end[j];
            host[2 * (size_t)n_iv + j] = running;
        }
    }
    cudaStream_t st = res->st;
    uint32_t *d_iv = nullptr;
    int32_t *d_f = nullptr;
    CUDA_TRY(dev_alloc(&d_iv, host.size() * sizeof(uint32_t), st));
    if (dev_alloc(&d_f, n * sizeof(int32_t), st) != cudaSuccess) {
        dev_free(d_iv, st);
        return fail(CRP_ERR_NOMEM, "cudaMalloc failed");
    }
    int rc = 0;
    if (cudaMemcpyAsync(d_iv, host.data(), host.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st) != cudaSuccess)
        rc = fail(CRP_ERR_CUDA, "H2D of intervals failed");
    uint64_t first = 0;
    for (size_t sgi = 0; sgi < cnt.size() && !rc; ++sgi) {
        const uint64_t m = cnt[sgi];
        if (m) {
            const uint64_t o = iv_offset[sgi];
            k_annotate<<<(unsigned)((m + 255) / 256), 256, 0, st>>>(res->pos[s] + first, m, s, d_iv + o, d_iv + n_iv + o,
                                                                   d_iv + 2 * (size_t)n_iv + o,
                                                                   (uint32_t)(iv_offset[sgi + 1] - o), d_f + first);
            g_ctx.launches++;
        }
        first += m;
    }
    if (!rc && (cudaMemcpyAsync(feature, d_f, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
                cudaStreamSynchronize(st) != cudaSuccess))
        rc = fail(CRP_ERR_CUDA, "annotate failed: %s", cudaGetErrorString(cudaGetLastError()));
    dev_free(d_iv, st);
    dev_free(d_f, st);
    return rc;
}

/* Runs of bytes that are not A C G T a c g t inside one segment (the gaps of an assembly: N, IUPAC codes,
 * anything else), at least min_len long: (start, length) in token coordinates, ascending. */
int crp_genome_other_runs(const crp_genome *g, uint32_t segment, uint32_t min_len, uint64_t capacity, uint32_t *start,
                          uint32_t *length, uint64_t *n_runs) {
    if (!g || !n_runs) return fail(CRP_ERR_ARG, "NULL argument");
    if (int rc = need_ctx()) return rc;
    if (!g->committed) return fail(CRP_ERR_STATE, "genome is not committed");
    if (segment >= g->segs.size()) return fail(CRP_ERR_ARG, "segment %u out of range", segment);
    if (capacity && (!start || !length)) return fail(CRP_ERR_ARG, "NULL output arrays");
    const Segment &sg = g->segs[segment];
    *n_runs = 0;
    if (!sg.n_tiles) return 0;
    cudaStream_t st = stream_of(g);
    // boundaries of ALL runs first (the length filter needs both ends); a segment rarely holds more than a few thousand
    uint32_t cap = 1u << 16;
    std::vector<uint32_t> hs, he;
    for (int attempt = 0; attempt < 2; ++attempt) {
        uint32_t *d = nullptr;
        unsigned int *d_n = nullptr;
        CUDA_TRY(dev_alloc(&d, 2 * (size_t)cap * sizeof(uint32_t), st));
        if (dev_alloc(&d_n, 2 * sizeof(unsigned int), st) != cudaSuccess) {
            dev_free(d, st);
            return fail(CRP_ERR_NOMEM, "cudaMalloc failed");
        }
        RunArgs a;
        a.records = g->records;
        a.first_tile = sg.first_tile;
        a.n_tiles = sg.n_tiles;
        a.seg_begin = (uint32_t)sg.begin;
        a.seg_end = (uint32_t)sg.end;
        a.starts = d;
        a.ends = d + cap;
        a.n_starts = d_n;
        a.n_ends = d_n + 1;
        a.capacity = cap;
        unsigned int n[2] = {0, 0};
        int rc = 0;
        const uint64_t items = (uint64_t)sg.n_tiles * kTileWords;
        if (cudaMemsetAsync(d_n, 0, 2 * sizeof(unsigned int), st) != cudaSuccess) rc = fail(CRP_ERR_CUDA, "memset failed");
        if (!rc) {
            k_other_runs<<<(unsigned)((items + 255) / 256), 256, 0, st>>>(a);
            g_ctx.launches++;
            if (cudaMemcpyAsync(n, d_n, sizeof n, cudaMemcpyDeviceToHost, st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess)
                rc = fail(CRP_ERR_CUDA, "run kernel failed: %s", cudaGetErrorString(cudaGetLastError()));
        }
        if (!rc && n[0] != n[1]) rc = fail(CRP_ERR_STATE, "run boundaries do not pair up (%u starts, %u ends)", n[0], n[1]);
        if (!rc && n[0] <= cap) {
            hs.resize(n[0]);
            he.resize(n[0]);
            if (n[0] && (cudaMemcpyAsync(hs.data(), a.starts, n[0] * sizeof(uint32_t), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
                         cudaMemcpyAsync(he.data(), a.ends, n[0] * sizeof(uint32_t), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
                         cudaStreamSynchronize(st) != cudaSuccess))
                rc = fail(CRP_ERR_CUDA, "D2H of run boundaries failed");
        }
        dev_free(d, st);
        dev_free(d_n, st);
        if (rc) return rc;
        if (n[0] <= cap) break;
        if (attempt == 1) return fail(CRP_ERR_RANGE, "more than %u runs in one segment", cap);
        cap = n[0];
    }
    std::sort(hs.begin(), hs.end());
    std::sort(he.begin(), he.end());
    uint64_t kept = 0;
    for (size_t i = 0; i < hs.size(); ++i) {
        const uint32_t len = he[i] - hs[i] + 1;
        if (len < min_len) continue;
        if (kept < capacity) {
            start[kept] = hs[i];
            length[kept] = len;
        }
        ++kept;
    }
    *n_runs = kept;
    if (kept > capacity) return fail(CRP_ERR_RANGE, "%llu runs, room for %llu", (unsigned long long)kept, (unsigned long long)capacity);
    return 0;
}

int crp_primer_windows(const crp_genome *g, uint64_t n, const uint32_t *segment, const uint32_t *lo, const uint32_t *hi,
                       const crp_primer_params *prm, uint32_t *n_fwd, uint32_t *n_rev, uint64_t *n_pairs,
                       uint16_t *first, uint8_t *status) {
    if (!g || !prm) return fail(CRP_ERR_ARG, "NULL argument");
    if (int rc = need_ctx()) return rc;
    if (!g->committed) return fail(CRP_ERR_STATE, "genome is not committed");
    if (n == 0) return 0;
    if (!segment || !lo || !hi) return fail(CRP_ERR_ARG, "NULL window arrays");
    if (prm->e < 1 || prm->e + prm->l > (uint32_t)kPrimerMaxRegion)
        return fail(CRP_ERR_ARG, "primer extension e=%u with l=%u unsupported: need 1 <= e and e + l <= %d", prm->e, prm->l,
                    kPrimerMaxRegion);
    PrimerClasses pc;
    memset(&pc, 0, sizeof pc);
    char msg[160];
    if (build_primer_classes((int)prm->s, (int)prm->l, prm->m, prm->x, prm->M, prm->X, prm->D, &pc, msg, sizeof msg))
        return fail(CRP_ERR_ARG, "%s", msg);
    std::vector<uint32_t> h(4 * n);             // first_tile | seg_begin | lo | hi
    for (uint64_t i = 0; i < n; ++i) {
        if (segment[i] >= g->segs.size()) return fail(CRP_ERR_ARG, "window %llu: segment %u out of range", (unsigned long long)i, segment[i]);
        const Segment &sg = g->segs[segment[i]];
        if (lo[i] > hi[i] || lo[i] < sg.begin || hi[i] > sg.end)
            return fail(CRP_ERR_ARG, "window %llu [%u, %u) is not inside the positions [%llu, %llu) segment %u owns",
                        (unsigned long long)i, lo[i], hi[i], (unsigned long long)sg.begin, (unsigned long long)sg.end, segment[i]);
        h[i] = sg.first_tile;
        h[n + i] = (uint32_t)sg.begin;
        h[2 * n + i] = lo[i];
        h[3 * n + i] = hi[i];
    }
    cudaStream_t st = stream_of(g);
    uint32_t *d_in = nullptr, *d_cnt = nullptr;
    unsigned long long *d_pairs = nullptr;
    uint16_t *d_first = nullptr;
    uint8_t *d_status = nullptr;
    PrimerClasses *d_cls = nullptr;
    int rc = 0;
    if (dev_alloc(&d_in, 4 * n * sizeof(uint32_t), st) || dev_alloc(&d_cnt, 2 * n * sizeof(uint32_t), st) ||
        dev_alloc(&d_pairs, n * sizeof(unsigned long long), st) || dev_alloc(&d_first, 4 * n * sizeof(uint16_t), st) ||
        dev_alloc(&d_status, n, st) || dev_alloc(&d_cls, sizeof(PrimerClasses), st)) {
        cudaGetLastError();
        rc = fail(CRP_ERR_NOMEM, "cudaMalloc of primer buffers failed");
    }
    if (!rc) {
        PrimerArgs a;
        a.records = g->records;
        a.cls = d_cls;
        a.first_tile = d_in;
        a.seg_begin = d_in + n;
        a.lo = d_in + 2 * n;
        a.hi = d_in + 3 * n;
        a.n = n;
        a.e = prm->e;
        a.n_fwd = d_cnt;
        a.n_rev = d_cnt + n;
        a.n_pairs = d_pairs;
        a.first = d_first;
        a.status = d_status;
        const uint64_t want = (n + 7) / 8, cap = (uint64_t)g_ctx.sm_count * 8;
        if (cudaMemcpyAsync(d_in, h.data(), 4 * n * sizeof(uint32_t), cudaMemcpyHostToDevice, st) != cudaSuccess ||
            cudaMemcpyAsync(d_cls, &pc, sizeof pc, cudaMemcpyHostToDevice, st) != cudaSuccess)
            rc = fail(CRP_ERR_CUDA, "H2D of primer windows failed");
        if (!rc) {
            k_primers<<<(unsigned)(want < cap ? want : cap), 256, 0, st>>>(a);
            g_ctx.launches++;
            auto back = [&](void *dst, const void *src, size_t bytes) {
                if (dst && !rc && cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDeviceToHost, st) != cudaSuccess)
                    rc = fail(CRP_ERR_CUDA, "D2H of primer results failed");
            };
            back(n_fwd, a.n_fwd, n * 4);
            back(n_rev, a.n_rev, n * 4);
            back(n_pairs, a.n_pairs, n * 8);
            back(first, a.first, n * 8);
            back(status, a.status, n);
            if (!rc && cudaStreamSynchronize(st) != cudaSuccess)
                rc = fail(CRP_ERR_CUDA, "primer kernel failed: %s", cudaGetErrorString(cudaGetLastError()));
        }
    }
    dev_free(d_in, st);
    dev_free(d_cnt, st);
    dev_free(d_pairs, st);
    dev_free(d_first, st);
    dev_free(d_status, st);
    dev_free(d_cls, st);
    return rc;
}

int crp_result_annotate(const crp_result *res, uint32_t segment, char strand, uint32_t n_intervals,
                        const uint32_t *start, const uint32_t *end, int32_t *feature) {
    if (!res) return fail(CRP_ERR_ARG, "res is NULL");
    if (int rc = need_ctx()) return rc;
    uint64_t first = 0, n = 0;
    if (int rc = segment_rows(res, segment, strand, &first, &n)) return rc;
    if (n == 0) return 0;
    if (!feature || (n_intervals && (!start || !end))) return fail(CRP_ERR_ARG, "NULL argument");
    std::vector<uint32_t> host(3 * (size_t)n_intervals + 1);
    uint32_t running = 0;
    for (uint32_t j = 0; j < n_intervals; ++j) {
        if (j && start[j] < start[j - 1]) return fail(CRP_ERR_ARG, "intervals must be sorted by start");
        if (end[j] < start[j]) return fail(CRP_ERR_ARG, "interval %u has end < start", j);
        running = end[j] > running ? end[j] : running;
        host[j] = start[j];
        host[n_intervals + j] = end[j];
        host[2 * (size_t)n_intervals + j] = running;
    }
    cudaStream_t st = res->st;
    uint32_t *d_iv = nullptr;
    int32_t *d_f = nullptr;
    CUDA_TRY(dev_alloc(&d_iv, host.size() * sizeof(uint32_t), st));
    if (dev_alloc(&d_f, n * sizeof(int32_t), st) != cudaSuccess) {
        dev_free(d_iv, st);
        return fail(CRP_ERR_NOMEM, "cudaMalloc failed");
    }
    int rc = 0;
    const int s = strand == '+' ? 0 : 1;
    if (cudaMemcpyAsync(d_iv, host.data(), host.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st) != cudaSuccess)
        rc = fail(CRP_ERR_CUDA, "H2D of intervals failed");
    if (!rc) {
        k_annotate<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(res->pos[s] + first, n, s, d_iv, d_iv + n_intervals,
                                                               d_iv + 2 * (size_t)n_intervals, n_intervals, d_f);
        g_ctx.launches++;
        if (cudaMemcpyAsync(feature, d_f, n * sizeof(int32_t), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaStreamSynchronize(st) != cudaSuccess)
            rc = fail(CRP_ERR_CUDA, "annotate failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
    dev_free(d_iv, st);
    dev_free(d_f, st);
    return rc;
}

int crp_rescore(const crp_genome *g, uint64_t n, const uint32_t *segment, const uint32_t *t, const char *strand,
                const uint8_t *cls, double *x_out) {
    if (!g) return fail(CRP_ERR_ARG, "g is NULL");
    if (int rc = need_ctx()) return rc;
    if (!g->committed) return fail(CRP_ERR_STATE, "genome not committed");
    if (n == 0) return 0;
    if (!segment || !t || !strand || !cls || !x_out) return fail(CRP_ERR_ARG, "NULL argument");
    std::vector<RescoreItem> items(n);
    for (uint64_t i = 0; i < n; ++i) {
        if (segment[i] >= g->segs.size()) return fail(CRP_ERR_ARG, "item %llu: bad segment", (unsigned long long)i);
        const Segment &s = g->segs[segment[i]];
        if (t[i] < s.begin || t[i] >= s.end)
            return fail(CRP_ERR_ARG, "item %llu: t=%u outside segment", (unsigned long long)i, t[i]);
        if (strand[i] != '+' && strand[i] != '-') return fail(CRP_ERR_ARG, "item %llu: bad strand", (unsigned long long)i);
        if ((cls[i] & 15u) > CRP_CLASS_SINGLE || (cls[i] >> 4) > CRP_CLASS_SINGLE) return fail(CRP_ERR_ARG, "item %llu: bad class", (unsigned long long)i);
        const uint64_t rel = t[i] - s.begin;
        items[i].tile = s.first_tile + (uint32_t)(rel / kTile);
        items[i].pl = (uint32_t)(rel % kTile);
        items[i].strand = (uint32_t)strand[i];
        items[i].cls = cls[i];
    }
    cudaStream_t st = stream_of(g);
    RescoreItem *d_items = nullptr;
    double *d_x = nullptr;
    CUDA_TRY(dev_alloc(&d_items, n * sizeof(RescoreItem), st));
    if (dev_alloc(&d_x, n * sizeof(double), st) != cudaSuccess) {
        dev_free(d_items, st);
        return fail(CRP_ERR_NOMEM, "cudaMalloc failed");
    }
    int rc = 0;
    do {
        if (cudaMemcpyAsync(d_items, items.data(), n * sizeof(RescoreItem), cudaMemcpyHostToDevice, st) != cudaSuccess) {
            rc = fail(CRP_ERR_CUDA, "H2D of rescore items failed");
            break;
        }
        k_rescore<<<(unsigned)((n + 127) / 128), 128, 0, st>>>(g->records, d_items, n, d_x);
        g_ctx.launches++;
        if (cudaMemcpyAsync(x_out, d_x, n * sizeof(double), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaStreamSynchronize(st) != cudaSuccess) {
            rc = fail(CRP_ERR_CUDA, "rescore failed: %s", cudaGetErrorString(cudaGetLastError()));
            break;
        }
    } while (0);
    dev_free(d_items, st);
    dev_free(d_x, st);
    return rc;
}

}  // extern "C"

// ------------------------------------------------------------------ off-target counts (offtarget.cuh)

// k_ot_queries' segment table of one strand stream (s = 0 '+', 1 '-'): row offsets [n_seg + 1], first tiles [n_seg],
// first positions [n_seg]
static std::vector<uint32_t> ot_segment_table(const crp_result *res, int s) {
    const std::vector<uint64_t> &cnt = s == 0 ? res->seg_plus : res->seg_minus;
    const uint32_t n_seg = (uint32_t)cnt.size();
    std::vector<uint32_t> seg(3 * (size_t)n_seg + 1);
    uint64_t row = 0;
    for (uint32_t i = 0; i < n_seg; ++i) {
        seg[i] = (uint32_t)row;
        row += cnt[i];
        seg[n_seg + 1 + i] = res->g->segs[i].first_tile;
        seg[2 * (size_t)n_seg + 1 + i] = (uint32_t)res->g->segs[i].begin;
    }
    seg[n_seg] = (uint32_t)row;
    return seg;
}

struct crp_offtarget {
    cudaStream_t st = nullptr;                 // own stream, ordered behind each genome's stream by an event
    cudaEvent_t ev[5] = {nullptr, nullptr, nullptr, nullptr, nullptr};   // sites start / end, count start / end, genome ready
    std::vector<const crp_genome *> genomes;
    unsigned long long *keys = nullptr;        // site keys of every genome added, any order
    unsigned long long *loci = nullptr;        // crp_offtarget_new_with_loci: the locus of every site, at its key's slot
    bool with_loci = false;
    uint32_t s2 = 8, s3 = 8;                   // code sets of PAM letters 2 and 3 (ot_pam_plus_sets): {G}, {G} is NGG
    bool own_site = true;                      // a candidate's own site is a site of the index: G in s2 and in s3
    uint64_t n_sites = 0;
    float ms_sites = 0.f, ms_count = 0.f;      // summed over add_genome / of the last count, list or score call
    uint64_t comparisons = 0;
};

// Join every query of d_keys (n rows, kOtInvalid = no key) against the index's sites, part pair by part pair, with
// k_ot_join<Op>: op takes every (query, site) pair within k mismatches into its outputs.  On ix->st; waits for the
// result.
template <class Op>
static int ot_join(crp_offtarget *ix, const unsigned long long *d_keys, uint64_t n, uint32_t k, const Op &op) {
    using Site = typename Op::Site;
    cudaStream_t st = ix->st;
    const size_t tbl = kOtBuckets + 1;
    uint32_t *d_tbl = nullptr;
    Site *d_sites = nullptr;
    uint2 *d_q = nullptr;
    unsigned long long *d_misc = nullptr;      // [0] comparisons, [1] overflow flag
    if (dev_alloc(&d_tbl, 7 * tbl * sizeof(uint32_t), st) != cudaSuccess ||
        dev_alloc(&d_sites, (ix->n_sites + 8) * sizeof(Site), st) != cudaSuccess ||
        dev_alloc(&d_q, (n + 1) * sizeof(uint2), st) != cudaSuccess ||
        dev_alloc(&d_misc, 2 * sizeof(unsigned long long), st) != cudaSuccess) {
        cudaGetLastError();
        dev_free(d_tbl, st);
        dev_free(d_sites, st);
        dev_free(d_q, st);
        return fail(CRP_ERR_NOMEM, "cudaMalloc of the off-target work buffers failed");
    }
    uint32_t *hist_s = d_tbl, *hist_q = d_tbl + tbl;
    OtScanArgs sa;
    sa.hist[0] = hist_s;
    sa.hist[1] = hist_q;
    sa.off[0] = d_tbl + 2 * tbl;
    sa.off[1] = d_tbl + 3 * tbl;
    sa.cursor[0] = d_tbl + 4 * tbl;
    sa.cursor[1] = d_tbl + 5 * tbl;
    sa.item_off = d_tbl + 6 * tbl;
    sa.comparisons = d_misc;
    sa.overflow = reinterpret_cast<unsigned int *>(d_misc + 1);
    OtJoin ja;
    ja.sites = d_sites;
    ja.queries = d_q;
    ja.soff = sa.off[0];
    ja.qoff = sa.off[1];
    ja.item_off = sa.item_off;
    ja.k = k;
    auto grid = [](uint64_t items) { return (unsigned)std::max<uint64_t>(1, std::min<uint64_t>((items + 255) / 256, (uint64_t)g_ctx.sm_count * 16)); };
    int rc = 0;
    unsigned long long misc[2] = {0, 0};
    if (cudaMemsetAsync(d_misc, 0, 2 * sizeof(unsigned long long), st) != cudaSuccess ||
        cudaEventRecord(ix->ev[2], st) != cudaSuccess)
        rc = fail(CRP_ERR_CUDA, "off-target setup failed");
    for (int p = 0; p < kOtPairs && !rc && n && ix->n_sites; ++p) {
        int i = 0, j = 0;
        ot_pair(p, i, j);
        ja.jm1 = (uint32_t)(j - 1);
        ja.pi = i;
        ja.pj = j;
        if (cudaMemsetAsync(d_tbl, 0, 2 * tbl * sizeof(uint32_t), st) != cudaSuccess) {
            rc = fail(CRP_ERR_CUDA, "memset failed");
            break;
        }
        k_ot_hist<<<grid(ix->n_sites), 256, 0, st>>>(ix->keys, ix->n_sites, i, j, hist_s);
        k_ot_hist<<<grid(n), 256, 0, st>>>(d_keys, n, i, j, hist_q);
        k_ot_scan<<<3, kOtScanThreads, 0, st>>>(sa);
        if constexpr (std::is_same_v<Site, uint2>)   // {rest key, site index}: the query form of the scatter
            k_ot_scatter<<<grid(ix->n_sites), 256, 0, st>>>(ix->keys, ix->n_sites, i, j, sa.cursor[0], nullptr, d_sites);
        else
            k_ot_scatter<<<grid(ix->n_sites), 256, 0, st>>>(ix->keys, ix->n_sites, i, j, sa.cursor[0], d_sites, nullptr);
        k_ot_scatter<<<grid(n), 256, 0, st>>>(d_keys, n, i, j, sa.cursor[1], nullptr, d_q);
        k_ot_join<Op><<<(unsigned)g_ctx.sm_count * 8, kOtThreads, 0, st>>>(ja, op);
        g_ctx.launches += 6;
        if (cudaGetLastError() != cudaSuccess) rc = fail(CRP_ERR_CUDA, "off-target launch failed");
    }
    if (!rc && (cudaEventRecord(ix->ev[3], st) != cudaSuccess ||
                cudaMemcpyAsync(misc, d_misc, sizeof misc, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
                cudaStreamSynchronize(st) != cudaSuccess ||
                cudaEventElapsedTime(&ix->ms_count, ix->ev[2], ix->ev[3]) != cudaSuccess))
        rc = fail(CRP_ERR_CUDA, "off-target join failed: %s", cudaGetErrorString(cudaGetLastError()));
    if (!rc && misc[1]) rc = fail(CRP_ERR_RANGE, "a part pair needs 2^32 work items or more");
    if (!rc) ix->comparisons = misc[0];
    dev_free(d_tbl, st);
    dev_free(d_sites, st);
    dev_free(d_q, st);
    dev_free(d_misc, st);
    return rc;
}

// The checks of a *_candidates call, in this order: CRP_ERR_ARG for a NULL index or result, a strand other than '+' /
// '-' or max_mm above 3; CRP_ERR_STATE if `loci` and the index keeps none, for a guide length other than 20, or if
// the result's genome is not in the index.  `what` names the mode's output.
static int ot_check_candidates(const crp_offtarget *ix, const crp_result *res, char strand, uint32_t max_mm,
                               const char *what, bool loci) {
    if (!ix || !res) return fail(CRP_ERR_ARG, "NULL argument");
    if (int rc = need_ctx()) return rc;
    if (strand != '+' && strand != '-') return fail(CRP_ERR_ARG, "strand must be '+' or '-'");
    if (max_mm > 3) return fail(CRP_ERR_ARG, "max_mm %u: at most 3 mismatches", max_mm);
    if (loci && !ix->with_loci) return fail(CRP_ERR_STATE, "listing needs an index with loci (crp_offtarget_new_with_loci)");
    if (res->guide_len != 20) return fail(CRP_ERR_STATE, "off-target %s are defined for guide_len 20 only", what);
    if (std::find(ix->genomes.begin(), ix->genomes.end(), res->g) == ix->genomes.end())
        return fail(CRP_ERR_STATE, "the result's genome has not been added to the index");
    return 0;
}

// The query keys of strand stream s of a checked result into *d_keys [n] (k_ot_queries), on ix->st behind the scan's
// stream.  d_counts [n][k1], when not NULL, gets every row's primed counts.  *d_seg keeps the segment table
// (ot_segment_table) for k_ot_gather.  The caller frees *d_keys and *d_seg, also after a failure.
static int ot_candidate_keys(crp_offtarget *ix, const crp_result *res, int s, uint32_t *d_counts, uint32_t k1,
                             unsigned long long **d_keys, uint32_t **d_seg) {
    const uint64_t n = s == 0 ? res->n_plus : res->n_minus;
    const uint32_t n_seg = (uint32_t)(s == 0 ? res->seg_plus : res->seg_minus).size();
    const std::vector<uint32_t> seg = ot_segment_table(res, s);
    cudaStream_t st = ix->st;
    CUDA_TRY(cudaEventRecord(ix->ev[4], res->st));             // the candidate streams are written on the scan's stream
    CUDA_TRY(cudaStreamWaitEvent(st, ix->ev[4], 0));
    if (dev_alloc(d_seg, seg.size() * sizeof(uint32_t), st) != cudaSuccess ||
        dev_alloc(d_keys, n * sizeof(unsigned long long), st) != cudaSuccess) {
        cudaGetLastError();
        return fail(CRP_ERR_NOMEM, "cudaMalloc of %llu query rows failed", (unsigned long long)n);
    }
    if (cudaMemcpyAsync(*d_seg, seg.data(), seg.size() * sizeof(uint32_t), cudaMemcpyHostToDevice, st) != cudaSuccess)
        return fail(CRP_ERR_CUDA, "H2D of the segment table failed");
    OtQueryArgs a;
    a.records = res->g->records;
    a.pos = res->pos[s];
    a.n = n;
    a.seg_row = *d_seg;
    a.seg_tile = *d_seg + n_seg + 1;
    a.seg_begin = *d_seg + 2 * (size_t)n_seg + 1;
    a.n_seg = n_seg;
    a.k1 = k1;
    a.minus = s;
    a.keys = *d_keys;
    a.counts = d_counts;
    a.own = ix->own_site ? 0xFFFFFFFFu : 0u;
    k_ot_queries<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(a);
    g_ctx.launches++;
    if (cudaGetLastError() != cudaSuccess) return fail(CRP_ERR_CUDA, "off-target query keys failed");
    return 0;
}

// The keys of a *_keys call: CRP_ERR_ARG if NULL or if a key has bits above bit 39, CRP_ERR_RANGE for more than
// 2^32 - 1 keys.
static int ot_check_keys(uint64_t n, const uint64_t *keys) {
    if (!keys) return fail(CRP_ERR_ARG, "keys is NULL");
    if (n > 0xFFFFFFFFull) return fail(CRP_ERR_RANGE, "at most 2^32 - 1 keys per call");
    for (uint64_t i = 0; i < n; ++i)
        if (keys[i] >> 40) return fail(CRP_ERR_ARG, "key %llu has bits above bit 39", (unsigned long long)i);
    return 0;
}

// Checked keys into *d_keys [n] on ix->st; the caller frees *d_keys, also after a failure.
static int ot_upload_keys(crp_offtarget *ix, uint64_t n, const uint64_t *keys, unsigned long long **d_keys) {
    if (dev_alloc(d_keys, n * sizeof(unsigned long long), ix->st) != cudaSuccess) {
        cudaGetLastError();
        return fail(CRP_ERR_NOMEM, "cudaMalloc of %llu keys failed", (unsigned long long)n);
    }
    if (cudaMemcpyAsync(*d_keys, keys, n * sizeof(uint64_t), cudaMemcpyHostToDevice, ix->st) != cudaSuccess)
        return fail(CRP_ERR_CUDA, "H2D of the keys failed");
    return 0;
}

// Counts of n queries whose keys are on the device: d_counts [n][k + 1], primed by the caller, to counts on the host.
static int ot_count(crp_offtarget *ix, const unsigned long long *d_keys, uint64_t n, uint32_t k, uint32_t *d_counts,
                    uint32_t *counts) {
    cudaStream_t st = ix->st;
    int rc = ot_join(ix, d_keys, n, k, OtCount{d_counts});
    if (!rc && (cudaMemcpyAsync(counts, d_counts, n * (k + 1) * sizeof(uint32_t), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
                cudaStreamSynchronize(st) != cudaSuccess))
        rc = fail(CRP_ERR_CUDA, "D2H of the off-target counts failed");
    return rc;
}

extern "C" {

int crp_offtarget_new(crp_offtarget **ix) {
    if (!ix) return fail(CRP_ERR_ARG, "ix is NULL");
    if (int rc = need_ctx()) return rc;
    crp_offtarget *o = new (std::nothrow) crp_offtarget();
    if (!o) return fail(CRP_ERR_NOMEM, "out of host memory");
    if (cudaStreamCreateWithFlags(&o->st, cudaStreamNonBlocking) != cudaSuccess) {
        delete o;
        return fail(CRP_ERR_CUDA, "cudaStreamCreate failed");
    }
    for (int i = 0; i < 5; ++i)
        if (cudaEventCreateWithFlags(&o->ev[i], i == 4 ? cudaEventDisableTiming : cudaEventDefault) != cudaSuccess) {
            crp_offtarget_free(o);
            return fail(CRP_ERR_CUDA, "cudaEventCreate failed");
        }
    *ix = o;
    return 0;
}

int crp_offtarget_new_with_loci(crp_offtarget **ix) {
    if (int rc = crp_offtarget_new(ix)) return rc;
    (*ix)->with_loci = true;
    return 0;
}

int crp_offtarget_new_pam(crp_offtarget **ix, const char *pam, int with_loci) {
    if (!ix || !pam) return fail(CRP_ERR_ARG, "NULL argument");
    // code sets (bit c = code c, A0 T1 C2 G3) of the IUPAC letters for one to three bases
    auto set_of = [](char ch) -> uint32_t {
        switch (ch & ~0x20) {
        case 'A': return 1; case 'T': return 2; case 'C': return 4; case 'G': return 8;
        case 'R': return 9; case 'Y': return 6; case 'S': return 12; case 'W': return 3;
        case 'K': return 10; case 'M': return 5; case 'B': return 14; case 'D': return 11;
        case 'H': return 7; case 'V': return 13;
        default: return 0;
        }
    };
    uint32_t s2 = 0, s3 = 0;
    if ((pam[0] & ~0x20) != 'N' || !(s2 = set_of(pam[1])) || !(s3 = set_of(pam[2])) || pam[3])
        return fail(CRP_ERR_ARG, "PAM pattern \"%.8s\": N and two of ACGTRYSWKMBDHV expected", pam);
    if (int rc = with_loci ? crp_offtarget_new_with_loci(ix) : crp_offtarget_new(ix)) return rc;
    (*ix)->s2 = s2;
    (*ix)->s3 = s3;
    (*ix)->own_site = (s2 & 8u) && (s3 & 8u);
    return 0;
}

int crp_offtarget_add_genome(crp_offtarget *ix, const crp_genome *g) {
    if (!ix || !g) return fail(CRP_ERR_ARG, "NULL argument");
    if (int rc = need_ctx()) return rc;
    if (!g->committed) return fail(CRP_ERR_STATE, "genome is not committed");
    if (std::find(ix->genomes.begin(), ix->genomes.end(), g) != ix->genomes.end())
        return fail(CRP_ERR_STATE, "genome already added to this index");
    if (ix->with_loci && g->segs.size() >= kOtMaxSegments)
        return fail(CRP_ERR_RANGE, "%zu segments: a locus holds 24 bits of segment index", g->segs.size());
    if (ix->with_loci && ix->genomes.size() >= kOtMaxGenomes)
        return fail(CRP_ERR_RANGE, "an index with loci takes at most %u genome handles", kOtMaxGenomes);
    cudaStream_t st = ix->st;
    CUDA_TRY(cudaEventRecord(ix->ev[4], stream_of(g)));        // the records are written on the genome's stream
    CUDA_TRY(cudaStreamWaitEvent(st, ix->ev[4], 0));
    const uint64_t items = (uint64_t)g->n_tiles * kTileWords;
    unsigned long long *d_n = nullptr, *h_n = static_cast<unsigned long long *>(pinned_get(sizeof(unsigned long long)));
    if (!h_n) return fail(CRP_ERR_NOMEM, "cudaHostAlloc failed");
    CUDA_TRY(dev_alloc(&d_n, sizeof(unsigned long long), st));
    OtSiteArgs a;
    a.records = g->records;
    a.n_tiles = g->n_tiles;
    a.keys = nullptr;
    a.base = ix->n_sites;
    a.n = d_n;
    a.loci = nullptr;
    a.genome = (uint32_t)ix->genomes.size();
    a.s2 = ix->s2;
    a.s3 = ix->s3;
    const bool ngg = ix->s2 == 8u && ix->s3 == 8u;          // the NGG kernels, as before patterns existed
    auto launch = [&](bool loci) {
        const unsigned blocks = (unsigned)((items + 255) / 256);
        if (loci && ngg) k_ot_sites<true, false><<<blocks, 256, 0, st>>>(a);
        else if (loci) k_ot_sites<true, true><<<blocks, 256, 0, st>>>(a);
        else if (ngg) k_ot_sites<false, false><<<blocks, 256, 0, st>>>(a);
        else k_ot_sites<false, true><<<blocks, 256, 0, st>>>(a);
        g_ctx.launches++;
    };
    int rc = 0;
    *h_n = 0;
    // pass 1 counts, pass 2 appends behind the sites already held (the key and locus arrays grow by one copy)
    if (cudaEventRecord(ix->ev[0], st) != cudaSuccess || cudaMemsetAsync(d_n, 0, sizeof *d_n, st) != cudaSuccess)
        rc = fail(CRP_ERR_CUDA, "off-target setup failed");
    if (!rc && items) launch(false);
    if (!rc && (cudaMemcpyAsync(h_n, d_n, sizeof *d_n, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
                cudaStreamSynchronize(st) != cudaSuccess))
        rc = fail(CRP_ERR_CUDA, "site count failed: %s", cudaGetErrorString(cudaGetLastError()));
    const uint64_t add = *h_n, total = ix->n_sites + add;
    if (!rc && total > 0xFFFFFFFFull) rc = fail(CRP_ERR_RANGE, "%llu sites exceed 2^32 - 1", (unsigned long long)total);
    if (!rc && add) {
        unsigned long long *keys = nullptr, *loci = nullptr;
        if (dev_alloc(&keys, total * sizeof(unsigned long long), st) != cudaSuccess ||
            (ix->with_loci && dev_alloc(&loci, total * sizeof(unsigned long long), st) != cudaSuccess)) {
            cudaGetLastError();
            dev_free(keys, st);
            rc = fail(CRP_ERR_NOMEM, "cudaMalloc of %llu site keys failed", (unsigned long long)total);
        } else {
            if (ix->n_sites && cudaMemcpyAsync(keys, ix->keys, ix->n_sites * sizeof(unsigned long long), cudaMemcpyDeviceToDevice,
                                               st) != cudaSuccess)
                rc = fail(CRP_ERR_CUDA, "copy of the site keys failed");
            if (!rc && loci && ix->n_sites &&
                cudaMemcpyAsync(loci, ix->loci, ix->n_sites * sizeof(unsigned long long), cudaMemcpyDeviceToDevice, st) != cudaSuccess)
                rc = fail(CRP_ERR_CUDA, "copy of the site loci failed");
            dev_free(ix->keys, st);
            dev_free(ix->loci, st);
            ix->keys = keys;
            ix->loci = loci;
            a.keys = keys;
            a.loci = loci;
            if (!rc && cudaMemsetAsync(d_n, 0, sizeof *d_n, st) != cudaSuccess) rc = fail(CRP_ERR_CUDA, "memset failed");
            if (!rc) launch(loci != nullptr);
            if (!rc && (cudaMemcpyAsync(h_n, d_n, sizeof *d_n, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
                        cudaEventRecord(ix->ev[1], st) != cudaSuccess || cudaStreamSynchronize(st) != cudaSuccess))
                rc = fail(CRP_ERR_CUDA, "site keys failed: %s", cudaGetErrorString(cudaGetLastError()));
            if (!rc && *h_n != add) rc = fail(CRP_ERR_STATE, "site passes disagree (%llu, %llu)", (unsigned long long)add, *h_n);
            if (rc) {                          // the old keys went with the old array: the index is emptied
                dev_free(ix->keys, st);
                dev_free(ix->loci, st);
                ix->keys = nullptr;
                ix->loci = nullptr;
                ix->n_sites = 0;
                ix->genomes.clear();
            }
        }
    } else if (!rc) {
        rc = cudaEventRecord(ix->ev[1], st) == cudaSuccess && cudaEventSynchronize(ix->ev[1]) == cudaSuccess
                 ? 0 : fail(CRP_ERR_CUDA, "event failed");
    }
    float ms = 0.f;
    if (!rc && cudaEventElapsedTime(&ms, ix->ev[0], ix->ev[1]) == cudaSuccess) ix->ms_sites += ms;
    if (!rc) {
        ix->n_sites = total;
        ix->genomes.push_back(g);
    }
    dev_free(d_n, st);
    pinned_put(h_n);
    return rc;
}

int crp_offtarget_num_sites(const crp_offtarget *ix, uint64_t *n) {
    if (!ix || !n) return fail(CRP_ERR_ARG, "NULL argument");
    *n = ix->n_sites;
    return 0;
}

int crp_offtarget_fetch_sites(const crp_offtarget *ix, uint64_t capacity, uint64_t *keys, uint64_t *n) {
    if (!ix || !n) return fail(CRP_ERR_ARG, "NULL argument");
    *n = ix->n_sites;
    if (capacity < ix->n_sites) return fail(CRP_ERR_RANGE, "%llu sites, room for %llu", (unsigned long long)ix->n_sites,
                                            (unsigned long long)capacity);
    if (!ix->n_sites) return 0;
    if (!keys) return fail(CRP_ERR_ARG, "keys is NULL");
    CUDA_TRY(cudaMemcpyAsync(keys, ix->keys, ix->n_sites * sizeof(uint64_t), cudaMemcpyDeviceToHost, ix->st));
    CUDA_TRY(cudaStreamSynchronize(ix->st));
    return 0;
}

int crp_offtarget_count_candidates(crp_offtarget *ix, const crp_result *res, char strand, uint32_t max_mm, uint32_t *counts) {
    if (int rc = ot_check_candidates(ix, res, strand, max_mm, "counts", false)) return rc;
    const int s = strand == '+' ? 0 : 1;
    const uint64_t n = s == 0 ? res->n_plus : res->n_minus;
    if (n == 0) return 0;
    if (!counts) return fail(CRP_ERR_ARG, "counts is NULL");
    cudaStream_t st = ix->st;
    const uint32_t k1 = max_mm + 1;
    uint32_t *d_seg = nullptr, *d_counts = nullptr;
    unsigned long long *d_keys = nullptr;
    int rc = 0;
    if (dev_alloc(&d_counts, n * k1 * sizeof(uint32_t), st) != cudaSuccess) {
        cudaGetLastError();
        rc = fail(CRP_ERR_NOMEM, "cudaMalloc of %llu query rows failed", (unsigned long long)n);
    }
    if (!rc) rc = ot_candidate_keys(ix, res, s, d_counts, k1, &d_keys, &d_seg);
    if (!rc) rc = ot_count(ix, d_keys, n, max_mm, d_counts, counts);
    dev_free(d_seg, st);
    dev_free(d_keys, st);
    dev_free(d_counts, st);
    return rc;
}

int crp_offtarget_count_keys(crp_offtarget *ix, uint64_t n, const uint64_t *keys, uint32_t max_mm, uint32_t *counts) {
    if (!ix) return fail(CRP_ERR_ARG, "ix is NULL");
    if (int rc = need_ctx()) return rc;
    if (max_mm > 3) return fail(CRP_ERR_ARG, "max_mm %u: at most 3 mismatches", max_mm);
    if (n == 0) return 0;
    if (!counts) return fail(CRP_ERR_ARG, "counts is NULL");
    if (int rc = ot_check_keys(n, keys)) return rc;
    cudaStream_t st = ix->st;
    const uint32_t k1 = max_mm + 1;
    unsigned long long *d_keys = nullptr;
    uint32_t *d_counts = nullptr;
    int rc = ot_upload_keys(ix, n, keys, &d_keys);
    if (!rc && dev_alloc(&d_counts, n * k1 * sizeof(uint32_t), st) != cudaSuccess) {
        cudaGetLastError();
        rc = fail(CRP_ERR_NOMEM, "cudaMalloc of %llu keys failed", (unsigned long long)n);
    }
    if (!rc && cudaMemsetAsync(d_counts, 0, n * k1 * sizeof(uint32_t), st) != cudaSuccess)
        rc = fail(CRP_ERR_CUDA, "memset failed");
    if (!rc) rc = ot_count(ix, d_keys, n, max_mm, d_counts, counts);
    dev_free(d_keys, st);
    dev_free(d_counts, st);
    return rc;
}

int crp_offtarget_fetch_loci(const crp_offtarget *ix, uint64_t capacity, uint64_t *loci, uint64_t *n) {
    if (!ix || !n) return fail(CRP_ERR_ARG, "NULL argument");
    if (!ix->with_loci) return fail(CRP_ERR_STATE, "the index keeps no loci (crp_offtarget_new_with_loci)");
    *n = ix->n_sites;
    if (capacity < ix->n_sites) return fail(CRP_ERR_RANGE, "%llu sites, room for %llu", (unsigned long long)ix->n_sites,
                                            (unsigned long long)capacity);
    if (!ix->n_sites) return 0;
    if (!loci) return fail(CRP_ERR_ARG, "loci is NULL");
    CUDA_TRY(cudaMemcpyAsync(loci, ix->loci, ix->n_sites * sizeof(uint64_t), cudaMemcpyDeviceToHost, ix->st));
    CUDA_TRY(cudaStreamSynchronize(ix->st));
    return 0;
}

}  // extern "C"

// The listing of n queries whose keys (and own-site loci, or NULL) are on the device: slices `first` [n + 1] on the
// host, site indices into `sites` [first[n]] on the host.  CRP_ERR_STATE, with nothing copied, if a row finds a
// number of sites other than its slice holds.
static int ot_list(crp_offtarget *ix, const unsigned long long *d_keys, const unsigned long long *d_own, uint64_t n,
                   uint32_t k, const uint64_t *first, uint32_t *sites) {
    cudaStream_t st = ix->st;
    const uint64_t total = first[n];
    unsigned long long *d_first = nullptr;
    uint32_t *d_cursor = nullptr, *d_out = nullptr;
    unsigned int *d_flag = nullptr;
    if (dev_alloc(&d_first, (n + 1) * sizeof(unsigned long long), st) != cudaSuccess ||
        dev_alloc(&d_cursor, n * sizeof(uint32_t), st) != cudaSuccess ||
        dev_alloc(&d_out, std::max<uint64_t>(total, 1) * sizeof(uint32_t), st) != cudaSuccess ||
        dev_alloc(&d_flag, sizeof(unsigned int), st) != cudaSuccess) {
        cudaGetLastError();
        dev_free(d_first, st);
        dev_free(d_cursor, st);
        dev_free(d_out, st);
        return fail(CRP_ERR_NOMEM, "cudaMalloc of a listing of %llu sites failed", (unsigned long long)total);
    }
    int rc = 0;
    if (cudaMemcpyAsync(d_first, first, (n + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st) != cudaSuccess ||
        cudaMemsetAsync(d_cursor, 0, n * sizeof(uint32_t), st) != cudaSuccess ||
        cudaMemsetAsync(d_flag, 0, sizeof(unsigned int), st) != cudaSuccess)
        rc = fail(CRP_ERR_CUDA, "listing setup failed");
    if (!rc) rc = ot_join(ix, d_keys, n, k, OtList{ix->loci, d_own, d_first, d_cursor, d_out, d_flag});
    std::vector<uint32_t> found(rc ? 0 : n);
    unsigned int flag = 0;
    if (!rc && (cudaMemcpyAsync(found.data(), d_cursor, n * sizeof(uint32_t), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
                cudaMemcpyAsync(&flag, d_flag, sizeof flag, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
                cudaStreamSynchronize(st) != cudaSuccess))
        rc = fail(CRP_ERR_CUDA, "D2H of the listing cursors failed");
    for (uint64_t i = 0; i < n && !rc; ++i)
        if (found[i] != first[i + 1] - first[i])
            rc = fail(CRP_ERR_STATE, "row %llu: %u sites found, its slice holds %llu", (unsigned long long)i, found[i],
                      (unsigned long long)(first[i + 1] - first[i]));
    if (!rc && flag) rc = fail(CRP_ERR_STATE, "a row found more sites than its slice holds");
    if (!rc && total && (cudaMemcpyAsync(sites, d_out, total * sizeof(uint32_t), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
                         cudaStreamSynchronize(st) != cudaSuccess))
        rc = fail(CRP_ERR_CUDA, "D2H of the listing failed");
    dev_free(d_first, st);
    dev_free(d_cursor, st);
    dev_free(d_out, st);
    dev_free(d_flag, st);
    return rc;
}

// first [n + 1] of a listing call: CRP_ERR_ARG unless it starts at 0 and never decreases
static int ot_check_first(uint64_t n, const uint64_t *first) {
    if (!first) return fail(CRP_ERR_ARG, "first is NULL");
    if (first[0] != 0) return fail(CRP_ERR_ARG, "first[0] must be 0");
    for (uint64_t i = 0; i < n; ++i)
        if (first[i + 1] < first[i]) return fail(CRP_ERR_ARG, "first[%llu] < first[%llu]", (unsigned long long)i + 1,
                                                 (unsigned long long)i);
    return 0;
}

extern "C" {

int crp_offtarget_list_candidates(crp_offtarget *ix, const crp_result *res, char strand, uint32_t max_mm, uint64_t n_rows,
                                  const uint32_t *rows, const uint64_t *first, uint32_t *sites) {
    if (int rc = ot_check_candidates(ix, res, strand, max_mm, "listings", true)) return rc;
    if (n_rows == 0) return 0;
    if (!rows) return fail(CRP_ERR_ARG, "rows is NULL");
    if (int rc = ot_check_first(n_rows, first)) return rc;
    if (first[n_rows] && !sites) return fail(CRP_ERR_ARG, "sites is NULL");
    const int s = strand == '+' ? 0 : 1;
    const uint64_t n = s == 0 ? res->n_plus : res->n_minus;
    for (uint64_t i = 0; i < n_rows; ++i)
        if (rows[i] >= n || (i && rows[i] <= rows[i - 1]))
            return fail(CRP_ERR_ARG, "rows[%llu] = %u: rows must be ascending, distinct and below %llu", (unsigned long long)i,
                        rows[i], (unsigned long long)n);
    cudaStream_t st = ix->st;
    uint32_t *d_seg = nullptr, *d_rows = nullptr;
    unsigned long long *d_keys = nullptr, *d_sel = nullptr;   // d_sel: [n_rows] keys, [n_rows] own loci
    unsigned int *d_invalid = nullptr;
    int rc = ot_candidate_keys(ix, res, s, nullptr, 0, &d_keys, &d_seg);   // every row's key, then the selected rows
    if (!rc && (dev_alloc(&d_rows, n_rows * sizeof(uint32_t), st) != cudaSuccess ||
                dev_alloc(&d_sel, 2 * n_rows * sizeof(unsigned long long), st) != cudaSuccess ||
                dev_alloc(&d_invalid, sizeof(unsigned int), st) != cudaSuccess)) {
        cudaGetLastError();
        rc = fail(CRP_ERR_NOMEM, "cudaMalloc of %llu selected rows failed", (unsigned long long)n_rows);
    }
    if (!rc && (cudaMemcpyAsync(d_rows, rows, n_rows * sizeof(uint32_t), cudaMemcpyHostToDevice, st) != cudaSuccess ||
                cudaMemsetAsync(d_invalid, 0, sizeof(unsigned int), st) != cudaSuccess))
        rc = fail(CRP_ERR_CUDA, "H2D of the listing rows failed");
    unsigned int invalid = 0;
    if (!rc) {
        OtGatherArgs ga;
        ga.keys = d_keys;
        ga.pos = res->pos[s];
        ga.rows = d_rows;
        ga.seg_row = d_seg;
        ga.n = n_rows;
        ga.n_seg = (uint32_t)(s == 0 ? res->seg_plus : res->seg_minus).size();
        ga.genome = (uint32_t)(std::find(ix->genomes.begin(), ix->genomes.end(), res->g) - ix->genomes.begin());
        ga.minus = s;
        ga.sel_keys = d_sel;
        ga.own = d_sel + n_rows;
        ga.invalid = d_invalid;
        k_ot_gather<<<(unsigned)((n_rows + 255) / 256), 256, 0, st>>>(ga);
        g_ctx.launches++;
        if (cudaGetLastError() != cudaSuccess ||
            cudaMemcpyAsync(&invalid, d_invalid, sizeof invalid, cudaMemcpyDeviceToHost, st) != cudaSuccess ||
            cudaStreamSynchronize(st) != cudaSuccess)
            rc = fail(CRP_ERR_CUDA, "off-target query keys failed: %s", cudaGetErrorString(cudaGetLastError()));
    }
    if (!rc && invalid) rc = fail(CRP_ERR_ARG, "a selected row has no protospacer (its counts are 0xFFFFFFFF)");
    if (!rc) rc = ot_list(ix, d_sel, d_sel + n_rows, n_rows, max_mm, first, sites);
    dev_free(d_seg, st);
    dev_free(d_keys, st);
    dev_free(d_rows, st);
    dev_free(d_sel, st);
    dev_free(d_invalid, st);
    return rc;
}

int crp_offtarget_list_keys(crp_offtarget *ix, uint64_t n, const uint64_t *keys, uint32_t max_mm, const uint64_t *first,
                            uint32_t *sites) {
    if (!ix) return fail(CRP_ERR_ARG, "ix is NULL");
    if (int rc = need_ctx()) return rc;
    if (max_mm > 3) return fail(CRP_ERR_ARG, "max_mm %u: at most 3 mismatches", max_mm);
    if (!ix->with_loci) return fail(CRP_ERR_STATE, "listing needs an index with loci (crp_offtarget_new_with_loci)");
    if (n == 0) return 0;
    if (int rc = ot_check_keys(n, keys)) return rc;
    if (int rc = ot_check_first(n, first)) return rc;
    if (first[n] && !sites) return fail(CRP_ERR_ARG, "sites is NULL");
    unsigned long long *d_keys = nullptr;
    int rc = ot_upload_keys(ix, n, keys, &d_keys);
    if (!rc) rc = ot_list(ix, d_keys, nullptr, n, max_mm, first, sites);
    dev_free(d_keys, ix->st);
    return rc;
}

}  // extern "C"

// The weight table of a score call, [kOtScoreSets]: CRP_ERR_ARG if NULL or if an entry of a set of size <= k is 2^31
// or more (2^32 sites of weight < 2^31 cannot overflow a uint64 sum); the entries of larger sets are not read.
static int ot_check_weights(uint32_t k, const uint32_t *weights) {
    static const uint32_t used[4] = {1, 21, 211, kOtScoreSets};
    if (!weights) return fail(CRP_ERR_ARG, "weights is NULL");
    for (uint32_t r = 0; r < used[k]; ++r)
        if (weights[r] >> 31) return fail(CRP_ERR_ARG, "weights[%u] = %u: at most 2^31 - 1", r, weights[r]);
    return 0;
}

// Weight sums of n queries whose keys are on the device: d_sums [n], primed by the caller, to sums on the host.
static int ot_score(crp_offtarget *ix, const unsigned long long *d_keys, uint64_t n, uint32_t k, const uint32_t *weights,
                    unsigned long long *d_sums, uint64_t *sums) {
    cudaStream_t st = ix->st;
    uint32_t *d_w = nullptr;
    if (dev_alloc(&d_w, kOtScoreSets * sizeof(uint32_t), st) != cudaSuccess) {
        cudaGetLastError();
        return fail(CRP_ERR_NOMEM, "cudaMalloc of the weight table failed");
    }
    int rc = 0;
    if (cudaMemcpyAsync(d_w, weights, kOtScoreSets * sizeof(uint32_t), cudaMemcpyHostToDevice, st) != cudaSuccess)
        rc = fail(CRP_ERR_CUDA, "H2D of the weight table failed");
    if (!rc) rc = ot_join(ix, d_keys, n, k, OtScore{d_w, d_sums});
    if (!rc && (cudaMemcpyAsync(sums, d_sums, n * sizeof(uint64_t), cudaMemcpyDeviceToHost, st) != cudaSuccess ||
                cudaStreamSynchronize(st) != cudaSuccess))
        rc = fail(CRP_ERR_CUDA, "D2H of the off-target scores failed");
    dev_free(d_w, st);
    return rc;
}

extern "C" {

int crp_offtarget_score_candidates(crp_offtarget *ix, const crp_result *res, char strand, uint32_t max_mm,
                                   const uint32_t *weights, uint64_t *sums) {
    if (int rc = ot_check_candidates(ix, res, strand, max_mm, "scores", false)) return rc;
    if (int rc = ot_check_weights(max_mm, weights)) return rc;
    const int s = strand == '+' ? 0 : 1;
    const uint64_t n = s == 0 ? res->n_plus : res->n_minus;
    if (n == 0) return 0;
    if (!sums) return fail(CRP_ERR_ARG, "sums is NULL");
    cudaStream_t st = ix->st;
    uint32_t *d_seg = nullptr;
    unsigned long long *d_keys = nullptr, *d_sums = nullptr;
    int rc = 0;
    if (dev_alloc(&d_sums, n * sizeof(unsigned long long), st) != cudaSuccess) {
        cudaGetLastError();
        rc = fail(CRP_ERR_NOMEM, "cudaMalloc of %llu query rows failed", (unsigned long long)n);
    }
    if (!rc) rc = ot_candidate_keys(ix, res, s, nullptr, 0, &d_keys, &d_seg);
    if (!rc) {                                                 // the query keys, then the primed sums
        k_ot_score_prime<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(d_keys, n, ix->own_site ? 0ull - weights[0] : 0ull,
                                                                      d_sums);
        g_ctx.launches++;
        if (cudaGetLastError() != cudaSuccess) rc = fail(CRP_ERR_CUDA, "off-target score priming failed");
    }
    if (!rc) rc = ot_score(ix, d_keys, n, max_mm, weights, d_sums, sums);
    dev_free(d_seg, st);
    dev_free(d_keys, st);
    dev_free(d_sums, st);
    return rc;
}

int crp_offtarget_score_keys(crp_offtarget *ix, uint64_t n, const uint64_t *keys, uint32_t max_mm, const uint32_t *weights,
                             uint64_t *sums) {
    if (!ix) return fail(CRP_ERR_ARG, "ix is NULL");
    if (int rc = need_ctx()) return rc;
    if (max_mm > 3) return fail(CRP_ERR_ARG, "max_mm %u: at most 3 mismatches", max_mm);
    if (int rc = ot_check_weights(max_mm, weights)) return rc;
    if (n == 0) return 0;
    if (!sums) return fail(CRP_ERR_ARG, "sums is NULL");
    if (int rc = ot_check_keys(n, keys)) return rc;
    cudaStream_t st = ix->st;
    unsigned long long *d_keys = nullptr, *d_sums = nullptr;
    int rc = ot_upload_keys(ix, n, keys, &d_keys);
    if (!rc && dev_alloc(&d_sums, n * sizeof(unsigned long long), st) != cudaSuccess) {
        cudaGetLastError();
        rc = fail(CRP_ERR_NOMEM, "cudaMalloc of %llu keys failed", (unsigned long long)n);
    }
    if (!rc && cudaMemsetAsync(d_sums, 0, n * sizeof(unsigned long long), st) != cudaSuccess)
        rc = fail(CRP_ERR_CUDA, "memset failed");
    if (!rc) rc = ot_score(ix, d_keys, n, max_mm, weights, d_sums, sums);
    dev_free(d_keys, st);
    dev_free(d_sums, st);
    return rc;
}

int crp_offtarget_timing(const crp_offtarget *ix, float *ms_sites, float *ms_count, uint64_t *comparisons) {
    if (!ix) return fail(CRP_ERR_ARG, "ix is NULL");
    if (ms_sites) *ms_sites = ix->ms_sites;
    if (ms_count) *ms_count = ix->ms_count;
    if (comparisons) *comparisons = ix->comparisons;
    return 0;
}

int crp_offtarget_free(crp_offtarget *ix) {
    if (!ix) return 0;
    if (ix->st) {
        dev_free(ix->keys, ix->st);
        dev_free(ix->loci, ix->st);
        cudaStreamSynchronize(ix->st);
    }
    for (cudaEvent_t e : ix->ev)
        if (e) cudaEventDestroy(e);
    if (ix->st) cudaStreamDestroy(ix->st);
    delete ix;
    return 0;
}

}  // extern "C"
